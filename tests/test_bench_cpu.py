"""CPU-only checks of bench.py's host logic: the four configurations against BASELINE.json / SURVEY §6, the reference arm's
model construction without the CUDA library, and the JSON contract keys of the reference arm on a tiny clip."""
import json
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_configs_match_the_baseline_table():
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert "kl_causal_488" in bench.METRIC and "kl_causal_488" in base["metric"]
    c = bench.CONFIGS
    assert set(c) == {"kl488", "fsq488", "v11long", "kl41616"}
    # the headline stays the default (BENCH / SCALE records of the driver)
    ap_default = [a for a in open(os.path.join(ROOT, "bench.py")).read().splitlines() if '"--config"' in a][0]
    assert 'default="kl488"' in ap_default
    # algorithmic FLOPs per clip (SURVEY §6 / BASELINE.md §2)
    assert c["kl488"]["flops"] == pytest.approx(20.691e12) and c["fsq488"]["flops"] == pytest.approx(20.690e12)
    assert c["v11long"]["flops"] == pytest.approx(160.38e12) and c["kl41616"]["flops"] == pytest.approx(85.627e12)
    assert c["fsq488"]["precision"] == "mixed" and c["kl488"]["precision"] == "bf16"
    assert c["v11long"]["tiling"] == (16, 4, True) and c["v11long"]["T"] == 129


@pytest.mark.parametrize("name,tensors", [("kl488", 416), ("fsq488", 416), ("kl41616", None), ("v11long", None)])
def test_reference_arm_builds_its_model_from_the_shape_table(name, tensors):
    """`--impl reference` must not touch the CUDA library: the weight manifest comes from the oracle's parameter table
    (416 tensors / 157.4 M parameters for the 488 models, SURVEY §8b)."""
    from oracle.vidtok_oracle import cfg_from_model_yaml, reference_param_shapes
    shapes = reference_param_shapes(cfg_from_model_yaml(bench.model_cfg(bench.CONFIGS[name])))
    n = sum(int(torch.tensor(s).prod()) for s in shapes.values())
    if tensors is not None:
        assert len(shapes) == tensors
        assert 157.0e6 < n < 157.8e6
    assert "encoder.conv_in.conv.weight" in shapes and "decoder.conv_out.conv.weight" in shapes


def test_importing_bench_does_not_load_the_cuda_library():
    import subprocess
    code = "import sys; sys.path.insert(0, %r); import bench; import ctypes; print(any('libvidtok_b200' in l for l in open('/proc/self/maps')))" % ROOT
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    assert out.stdout.strip().endswith("False")


def test_dump_outputs_fit_the_budget_in_float32_and_sample_reproducibly(tmp_path):
    import numpy as np
    g = torch.Generator().manual_seed(0)
    outs = {"z": torch.randn(8, 4, 5, 32, 32, generator=g).bfloat16(), "dec": torch.randn(8, 3, 17, 256, 256, generator=g),
            "kl_loss": torch.tensor(2.5), "indices": torch.randint(0, 32768, (8, 5, 32, 32), generator=g, dtype=torch.int32)}
    shapes = bench.dump_outputs(str(tmp_path / "a"), outs)
    assert set(shapes) == {"z", "kl_loss", "indices", "dec_sample"}
    assert shapes["z"] == [8, 4, 5, 32, 32] and shapes["kl_loss"] == [] and shapes["indices"] == [8, 5, 32, 32]
    files = sorted(os.listdir(tmp_path / "a"))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64e6
    a = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    assert all(v.dtype == np.float32 for v in a.values())
    assert np.array_equal(a["z"], outs["z"].float().numpy()) and float(a["kl_loss"]) == 2.5
    assert np.array_equal(a["indices"], outs["indices"].numpy().astype(np.float32))
    assert np.isin(a["dec_sample"][:1000], outs["dec"].numpy()).all()
    bench.dump_outputs(str(tmp_path / "b"), outs)
    assert np.array_equal(np.load(tmp_path / "b" / "dec_sample.npy"), a["dec_sample"])
    # two arrays over the budget share it: neither sample is empty
    shapes = bench.dump_outputs(str(tmp_path / "c"), {"a": torch.zeros(20_000_000), "b": torch.zeros(30_000_000)})
    assert shapes == {"a_sample": [bench.DUMP_BYTES // 8], "b_sample": [bench.DUMP_BYTES // 8]}


def test_stale_library_is_rebuilt_outside_the_tree():
    """bench.py never times a library older than its sources, and never writes into the tree: a stale (here: missing)
    in-tree library makes it compile the current sources into a temporary directory and load that."""
    import subprocess
    from vidtok_b200 import build as vb
    before = {p: os.path.getmtime(p) for p in (vb.LIB, vb.OBJ)}
    code = ("import sys; sys.path.insert(0, %r); import bench; from vidtok_b200 import build as vb, _native as N; "
            "vb.LIB = vb.LIB + '.missing'; assert vb.is_stale(); bench.native_library(); print(N.LIB_PATH)" % ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stderr[-3000:]
    built = r.stdout.strip().splitlines()[-1]
    assert not built.startswith(ROOT) and "older than its sources" in r.stderr
    assert not os.path.exists(built)   # the temporary build is removed at exit
    assert before == {p: os.path.getmtime(p) for p in (vb.LIB, vb.OBJ)} and not os.path.exists(vb.LIB + ".missing")
    assert not vb.is_stale()


def test_cpu_sample_scaling_is_in_full_size_frames():
    c = bench.CONFIGS["kl488"]
    assert bench.cpu_units_scale(c, 17, 256) == pytest.approx(17.0)
    assert bench.cpu_units_scale(c, 17, 128) == pytest.approx(17.0 / 4)
    v = bench.CONFIGS["v11long"]
    assert bench.cpu_units_scale(v, 33, 256) == pytest.approx(33.0)
