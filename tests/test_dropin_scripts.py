"""Script-level drop-in (SURVEY.md section 8f-1): with this repo AND a reference checkout on PYTHONPATH, the reference's own
scripts import unchanged -- hot-path modules resolve to the B200 shims, everything else (vidtok.data.*, vidtok.modules.lpips)
to the reference -- and `load_model_from_config` (scripts/inference_evaluate.py:26-32) builds the B200 engine.

The reference checkout is the one oracle/ref_shim.py locates (VIDTOK_REFERENCE_ROOT overrides it), the same one the golden
fixtures were made from.  Without one, the checks run against a stand-in checkout with the reference's package layout,
and the configs come from tests/golden/zoo_manifest.json.gz (the `model:` sections of the reference's YAMLs): where the
overlay resolves each module, which engine the config builds, and its parameter count.  What only the reference's own
scripts can show -- that they import unchanged, that their compute_ssim is ours and that their dataset derives from the
checkout's vidtok.data.vidtok -- is checked with the reference only.  Runs in subprocesses so the import state of the
test process is untouched.  Also: the oracle pin is reproducible (oracle/make_golden.py, needs the reference), the oracle's
parameter table equals the reference's state_dict, and compute_ssim equals the reference formula."""
import gzip
import json
import os
import subprocess
import sys
import tempfile
import textwrap

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import GOLDEN_DIR, ROOT, golden_cases, load_golden
from oracle import ref_shim

REF = ref_shim.REFERENCE_ROOT
HAVE_REF = ref_shim.reference_available()
needs_ref = pytest.mark.skipif(not HAVE_REF, reason="reference checkout not present")
ZOO = json.load(gzip.open(os.path.join(GOLDEN_DIR, "zoo_manifest.json.gz"), "rt"))

# The part of the reference's layout that the inference scripts import from and vidtok/__init__.py looks for: `vidtok` is a
# namespace package (no __init__.py) holding data/ and modules/util.py.
STANDIN = {
    "vidtok/data/vidtok.py": "class VidTokValDataset:\n    pass\n",
    "vidtok/modules/util.py": "",
    "vidtok/modules/lpips.py": "class LPIPS:\n    pass\n",
}


@pytest.fixture
def checkout(tmp_path):
    if HAVE_REF:
        return REF
    for rel, text in STANDIN.items():
        (tmp_path / rel).parent.mkdir(parents=True, exist_ok=True)
        (tmp_path / rel).write_text(text)
    return str(tmp_path)


# Modules the scripts import that are absent offline (SURVEY.md section 0.5).  Stubs only: no behaviour is borrowed.
STUBS = textwrap.dedent('''
    import sys, types, copy, yaml
    def _mod(name, **attrs):
        m = types.ModuleType(name); m.__dict__.update(attrs); sys.modules[name] = m; return m
    class _Cfg(dict):
        """attribute access + item access, like an OmegaConf DictConfig"""
        def __getattr__(self, k):
            try: return self[k]
            except KeyError: raise AttributeError(k)
        def __setattr__(self, k, v): self[k] = v
    def _wrap(o):
        if isinstance(o, dict): return _Cfg({k: _wrap(v) for k, v in o.items()})
        if isinstance(o, list): return [_wrap(v) for v in o]
        return o
    def _load(path):
        cfg = yaml.safe_load(open(path))
        dp = cfg["model"]["params"]["decoder_config"]
        if isinstance(dp.get("params"), str):   # ${model.params.encoder_config.params}
            dp["params"] = copy.deepcopy(cfg["model"]["params"]["encoder_config"]["params"])
        return _wrap(cfg)
    _mod("omegaconf", OmegaConf=types.SimpleNamespace(load=_load), ListConfig=list)
    _mod("decord", bridge=types.SimpleNamespace(set_bridge=lambda *_: None), VideoReader=object, cpu=lambda *_: None)
    lt = _mod("lightning"); pl = _mod("lightning.pytorch", seed_everything=lambda *a, **k: None)
    lt.pytorch = pl
    ut = _mod("lightning.pytorch.utilities"); rz = _mod("lightning.pytorch.utilities.rank_zero", rank_zero_only=lambda f: f)
    ut.rank_zero = rz; ut.rank_zero_only = rz.rank_zero_only; pl.utilities = ut
    import torchvision.io as _tvio
    if not hasattr(_tvio, "write_video"):   # removed from recent torchvision; the script only calls it when saving mp4s
        _tvio.write_video = lambda *a, **k: None
''')


def run_py(checkout, *parts):
    """Runs the code `parts` (each dedented) in a fresh interpreter with this repo, then `checkout`, on PYTHONPATH."""
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([ROOT, checkout])   # INTEGRATION.md: this repo first, then the reference checkout
    code = "".join(textwrap.dedent(p) for p in ((STUBS,) if HAVE_REF else ()) + parts)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=tempfile.gettempdir(),
                       timeout=600)
    assert r.returncode == 0, r.stdout + "\n" + r.stderr
    return r.stdout


def load_model_code(config):
    """Code that builds `model` from the reference config `config` (a path under configs/) as scripts/inference_evaluate.py
    does, and names the script, its compute_ssim and the base class of its dataset (all None with the stand-in).  With the reference:
    its own script, unmodified, on the YAML.  With the stand-in: the script's imports (:20-23) and the steps of its
    load_model_from_config (:26-32) on the recorded `model:` section."""
    if HAVE_REF:
        return f"""
            import inspect
            import scripts.inference_evaluate as ev          # the reference's script, unmodified
            import scripts.inference_reconstruct as rc
            model = ev.load_model_from_config({os.path.join(REF, "configs", config)!r}, None)
            script, ssim_fn, dataset_cls = inspect.getfile(ev), ev.compute_ssim, ev.MultiVideoDataset.__mro__[1].__module__
        """
    return f"""
        from vidtok.data.vidtok import VidTokValDataset
        from vidtok.modules.lpips import LPIPS
        from vidtok.modules.util import compute_psnr, compute_ssim, instantiate_from_config, print0
        cfg = {ZOO[config]["model"]!r}
        cfg["params"].update(ckpt_path=None, ignore_keys=[], verbose=False)
        model = instantiate_from_config(cfg)
        script = ssim_fn = dataset_cls = None
    """


def test_reference_scripts_import_unchanged_and_build_the_b200_engine(checkout):
    out = run_py(checkout, load_model_code("vidtok_kl_causal_488_4chn.yaml"), '''
        import inspect, json
        import vidtok, vidtok.data.vidtok, vidtok.modules.lpips, vidtok.modules.util, vidtok.models.autoencoder
        print(json.dumps({
            "script": script, "dataset": inspect.getfile(vidtok.data.vidtok), "lpips": inspect.getfile(vidtok.modules.lpips),
            "util": inspect.getfile(vidtok.modules.util),
            "engine": inspect.getfile(type(model)), "engine_cls": type(model).__name__, "is_causal": model.is_causal,
            "tdf": model.encoder.time_downsample_factor, "has_tiling": hasattr(model, "use_tiling"),
            "ssim": ssim_fn is vidtok.modules.util.compute_ssim, "nparams": len(model.state_dict()), "dataset_cls": dataset_cls,
        }))
    ''')
    info = json.loads(out.strip().splitlines()[-1])
    if HAVE_REF:
        assert info["script"].startswith(REF) and info["ssim"] is True and info["dataset_cls"] == "vidtok.data.vidtok"
    assert info["dataset"].startswith(checkout) and info["lpips"].startswith(checkout) and info["util"].startswith(ROOT)
    assert info["engine"].startswith(ROOT) and info["engine_cls"] == "AutoencodingEngine"
    assert info["is_causal"] is True and info["tdf"] == 4 and info["has_tiling"] is False and info["nparams"] == 416


def test_v11_config_resolves_to_the_tiling_engine(checkout):
    out = run_py(checkout, load_model_code("vidtok_v1_1/vidtok_kl_causal_488_16chn_v1_1.yaml"), '''
        import json
        # scripts/inference_evaluate.py:144-150
        assert hasattr(model, "use_tiling")
        model.use_tiling = True; model.t_chunk_enc = 16
        model.t_chunk_dec = model.t_chunk_enc // model.encoder.time_downsample_factor; model.use_overlap = True
        print(json.dumps({"cls": type(model).__name__, "z": model.spec.z_channels, "interp": model.spec.interpolation_mode,
                          "chunks": model.build_chunk_start_end(129)[:3]}))
    ''')
    info = json.loads(out.strip().splitlines()[-1])
    assert info == {"cls": "AutoencodingEngineV11", "z": 16, "interp": "trilinear", "chunks": [[0, 1], [1, 17], [17, 33]]}


@needs_ref
def test_golden_fixture_regenerates_bit_identically(tmp_path):
    """python oracle/make_golden.py runs as committed (the shim package no longer shadows the reference) and reproduces
    the committed fixture bit for bit."""
    env = dict(os.environ)
    env["VIDTOK_GOLDEN_OUT"] = str(tmp_path)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "make_golden.py"), "tiny_kl_v10"], capture_output=True, text=True,
                       env=env, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    a, b = np.load(tmp_path / "tiny_kl_v10.npz"), np.load(os.path.join(GOLDEN_DIR, "tiny_kl_v10.npz"))
    assert set(a.files) == set(b.files)
    for k in a.files:
        if k != "meta_json":
            assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("case", golden_cases())
def test_oracle_param_table_equals_reference_state_dict(case):
    from oracle.vidtok_oracle import cfg_from_model_yaml, reference_param_shapes
    d, meta = load_golden(case)   # meta["shapes"] = state_dict() shapes of the unmodified reference (oracle/make_golden.py)
    assert reference_param_shapes(cfg_from_model_yaml(meta["model"])) == {k: tuple(v) for k, v in meta["shapes"].items()}


def test_compute_ssim_matches_the_reference_formula():
    """vidtok/modules/util.py:157-178 stated directly (2-D 11x11 Gaussian window) vs the separable implementation."""
    from vidtok_b200.compat_util import compute_ssim
    g = torch.Generator().manual_seed(0)
    for shape in [(2, 3, 5, 64, 48), (1, 3, 2, 600, 520)]:   # the second exercises the avg-pool prefilter (f = 2)
        x = torch.rand(shape, generator=g)
        y = (x + 0.1 * torch.randn(shape, generator=g)).clamp(0, 1)
        a = x.permute(0, 2, 1, 3, 4).reshape(-1, 3, *shape[3:])
        b = y.permute(0, 2, 1, 3, 4).reshape(-1, 3, *shape[3:])
        f = max(1, round(min(shape[3:]) / 256))
        if f > 1:
            a, b = F.avg_pool2d(a, f), F.avg_pool2d(b, f)
        t = torch.arange(11, dtype=torch.float32) - 5.0
        k = torch.exp(-(t[None] ** 2 + t[:, None] ** 2) / (2 * 1.5 ** 2))
        k = (k / k.sum())[None, None].repeat(3, 1, 1, 1)
        blur = lambda v: F.conv2d(v, k, groups=3)  # noqa: E731
        mx, my = blur(a), blur(b)
        sxx, syy, sxy = blur(a * a) - mx * mx, blur(b * b) - my * my, blur(a * b) - mx * my
        cs = (2 * sxy + 0.03 ** 2) / (sxx + syy + 0.03 ** 2)
        ss = (2 * mx * my + 0.01 ** 2) / (mx * mx + my * my + 0.01 ** 2) * cs
        ref = ss.mean(dim=(-1, -2)).mean(1).mean(0)
        got = compute_ssim(x, y)
        assert abs(float(got) - float(ref)) < 2e-6, (float(got), float(ref))
        assert float(compute_ssim(x, x)) > 0.999999
