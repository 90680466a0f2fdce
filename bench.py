#!/usr/bin/env python
"""Benchmark of the tokenizer hot path: frames/sec for full encode -> regularize -> decode on synthetic clips.

  python bench.py --gpus N --steps K --warmup W                       # B200 arm, BASELINE.json configs[1] (the headline)
  python bench.py --config {kl488,fsq488,v11long,kl41616} [--precision {bf16,exact,mixed,fma}]
  python bench.py --impl reference [--config ...] --steps K ...        # reference arm: the reference's CPU path (oracle port)
  python bench.py ... --dump-outputs DIR                               # also write the last timed step's outputs as DIR/*.npy

A "step" is one pass of the hot path over one batch of clips per GPU (weak scaling; one process per GPU under torchrun for
N > 1).  `value` is timed with CUDA events with the inputs already resident in HBM; `e2e` goes through the public Python API
(AutoencodingEngine.forward resolved from the YAML target strings) from pinned host memory and back.  One JSON line on rank 0.

configs (BASELINE.json `configs`, SURVEY.md section 8d):
  kl488    [1] vidtok_kl_causal_488_4chn, 8 clips 17x256x256 per GPU, bf16 (default: the metric BASELINE.json is quoted on)
  fsq488   [2] vidtok_fsq_causal_488_32768, 8 clips 17x256x256 per GPU, "mixed" = encoder fp16x3 split operands (bit-exact codes), decoder bf16
  v11long  [3] vidtok_kl_causal_488_16chn v1.1, one 129x256x256 video per GPU, tiled t_chunk_enc=16 with overlap, bf16
  kl41616  [4] vidtok_kl_causal_41616_4chn, 4 clips 17x512x512 per GPU (32 clips over 8 GPUs), bf16
"""
from __future__ import annotations

import argparse
import atexit
import json
import math
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "frames/sec encode+decode, kl_causal_488 17x256x256"

# flops: algorithmic FLOPs per clip / video (BASELINE.md section 2, FlopCounterMode over the reference graph)
CONFIGS = {
    "kl488": dict(idx=1, name="vidtok_kl_causal_488_4chn", metric=METRIC, version="v1_0", reg="kl", z=4, ch_mult=(1, 2, 4, 4),
                  T=17, H=256, W=256, batch=8, flops=20.691e12, precision="bf16", tiling=None),
    "fsq488": dict(idx=2, name="vidtok_fsq_causal_488_32768", metric="frames/sec encode+decode, fsq_causal_488_32768 17x256x256",
                   version="v1_0", reg="fsq", z=5, ch_mult=(1, 2, 4, 4), T=17, H=256, W=256, batch=8, flops=20.690e12,
                   precision="mixed", tiling=None),
    "v11long": dict(idx=3, name="vidtok_kl_causal_488_16chn v1.1", metric="frames/sec encode+decode, kl_causal_488_16chn_v1_1 129x256x256 tiled",
                    version="v1_1", reg="kl", z=16, ch_mult=(1, 2, 4, 4), T=129, H=256, W=256, batch=1, flops=160.38e12,
                    precision="bf16", tiling=(16, 4, True)),
    "kl41616": dict(idx=4, name="vidtok_kl_causal_41616_4chn", metric="frames/sec encode+decode, kl_causal_41616 17x512x512",
                    version="v1_0", reg="kl", z=4, ch_mult=(1, 2, 4, 4, 4), T=17, H=512, W=512, batch=4, flops=85.627e12,
                    precision="bf16", tiling=None),
}
DTYPE_OF = {"bf16": "bf16", "exact": "fp16x3 (hi|lo split fp16 operands, 3 MMAs per K step, fp32-class results)", "mixed": "encoder fp16x3, decoder bf16",
            "fma": "f32"}


def model_cfg(c, ch=128):
    """model section of configs/<name>.yaml (e.g. configs/vidtok_kl_causal_488_4chn.yaml:1-36)."""
    v11 = c["version"] == "v1_1"
    ep = dict(double_z=(c["reg"] == "kl"), z_channels=c["z"], in_channels=3, out_ch=3, ch=ch, ch_mult=list(c["ch_mult"]),
              time_downsample_factor=4, num_res_blocks=2, dropout=0.0, use_checkpoint=False,
              init_pad_mode="replicate", norm_type="layernorm", fix_encoder=False, fix_decoder=False)
    if v11:
        ep["interpolation_mode"] = "trilinear"   # configs/vidtok_v1_1/*.yaml:27
    mod = "vidtok.modules.model_3dcausal_v1_1" if v11 else "vidtok.modules.model_3dcausal"
    if c["reg"] == "fsq":
        rc = {"target": "vidtok.modules.regularizers.FSQRegularizer",
              "params": {"levels": [8, 8, 8, 8, 8], "entropy_loss_weight": 0.1, "entropy_loss_annealing_factor": 1.2,
                         "commitment_loss_weight": 0.25}}
    else:
        rc = {"target": "vidtok.modules.regularizers.DiagonalGaussianRegularizer"}
    return {
        "target": "vidtok.models.autoencoder_v1_1.AutoencodingEngine" if v11 else "vidtok.models.autoencoder.AutoencodingEngine",
        "params": {
            "monitor": "val/rec_loss", "mode": "min", "ignore_keys": [],
            "encoder_config": {"target": mod + ".EncoderCausal3DPadding", "params": ep},
            "decoder_config": {"target": mod + ".DecoderCausal3DPadding", "params": dict(ep)},
            "regularizer_config": rc,
            "loss_config": {"target": "vidtok.modules.losses.GeneralLPIPSWithDiscriminator"},
        },
    }


def workload_string(c, precision, B):
    what = f"{c['name']} {precision}: batch {B} clip{'s' if B > 1 else ''} {c['T']}x{c['H']}x{c['W']} per GPU"
    if c["tiling"]:
        what += f", tiled t_chunk_enc={c['tiling'][0]} t_chunk_dec={c['tiling'][1]} use_overlap={c['tiling'][2]}"
    return what + f" (BASELINE.json configs[{c['idx']}])"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"tflops": float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1431.0))), "hbm_gbs": float(d.get("hbm_gbs", 6568.0)),
                "source": "MEASURED_PEAKS.json (bf16_tflops_sustained: kernel timed inside a long step)"}
    return {"tflops": 1400.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md: ~1.4 PFLOP/s sustained)"}


DUMP_BYTES = 60 << 20    # array data of all of --dump-outputs together: the files, headers included, stay under 64 MB
DUMP_SAMPLE_SEED = 0


def dump_outputs(out_dir, arrays):
    """Writes what one step returned to the caller as out_dir/<name>.npy in float32, so that two builds can be compared
    output for output.  Arrays go smallest first, each with an equal share of the DUMP_BYTES not yet used by the ones before
    it.  An array larger than its share is written as <name>_sample.npy: the flattened array at sorted positions drawn
    uniformly (with replacement) from a CPU generator seeded with DUMP_SAMPLE_SEED, as many as the share holds.  The
    positions depend only on the element count, so the same workload gives the same sample."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_BYTES
    written = {}
    for i, (name, t) in enumerate(sorted(arrays.items(), key=lambda kv: kv[1].numel())):
        t = t.detach().float()
        share = left // (len(arrays) - i)
        if 4 * t.numel() > share:
            pos = torch.randint(t.numel(), (share // 4,), generator=torch.Generator().manual_seed(DUMP_SAMPLE_SEED)).sort().values
            t, name = t.flatten()[pos.to(t.device)], name + "_sample"
        a = t.cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a)
        left -= a.nbytes
        written[name] = list(a.shape)
    return written


# --------------------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index = index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
        else:
            atexit.register(self.proc.kill)   # a run that fails before stop() must not leave nvidia-smi polling

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        for line in out.strip().splitlines():
            f = [s.strip() for s in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])), mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
# CPU reference (oracle port of the reference's PyTorch CPU path).  No CUDA library is touched here: the weight shapes
# come from the oracle's parameter table (pinned against the reference's state_dict in tests/test_oracle_golden.py).
# --------------------------------------------------------------------------------------------------
def oracle_model(c, sd=None):
    from oracle.vidtok_oracle import OracleModel, cfg_from_model_yaml, reference_param_shapes
    from vidtok_b200.synth import synth_state_dict
    ocfg = cfg_from_model_yaml(model_cfg(c))
    if sd is None:
        sd = synth_state_dict(reference_param_shapes(ocfg), seed=0)
    om = OracleModel(ocfg, sd)
    if c["tiling"]:
        om.use_tiling, om.t_chunk_enc, om.t_chunk_dec, om.use_overlap = True, c["tiling"][0], c["tiling"][1], c["tiling"][2]
    return om


def cpu_forward_timed(om, x, noise_seed=4321):
    torch.manual_seed(noise_seed)
    t0 = time.perf_counter()
    z, dec, log = om.forward(x)
    return time.perf_counter() - t0, dec, log


def pick_cpu_threads(om):
    """The reference would run with torch's default (all host cores).  On cgroup-limited hosts that oversubscribes
    badly (128 visible cores, far fewer usable), so probe a few thread counts on a tiny clip and keep the fastest."""
    from vidtok_b200.synth import synth_clip
    cores = os.cpu_count() or 1
    try:
        cores = min(cores, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    x = synth_clip(1, 17, 32, 32)
    best_t, best_n = None, cores
    for n in sorted({cores, max(cores // 2, 1), max(cores // 4, 1), 32, 16, 8}):
        if n > cores:
            continue
        torch.set_num_threads(n)
        t = min(cpu_forward_timed(om, x)[0], cpu_forward_timed(om, x)[0])
        if best_t is None or t < best_t:
            best_t, best_n = t, n
        elif t > 1.5 * best_t:  # more threads only oversubscribe from here on
            break
    torch.set_num_threads(best_n)
    return best_n


def cpu_sample_shape(c, om, budget_s: float, steps: int):
    """Largest sample (T_s x S x S) of the config's workload whose `steps` forwards fit the budget, from a 64x64 probe.
    The spatial size shrinks first (256/512 -> 128 -> 64); the tiled long video also shrinks to 33 frames (three chunks:
    first frame, two full chunks with look-ahead)."""
    from vidtok_b200.synth import synth_clip
    T_s = c["T"] if not c["tiling"] else 33
    t64 = min(cpu_forward_timed(om, synth_clip(1, T_s, 64, 64))[0], cpu_forward_timed(om, synth_clip(1, T_s, 64, 64))[0])
    sizes = [s for s in (c["H"], 256, 128, 64) if s <= c["H"]]
    for S in dict.fromkeys(sizes):
        if t64 * (S / 64) ** 2 * steps <= budget_s:
            return T_s, S
    return T_s, 64


def cpu_units_scale(c, T_s, S):
    """frames of the full-size workload that one sample forward is worth (pixel-count scaling; stated in `sample`)"""
    return (T_s * S * S) / float(c["T"] * c["H"] * c["W"]) * c["T"]


def run_reference_arm(args, c):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from vidtok_b200.synth import synth_clip
    om = oracle_model(c)
    cores = pick_cpu_threads(om)
    total = args.steps + args.warmup
    T_s, S = cpu_sample_shape(c, om, budget_s=240.0, steps=total)
    x = synth_clip(1, T_s, S, S)
    for _ in range(args.warmup):
        cpu_forward_timed(om, x)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_forward_timed(om, x)
    el = time.perf_counter() - t0
    fps = cpu_units_scale(c, T_s, S) * args.steps / el
    full = (T_s, S) == (c["T"], c["H"])
    sample = f"1 clip 3x{T_s}x{S}x{S} per step on {cores} host threads of {os.cpu_count()} visible (oracle port of the reference PyTorch CPU path, fp32)"
    if not full:
        sample += (f"; a full-size {c['T']}x{c['H']}x{c['W']} step does not fit the few-minute budget of {total} steps on the CPU, so the value is the "
                   f"sample's voxels/s converted to {c['H']}x{c['W']}-frame units (x{(S * S) / float(c['H'] * c['W']):.4f} per frame)")
    line = {
        "impl": "reference", "metric": c["metric"], "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{c['name']}: clips {c['T']}x{c['H']}x{c['W']} (reference CPU path, fp32; BASELINE.json configs[{c['idx']}])",
                   "sample": sample, "full_size_step": full},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------------------------------
def native_library():
    """The CUDA library as the current sources build it.  That is the one build() left in the tree while it is at least as
    new as every source and header; otherwise the sources are compiled into a temporary directory, removed at exit, and that
    build is loaded.  So the timed kernels always match the sources, and nothing is written into the tree, which may be
    read-only."""
    from vidtok_b200 import _native as N
    from vidtok_b200 import build as vb
    if vb.is_stale():
        tmp = tempfile.mkdtemp(prefix="vidtok_b200_")
        atexit.register(shutil.rmtree, tmp, True)
        print(f"bench.py: {vb.LIB} is missing or older than its sources; building them in {tmp}", file=sys.stderr, flush=True)
        N.LIB_PATH = vb.build(force=True, out_dir=tmp)
    lib = N.lib()
    assert lib.vt_abi_version() == 2
    return lib


def run_b200_arm(args, c):
    native_library()   # before anything loads the library
    from vidtok_b200 import _native as N
    from vidtok_b200 import dist as vdist
    from vidtok_b200.compat_util import instantiate_from_config
    from vidtok_b200.synth import synth_clip, synth_state_dict

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the B200 arm has no CPU fallback; use --impl reference for the CPU path)")
    rank, world, local = vdist.init_from_env("nccl")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    B = args.batch or c["batch"]
    T, H, W = c["T"], c["H"], c["W"]
    precision = args.precision or c["precision"]
    model = instantiate_from_config(model_cfg(c))
    sd = synth_state_dict({k: tuple(v.shape) for k, v in model.state_dict().items()}, seed=0)
    model.load_state_dict(sd)
    model = model.to(dev).eval()
    model.precision = precision
    if c["tiling"]:
        # exactly what scripts/inference_evaluate.py:144-150 does
        model.use_tiling = True
        model.t_chunk_enc, model.t_chunk_dec, model.use_overlap = c["tiling"]
    lib = N.lib()

    x_host = synth_clip(B, T, H, W, seed=1234 + rank).pin_memory()
    out_host = torch.empty_like(x_host).pin_memory()
    x_dev = x_host.to(dev)
    torch.manual_seed(4321)

    def step_resident():
        with torch.no_grad():
            return model(x_dev)

    # End-to-end leg: the call a user makes (model(x) on the current stream) with every step's input coming from pinned host
    # memory and every step's reconstruction going back to pinned host memory.  The copies run on a second stream, double
    # buffered: H2D of step k+1 and D2H of step k-1 overlap the kernels of step k (each step's copies stay inside the timed
    # region: the first H2D and the last D2H are not hidden).
    copy_stream = torch.cuda.Stream(device=dev)
    in_bufs = [torch.empty_like(x_dev), torch.empty_like(x_dev)]

    def run_e2e_clips(steps):
        main = torch.cuda.current_stream(dev)
        ready = [torch.cuda.Event(), torch.cuda.Event()]   # input buffer i holds its step's clip
        freed = [torch.cuda.Event(), torch.cuda.Event()]   # the step that read input buffer i has finished
        dec = None
        with torch.no_grad():
            with torch.cuda.stream(copy_stream):
                in_bufs[0].copy_(x_host, non_blocking=True)
                ready[0].record(copy_stream)
            for k in range(steps):
                cur = k & 1
                main.wait_event(ready[cur])
                _, dec, _ = model(in_bufs[cur])
                freed[cur].record(main)
                dec.record_stream(copy_stream)
                with torch.cuda.stream(copy_stream):
                    if k + 1 < steps:
                        if k >= 1:
                            copy_stream.wait_event(freed[cur ^ 1])
                        in_bufs[cur ^ 1].copy_(x_host, non_blocking=True)
                        ready[cur ^ 1].record(copy_stream)
                    copy_stream.wait_event(freed[cur])
                    out_host.copy_(dec, non_blocking=True)
        main.wait_stream(copy_stream)
        return dec

    # Tiled long video: the library stages the chunks itself (vt_encode_video reads the pinned host video chunk by chunk on its
    # copy stream while the previous chunk computes; vt_decode_video copies each decoded chunk to pinned host memory while the
    # next one computes) -- the user-facing calls are model.encode(host_video) and model.tile_decode(z, out=host_buffer).
    out_host_video = None

    def run_e2e_video(steps):
        nonlocal out_host_video
        dec = None
        with torch.no_grad():
            for _ in range(steps):
                zz = model.encode(x_host)
                if out_host_video is None:
                    nf = int(zz.shape[2])
                    t_out = int(lib.vt_decode_video_frames(model._rt.sync().handle, nf, int(model.t_chunk_dec), int(bool(model.use_overlap))))
                    out_host_video = torch.empty((B, 3, t_out, H, W), dtype=torch.float32).pin_memory()
                dec = model.tile_decode(zz, out=out_host_video)
        return dec[:, :, -T:].to(dev, non_blocking=True)

    run_e2e = run_e2e_video if c["tiling"] else run_e2e_clips

    # the clock sampler starts BEFORE the warm-up: nvidia-smi takes ~1 s to initialise NVML, and doing that inside the
    # timed region cost the first steps ~10 % (profiles/notes_r1.md); its samples cover warm-up + timed steps, all under load
    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(max(args.warmup, 3)):
        step_resident()
    torch.cuda.synchronize(dev)

    # ---- device-timed region (inputs resident in HBM)
    vdist.barrier()
    torch.cuda.synchronize(dev)
    lib.vt_launch_count(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        z, dec, log = step_resident()
    e1.record()
    torch.cuda.synchronize(dev)
    vdist.barrier()
    launches = int(lib.vt_launch_count(0))
    clocks = sampler.stop()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    ms = float(vdist.allreduce_max(ms)[0])
    frames = world * B * T * args.steps
    value = frames / (ms / 1e3)
    dumped = None
    if args.dump_outputs and rank == 0:   # what the last timed step returned (z, dec, reg_log), copied after the timed region
        dumped = dump_outputs(args.dump_outputs, {"z": z, "dec": dec, **log})

    # ---- end to end through the public API with host buffers
    run_e2e(2)
    torch.cuda.synchronize(dev)
    vdist.barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    dec = run_e2e(args.steps)
    e3.record()
    torch.cuda.synchronize(dev)
    vdist.barrier()
    ms_e2e = torch.tensor([e2.elapsed_time(e3)], dtype=torch.float64, device=dev)
    ms_e2e = float(vdist.allreduce_max(ms_e2e)[0])
    e2e_value = frames / (ms_e2e / 1e3)

    # ---- the one collective: global PSNR(input, reconstruction) from per-rank partial sums (NCCL all-reduce)
    psnr_b200 = vdist.global_psnr(vdist.psnr_partial(x_dev, dec.float()))

    # ---- per-kernel attribution of one step (CUDA events around every launch, on the launch stream)
    peaks = load_peaks()
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "ncu_conv_tc_r2.json")
    if not os.path.exists(tpath):
        tpath = os.path.join(ROOT, "profiles", "ncu_conv_tc_r1.json")
    if os.path.exists(tpath) and args.config == "kl488":  # dram__bytes_read+write per launch from the committed `ncu --set full` capture
        try:
            cap = json.load(open(tpath))
            vals = [l["dram_read_bytes"] + l["dram_write_bytes"] for l in cap["launches"] if l.get("dram_read_bytes") is not None]
            traffic = {"bytes_per_launch_avg": sum(vals) / len(vals), "launches_captured": len(vals), "source": os.path.relpath(tpath, ROOT)}
        except Exception:
            traffic = None
    roof = None
    if rank == 0:
        # PROF_STEPS steps back to back under the profiler, long enough to be at the sustained (power-capped) clock and for
        # nvidia-smi to sample it: the per-kernel sum, the event-timed wall time of the same steps and the clock during them,
        # so that "step time - kernel sum" can be split into bubbles and clock
        PROF_STEPS = max(5, int(math.ceil(2500.0 / (ms / args.steps))))   # >= 2.5 s: nvidia-smi's first second yields no samples
        PROF_STEPS = max(5, min(PROF_STEPS, 8000 // max(launches // max(args.steps, 1), 1)))   # bound the events the profiler holds
        samp2 = ClockSampler(local)
        samp2.start()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        lib.vt_profile_start()
        p0.record()
        for _ in range(PROF_STEPS):
            step_resident()
        p1.record()
        torch.cuda.synchronize(dev)
        buf = __import__("ctypes").create_string_buffer(1 << 16)
        n = lib.vt_profile_stop(buf, len(buf))
        clocks_prof = samp2.stop()
        prof_wall_ms = p0.elapsed_time(p1) / PROF_STEPS
        prof = json.loads(buf.value.decode()) if n > 0 else {}
        for v in prof.values():   # per step
            v["ms"] /= PROF_STEPS
            v["flops"] /= PROF_STEPS
            v["bytes"] /= PROF_STEPS
            v["launches"] = int(round(v["launches"] / PROF_STEPS))
        tot_ms = sum(v["ms"] for v in prof.values()) or 1.0
        dom = max(prof.items(), key=lambda kv: kv[1]["ms"])[0] if prof else None
        if dom is not None:
            d = prof[dom]
            ach = d["flops"] / (d["ms"] / 1e3) / 1e12 if d["flops"] > 0 else d["bytes"] / (d["ms"] / 1e3) / 1e9
            bound = "tensor" if d["flops"] > 0 and dom.startswith("conv") else "hbm"
            peak = peaks["tflops"] if bound == "tensor" else peaks["hbm_gbs"]
            roof = {"kernel": dom, "bound": bound, "achieved": ach, "peak": peak, "unit": "TFLOP/s" if bound == "tensor" else "GB/s",
                    "frac": ach / peak, "traffic": traffic, "launches_per_step": d["launches"],
                    "avg_launch_ms": d["ms"] / max(d["launches"], 1), "share_of_step": d["ms"] / tot_ms,
                    "algorithmic_flops_per_step": d["flops"], "peak_source": peaks["source"],
                    "note": ("achieved = algorithmic FLOPs of the kernel's launches / their summed durations; conv_tc3 (split operands) executes "
                             "3 tensor-core MACs per algorithmic MAC, so its ceiling against the bf16 peak is 1/3"),
                    "whole_path": {"achieved": c["flops"] * B * args.steps / (ms / 1e3) / 1e12, "unit": "TFLOP/s per GPU (algorithmic)",
                                   "frac": c["flops"] * B * args.steps / (ms / 1e3) / 1e12 / peaks["tflops"]},
                    "sum_kernel_ms": tot_ms,
                    "profiled": {"steps": PROF_STEPS, "wall_ms_per_step": prof_wall_ms, "sum_kernel_ms_per_step": tot_ms,
                                 "sm_mhz": clocks_prof.get("sm_mhz"),
                                 "note": "the same steps timed as a whole (CUDA events) and per launch (the library's profiler brackets every "
                                         "launch with events, which serialises launches and adds ~2 event records per kernel)"},
                    "kernels_ms": {k: round(v["ms"], 3) for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])}}

    # ---- CPU baseline + parity on one sample (rank 0, N == 1 only): PSNR for KL, code mismatches for FSQ
    cpu = None
    parity = {"psnr_b200_all_clips": psnr_b200}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        om = oracle_model(c, sd)
        cores = pick_cpu_threads(om)
        T_s, S = cpu_sample_shape(c, om, budget_s=40.0, steps=1)
        xs = x_host[:1] if (T_s, S) == (T, H) else synth_clip(1, T_s, S, S)
        el, dec_ref, log_ref = cpu_forward_timed(om, xs)
        sample = (f"1 clip 3x{T_s}x{S}x{S}, 1 forward, fp32, {cores} host threads of {os.cpu_count()} visible (oracle port of the "
                  "reference PyTorch CPU path)")
        if (T_s, S) != (T, H):
            sample += f"; value = the sample's voxels/s in {H}x{W}-frame units"
        cpu = {"value": cpu_units_scale(c, T_s, S) / el, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample}
        with torch.no_grad():
            torch.manual_seed(4321)
            _, dec_g, log_g = model(xs.to(dev))
        from vidtok_b200.dist import psnr_partial
        pg = psnr_partial(xs, dec_g.float().cpu())
        pr = psnr_partial(xs, dec_ref)
        parity.update({"clip": f"3x{T_s}x{S}x{S}", "precision": precision, "psnr_b200": float(pg[0] / pg[1]),
                       "psnr_reference_cpu_fp32": float(pr[0] / pr[1]),
                       "psnr_abs_diff_db": abs(float(pg[0] / pg[1]) - float(pr[0] / pr[1])), "psnr_gate_db": 0.01,
                       "max_abs_diff": float((dec_g.float().cpu() - dec_ref).abs().max())})
        if c["reg"] == "fsq":
            bad = log_g["indices"].cpu() != log_ref["indices"]
            parity.update({"fsq_code_mismatches": int(bad.sum()), "fsq_codes": int(bad.numel()),
                           "fsq_gate": "0 mismatches outside the 1e-4 tie band (tests/test_gpu_full.py::test_config3)"})

    if rank == 0:
        nbytes = x_host.numel() * x_host.element_size()
        Tz = int(z.shape[2])
        noise_bytes = 4 * B * c["z"] * Tz * int(z.shape[3]) * int(z.shape[4]) if c["reg"] == "kl" else 0
        line = {
            "metric": c["metric"], "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE_OF[precision],
            "data": "synthetic",
            "config": {"workload": workload_string(c, precision, B), "bench_config": args.config, "precision": precision,
                       "clips_per_gpu": B, "parallelism": f"dp{world} (clips sharded, no data-path collective)",
                       "weights": "random (synth_state_dict seed 0)", "algorithmic_flops_per_clip": c["flops"],
                       "l2": "per-step activations are GBs, far larger than the 126 MB L2"},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "frames/s", "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": nbytes + noise_bytes, "d2h_bytes_per_step": nbytes,
                    "pipeline": ("the library stages the pinned host video chunk by chunk on its copy stream while the previous chunk computes "
                                 "and copies every decoded chunk back to pinned host memory while the next one computes (vt_encode_video / "
                                 "vt_decode_video)") if c["tiling"] else
                                ("every step copies its clips from pinned host memory and its reconstruction back; the copies run on a "
                                 "second stream, double buffered against the previous / next step's kernels")},
            "gpu_launches": launches,
            "roofline": roof,
            "cpu_baseline": cpu,
            "psnr": parity,
            "parity": parity,   # same record under the name VERDICT r1 asked for (PSNR delta; FSQ code mismatches for fsq488)
        }
        if dumped is not None:
            line["dumped_outputs"] = {"dir": args.dump_outputs, "shapes": dumped, "sample_seed": DUMP_SAMPLE_SEED}
        print(json.dumps(line), flush=True)
    if torch.distributed.is_initialized():
        torch.distributed.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="kl488", choices=sorted(CONFIGS.keys()))
    ap.add_argument("--precision", default=None, choices=["bf16", "exact", "mixed", "fma"], help="default: the config's")
    ap.add_argument("--batch", type=int, default=0, help="clips per GPU (default: the config's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy (float32, at most 64 MB; B200 arm, rank 0)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the B200 arm's outputs")
    c = CONFIGS[args.config]
    if args.impl == "reference":
        run_reference_arm(args, c)   # CPU only: the CUDA library is neither built nor loaded here
    else:
        run_b200_arm(args, c)


if __name__ == "__main__":
    main()
