#!/usr/bin/env python
"""bench.py — BEV frames/s of the ST-P3 camera->BEV perception hot path on B200 (see DESIGN.md, Measurement).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload perceive|lift_splat] [--batch b_per_gpu]
  python bench.py --impl reference ...     # the reference's CPU path (oracle port) on the host cores
  python bench.py ... --dump-outputs DIR   # also write the last timed step's outputs as DIR/<name>.npy

One "step" = one pass of the hot path over one batch of synthetic samples (6 cameras x 3 frames, 200x200 BEV);
one "frame" of the metric = one sample's BEV perception output.  Rank 0 prints ONE JSON line.

  perceive   (default; BASELINE configs[3], the configuration the metric is quoted on): encoder outputs ->
             lift-splat -> ego-motion + 3-D temporal block + DeepLab head -> BEV decoder heads (segmentation,
             pedestrian, hdmap logits).  The EfficientNet trunk is third-party, absent from the image and excluded on
             both arms (BASELINE.md §4): inputs enter as the trunk-head outputs (context features + depth logits).
  lift_splat (BASELINE configs[2] lift stage): lift-splat only, output = (B,3,64,200,200) BEV features.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from stp3_b200.utils import geometry as G  # noqa: E402
from stp3_b200.utils import synthetic as syn  # noqa: E402

METRIC = "bev_frames_per_sec"
UNIT = "frames/s"
# SURVEY.md §8d / BASELINE.md §3: 2*MAC, unpadded channels, counted on the reference modules
GFLOP_TEMPORAL, GFLOP_DECODER, GFLOP_HEADS = 134.7, 59.3, 27.4
WORKLOADS = {
    "perceive": "perceive: 6 cam x 3 t x (28x60x48 frustum) -> lift-splat -> ego-warp + 3-D temporal block + DeepLab "
                "head -> BEV decoder heads (seg/ped/hdmap), 200x200x64 BEV (BASELINE configs[3]; EfficientNet trunk "
                "excluded on both arms)",
    "perceive_heads": "perceive_heads: trunk endpoints r3 (18x56x28x60) + r4 (18x160x14x30) per sample -> encoder heads "
                      "(DeepLabHead + UpsamplingConcat, features + depth logits) -> lift-splat (channels-last hand-off) -> "
                      "temporal block + DeepLab head -> decoder heads; perceive (BASELINE configs[3]) plus SURVEY.md row f1",
    "lift_splat": "lift_splat: 6 cam x 3 t x (28x60x48 frustum) -> 200x200x64 BEV, ego-warp + discount "
                  "(BASELINE configs[2] lift-splat stage)",
    "stress": "stress: 6 cam x 5 t x (28x60x96 frustum), C=128 -> lift-splat -> 4 temporal blocks + DeepLab head -> BEV "
              "decoder heads, 400x400 BEV (BASELINE configs[4]; a robustness / maximum-size run, not the headline metric)",
}
# the whole perception path runs for these workloads (the others stop after the lift-splat)
PERCEPTION = ("perceive", "stress", "perceive_heads")


def algorithmic_bytes_lift_splat(cfg, batch):
    """SURVEY.md §8d / BASELINE.md §3: read features + depth logits once, write every output frame once."""
    S, N, C, D = cfg.receptive_field, cfg.n_cameras, cfg.out_channels, cfg.n_depth
    Hf, Wf = cfg.feat_hw
    X, Y = cfg.bev_xy
    per_sample = 4 * S * N * Hf * Wf * (C + D) + 4 * S * C * X * Y + 4 * S * N * 25
    return per_sample * batch


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi sampled every 100 ms DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu_index)], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def trunk_endpoints(cfg, batch, seed):
    """Synthetic outputs of the (third-party, excluded) EfficientNet-b4 trunk: r3 (B,S,N,56,Hf,Wf), r4 (B,S,N,160,Hf/2,Wf/2),
    per-sample seeded like the other inputs."""
    Hf, Wf = cfg.feat_hw
    S, N = cfg.receptive_field, cfg.n_cameras
    r_lo, r_hi = [], []
    for i in range(batch):
        g = torch.Generator().manual_seed(1000 + seed + i)
        r_lo.append(syn.exact_gauss((1, S, N, 56, Hf, Wf), g))
        r_hi.append(syn.exact_gauss((1, S, N, 160, Hf // 2, Wf // 2), g))
    return torch.cat(r_lo), torch.cat(r_hi)


def make_problem(cfg, batch, seed, tilt_deg=0.0):
    """Batch of `batch` samples with per-sample seeds seed, seed+1, ...: sample i == lift_inputs(cfg, 1, seed+i), so
    the sample with seed 0 is the one the end-to-end reference fixture (tests/golden/e2e_perceive_*.npz) was recorded on."""
    inp = syn.stack_samples(cfg, [seed + i for i in range(batch)], tilt_deg=tilt_deg)
    cam_M, cam_t, ego_R, ego_t = G.lift_matrices(inp["intrinsics"], inp["extrinsics"], inp["future_egomotion"])
    xs, ys, ds = G.frustum_axes(cfg.final_dim, cfg.downsample, cfg.d_bound)
    res, start, dim = G.calculate_birds_eye_view_parameters(cfg.x_bound, cfg.y_bound, cfg.z_bound)
    return dict(inp=inp, mats=(cam_M, cam_t, ego_R, ego_t), axes=(xs, ys, ds), res=res, start=start, dim=dim,
                off=G.bev_offset(start, res))


DUMP_LIMIT_BYTES = 64 * 10**6


def dump_outputs(outputs, directory, limit=DUMP_LIMIT_BYTES):
    """--dump-outputs: every tensor of `outputs` (what the timed step returned) as <directory>/<name>.npy, float64 kept,
    anything else as float32.  When together they exceed `limit` bytes, each file holds a fixed sample of its array's
    flattened entries instead (indices drawn with seed 0 and sorted: the same for the same shapes in every run), sized
    so that all files fit.  Inputs are seeded, so two builds run with the same arguments can be compared file by file."""
    import numpy as np
    arrays = {}
    for name, t in outputs.items():
        if isinstance(t, torch.Tensor):
            t = t.detach()
            arrays[name] = (t if t.dtype == torch.float64 else t.float()).cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    budget = limit - 1024 * len(arrays)          # room for the .npy headers
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        if total > limit:
            keep = max(1, a.size * budget // total)
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(directory, f"{name}.npy"), a)


def build_model(device=None, lcfg=None):
    """Random-init (seeded, machine-independent) perception model; the trunk is not needed (inputs enter after it)."""
    from stp3_b200.config import get_cfg
    from stp3_b200.models.stp3 import STP3
    over = None
    if lcfg is not None and lcfg is not syn.CONFIGS["perceive"]:
        over = {"LIFT": {"X_BOUND": list(lcfg.x_bound), "Y_BOUND": list(lcfg.y_bound), "Z_BOUND": list(lcfg.z_bound),
                         "D_BOUND": list(lcfg.d_bound)},
                "TIME_RECEPTIVE_FIELD": lcfg.receptive_field, "MODEL": {"ENCODER": {"OUT_CHANNELS": lcfg.out_channels}}}
    cfg = get_cfg(over)
    with torch.no_grad():
        model = STP3(cfg, backbone=torch.nn.Identity())
        geo = {k: getattr(model, k).detach().clone() for k in ("frustum", "bev_resolution", "bev_start_position", "bev_dimension")}
        syn.init_exact(model, seed=0)
        for k, v in geo.items():
            getattr(model, k).copy_(v)
    model.eval()
    return model.to(device) if device is not None else model


# ------------------------------------------------------------------------------------------------ reference arm
def workload_config(args, cfg, world):
    """`config` of the JSON line: identical for the B200 arm and the reference arm (it names the workload)."""
    X, Y = cfg.bev_xy
    return {"workload": WORKLOADS[args.workload], "samples_per_gpu_per_step": args.batch,
            "global_batch": args.batch * world, "cameras": cfg.n_cameras, "frames": cfg.receptive_field, "bev": [X, Y],
            "channels": cfg.out_channels, "depth_bins": cfg.n_depth,
            "parallelism": f"dp{world} (batch sharded, no collective on the forward path)",
            "l2": "flushed between timed iterations (256 MiB write)", "weights": "random init, seeded",
            "rig": "level cameras (SURVEY.md 8d); roofline_lift_splat also times the 1-degree tilted rig"}


class ReferenceArm:
    """The reference's own CPU implementation of the path on the host cores.  kind "reference": the UNMODIFIED
    reference package (installed by oracle/build_ref.py into the git-ignored oracle/_ref/, or the checkout named by
    STP3_REFERENCE_ROOT) -- its STP3.get_geometry / projection_to_birds_eye_view, TemporalModel and Decoder -- imported
    through oracle/ref_loader.py; kind "port": the op-for-op CPU port under oracle/ when that install is absent."""

    def __init__(self, workload, cfg):
        from oracle import ref_loader
        self.workload, self.cfg = workload, cfg
        self.prob = make_problem(cfg, 1, seed=0)
        self.model = build_model(lcfg=cfg) if workload in PERCEPTION else None
        self.kind = "port"
        if ref_loader.reference_available():
            try:
                self._init_reference(ref_loader)
                self.kind = "reference"
            except Exception as e:              # e.g. a stub missing on this box: fall back to the port, say so
                print(f"reference import failed ({type(e).__name__}: {e}); timing the CPU port instead", file=sys.stderr)

    def _init_reference(self, ref_loader):
        from oracle.make_golden_dense import GATES_PERCEIVE
        self.ref = ref_loader.load_reference()
        cfg = self.cfg
        if self.model is not None:
            X, Y = cfg.bev_xy
            with torch.no_grad():
                self.ref_tm = self.ref.temporal_model.TemporalModel(cfg.out_channels + 6, cfg.receptive_field, (X, Y),
                                                                    start_out_channels=64).eval()
                self.ref_tm.load_state_dict(self.model.temporal_model.state_dict(), strict=True)
                self.ref_dec = self.ref.decoder.Decoder(64, 2, cfg.receptive_field, 2, GATES_PERCEIVE).eval()
                self.ref_dec.load_state_dict(self.model.decoder.state_dict(), strict=True)

    def step(self):
        """One sample through the path."""
        inp, cfg = self.prob["inp"], self.cfg
        with torch.no_grad():
            if self.kind == "reference":
                from oracle.make_golden import run_reference
                bev = run_reference(self.ref, cfg, inp)[3]
            else:
                from oracle import torch_port as TP
                xs, ys, ds = self.prob["axes"]
                bev = TP.lift_splat(inp["feat"], inp["depth_logits"], inp["intrinsics"], inp["extrinsics"],
                                    inp["future_egomotion"], xs, ys, ds, self.prob["res"], self.prob["start"],
                                    self.prob["dim"], cfg.discount)
            if self.workload == "lift_splat":
                return bev
            ego = inp["future_egomotion"]
            ego = torch.cat([torch.zeros_like(ego[:, :1]), ego[:, :-1]], 1)
            x = torch.cat([bev, ego.view(1, -1, 6, 1, 1).expand(1, ego.shape[1], 6, *bev.shape[-2:])], dim=2)
            if self.kind == "reference":
                return self.ref_dec(self.ref_tm(x))
            from oracle import torch_dense as TD
            return TD.decoder(TD.temporal_model(x, self.model.temporal_model), self.model.decoder)

    def pick_threads(self):
        """Thread count by timing the WHOLE step (after one warm-up step at the first candidate): the eager CPU path
        mixes tiny ops (which slow down when oversubscribed) with 194 GFLOP of convolutions (which want the cores)."""
        cores = os.cpu_count() or 1
        cands = sorted({min(cores, c) for c in (8, 16, 32, 64, cores)})
        torch.set_num_threads(cands[0])
        self.step()
        best, best_t, sweep = cands[0], float("inf"), {}
        for n in cands:
            torch.set_num_threads(n)
            t0 = time.perf_counter()
            self.step()
            sweep[n] = time.perf_counter() - t0
            if sweep[n] < best_t:
                best, best_t = n, sweep[n]
            elif sweep[n] > 1.5 * best_t:        # oversubscribed: more threads only get slower (128 threads: 20x)
                break
        torch.set_num_threads(best)
        return best, sweep

    def time(self, steps, warmup):
        threads, sweep = self.pick_threads()
        for _ in range(warmup):
            self.step()
        times = []
        for _ in range(steps):
            t0 = time.perf_counter()
            self.last = self.step()
            times.append(time.perf_counter() - t0)
        dt = statistics.median(times)
        return {"fps": 1.0 / dt, "dt": dt, "threads": threads, "times": times,
                "sweep": {str(k): round(v, 3) for k, v in sweep.items()}}

    def describe(self, r, steps, warmup):
        what = ("unmodified reference package (oracle/_ref or STP3_REFERENCE_ROOT via oracle/ref_loader.py): STP3.get_geometry + "
                "projection_to_birds_eye_view" + (" + TemporalModel + Decoder" if self.workload in PERCEPTION else "")
                if self.kind == "reference" else
                "op-for-op CPU port of the reference (oracle/torch_port.py" + (" + oracle/torch_dense.py)" if self.workload in PERCEPTION else ")"))
        return (f"1 sample (6 cam x {self.cfg.receptive_field} t) of the step's batch per timed step through the {what}; median of "
                f"{steps} step(s) after {warmup} warm-up; {r['threads']} of {os.cpu_count()} host threads = best of a whole-step "
                f"sweep {r['sweep']} s")


def run_reference_arm(args, cfg):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    steps, warmup = max(1, min(args.steps, 40)), min(args.warmup, 5)      # bounded: one sample takes seconds
    arm = ReferenceArm(args.workload, cfg)
    r = arm.time(steps, warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["fps"], "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": r["dt"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(args, cfg, world),
        "cpu_baseline": {"value": r["fps"], "unit": UNIT, "cores": r["threads"], "kind": arm.kind,
                         "sample": arm.describe(r, steps, warmup)},
        "e2e": {"value": r["fps"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if args.dump_outputs:
        dump_outputs(arm.last if isinstance(arm.last, dict) else {"bev": arm.last}, args.dump_outputs)
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ B200 arm
OUR_KERNELS = ("conv_igemm", "aspp_fused", "block_fused", "lift_splat", "bev_finalize", "bev_discount", "pool_reduce", "pool_bias", "small_linear",
               "upsample2x", "col_sum_reduce", "hilo", "spatial_sum", "clear_bytes", "lift_splat_bwd")


def count_launches(step_fn, dev):
    """Kernel launches of ONE step, observed with CUPTI (torch.profiler) in this run: (this repository's kernels,
    all kernels, device time of the conv_igemm family in ms).  Not inside the timed region."""
    try:
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.synchronize(dev)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step_fn()
            torch.cuda.synchronize(dev)
        ours = total = 0
        conv_us = 0.0
        for ev in prof.events():
            if "memcpy" in ev.name.lower() or "memset" in ev.name.lower():
                continue
            total += 1
            if any(k in ev.name for k in OUR_KERNELS):
                ours += 1
            if "conv_igemm" in ev.name or "aspp_fused" in ev.name or "block_fused" in ev.name:
                conv_us += float(getattr(ev, "device_time", 0.0) or getattr(ev, "cuda_time", 0.0) or 0.0)
        return ours, total, conv_us * 1e-3
    except Exception as e:                                  # CUPTI unavailable: say so instead of guessing
        print(f"launch count unavailable: {type(e).__name__}: {e}", file=sys.stderr)
        return None, None, None


def fast_path_fraction(ranks):
    """Share of (image, depth bin, image column) segments whose in-grid points all fall into ONE pillar -- the case the
    scatter kernel handles with 8 FFMA per LDS.128; the others take the segmented walk.  ranks (B,S,N,D,Hf,Wf) int32."""
    r = ranks.long()
    valid = r >= 0
    big = torch.where(valid, r, torch.full_like(r, 1 << 40)).amin(dim=-2)
    small = torch.where(valid, r, torch.full_like(r, -1)).amax(dim=-2)
    some = valid.any(dim=-2)
    uni = (big == small) & some
    return float(uni.sum().item()) / max(1.0, float(some.sum().item()))


def check_parity(res, cfg):
    """One replayed step's outputs for sample 0 (seed 0) against the end-to-end reference fixture (the unmodified
    reference and the fp64 oracle at the headline size).  Raises if the north-star bar (1e-3 of max) is missed."""
    import numpy as np
    path = os.path.join(ROOT, "tests", "golden", "e2e_perceive_level.npz")
    g = np.load(path)
    worst_o = worst_r = 0.0
    for k in ("segmentation", "pedestrian", "hdmap"):
        flat = res[k][0].detach().double().cpu().numpy().reshape(-1)
        got = flat[g[f"{k}_index"]]
        m = float(g[f"{k}_max"])
        worst_o = max(worst_o, float(np.abs(got - g[f"{k}_oracle"]).max()) / m)
        worst_r = max(worst_r, float(np.abs(got - g[f"{k}_ref"].astype(np.float64)).max()) / m)
    if not (worst_r <= 1e-3 and worst_o <= 1e-3):
        raise SystemExit(f"bench.py: the timed step's logits miss the parity bar: {worst_o:.2e} of max vs the fp64 oracle, "
                         f"{worst_r:.2e} vs the reference (bar 1e-3) -- refusing to report a throughput for wrong results")
    return {"fixture": "tests/golden/e2e_perceive_level.npz (reference end to end at 200x200, sample seed 0)",
            "max_err_vs_fp64_oracle": worst_o, "max_err_vs_reference_fp32": worst_r, "bar": 1e-3,
            "checked": "segmentation, pedestrian, hdmap logits of sample 0 of a replayed (graphed) step, 40k entries each"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="perceive", choices=list(WORKLOADS))
    ap.add_argument("--batch", type=int, default=4, help="samples per GPU per step (perceive config 4: 32 / 8 GPUs)")
    ap.add_argument("--rig", default="level", choices=["level", "tilted"],
                    help="camera rig of the timed workload (the lift-splat roofline always reports both)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from Python instead of one CUDA graph")
    ap.add_argument("--no-pipeline", action="store_true", help="e2e: serialise H2D, compute and D2H of every step")
    ap.add_argument("--no-extras", action="store_true", help="skip the sustained run, the second rig and the latency mode")
    ap.add_argument("--profiler-range", action="store_true",
                    help="bracket the resident timed steps with cudaProfilerStart/Stop (ncu --profile-from-start off)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the outputs of the last one as DIR/<name>.npy (rank 0's shard; "
                         f"at most {DUMP_LIMIT_BYTES // 10**6} MB in all, a fixed seeded sample of each output beyond that)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = syn.CONFIGS["stress" if args.workload == "stress" else "perceive"]
    if os.environ.get("STP3_BENCH_DUMP_AFTER"):      # debugging aid: Python stacks of every thread after N seconds, then exit
        import faulthandler
        faulthandler.dump_traceback_later(float(os.environ["STP3_BENCH_DUMP_AFTER"]), exit=True)

    if args.impl == "reference":
        run_reference_arm(args, cfg)
        return

    from stp3_b200 import ops
    # the host side of a step is a few hundred floats of calibration math (torch.inverse etc.); with the default
    # 64-128 intra-op threads every such call pays a multi-millisecond OpenMP wake-up, so keep the pool small
    torch.set_num_threads(min(4, os.cpu_count() or 1))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py (impl b200) needs a CUDA device; there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        # NCCL prints its version banner to STDOUT at the VERSION and WARN levels; rank 0's stdout is ONE JSON line
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
            del os.environ["NCCL_DEBUG"]
        dist.init_process_group("nccl", device_id=dev)
    W, K, b = max(args.warmup, 3), args.steps, args.batch
    perceive = args.workload in PERCEPTION
    tilt = 1.0 if args.rig == "tilted" else 0.0

    prob = make_problem(cfg, b, seed=rank * b, tilt_deg=tilt)   # every rank works on its own shard of the global batch
    inp = prob["inp"]
    host = {k: inp[k].pin_memory() for k in ("feat", "depth_logits", "intrinsics", "extrinsics", "future_egomotion")}
    host_mats = [m.pin_memory() for m in prob["mats"]]
    xs, ys, ds = (a.to(dev) for a in prob["axes"])
    heads = args.workload == "perceive_heads"
    if heads:        # the step enters at the trunk endpoints: they take the place of (feat, depth_logits) everywhere below
        r_lo, r_hi = trunk_endpoints(cfg, b, rank * b)
        host["feat"], host["depth_logits"] = r_lo.pin_memory(), r_hi.pin_memory()
    d_feat, d_depth = host["feat"].to(dev), host["depth_logits"].to(dev)
    d_mats = [m.to(dev) for m in host_mats]
    X, Y = cfg.bev_xy
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2
    model = build_model(dev, cfg) if perceive else None
    graphed = None
    if perceive and not args.no_graph:
        from stp3_b200.models.stp3 import GraphedPerception
        graphed = GraphedPerception(model, b, cfg.n_cameras, dev, entry="heads" if heads else "lift")
        graphed(d_feat, d_depth, inp["intrinsics"], inp["extrinsics"], inp["future_egomotion"])   # fill the static inputs
    if perceive:
        host_out = {"segmentation": torch.empty((b, cfg.receptive_field, 2, X, Y)).pin_memory(),
                    "pedestrian": torch.empty((b, cfg.receptive_field, 2, X, Y)).pin_memory(),
                    "hdmap": torch.empty((b, 4, X, Y)).pin_memory()}
    else:
        out = torch.empty((b, cfg.receptive_field, cfg.out_channels, X, Y), dtype=torch.float32, device=dev)
        host_out = {"bev": torch.empty(out.shape, dtype=torch.float32).pin_memory()}

    def step_resident():
        with torch.no_grad():
            if graphed is not None:
                graphed.graph.replay()            # inputs already resident in the graph's static buffers
                return graphed.out
            if perceive:
                fwd = model.forward_trunk_features if heads else model.forward_features
                return fwd(d_feat, d_depth, inp["intrinsics"], inp["extrinsics"], inp["future_egomotion"])
            ops.lift_splat(d_feat, d_depth, *d_mats, xs, ys, ds, prob["off"], prob["res"], prob["dim"], cfg.discount, out=out)
            return {"bev": out}

    def step_e2e():
        """The call a user makes: host (pinned) inputs in, host results out."""
        with torch.no_grad():
            if graphed is not None:
                res = graphed(host["feat"], host["depth_logits"], host["intrinsics"], host["extrinsics"],
                              host["future_egomotion"])
            elif perceive:
                f = host["feat"].to(dev, non_blocking=True)
                d = host["depth_logits"].to(dev, non_blocking=True)
                fwd = model.forward_trunk_features if heads else model.forward_features
                res = fwd(f, d, host["intrinsics"], host["extrinsics"], host["future_egomotion"])
            else:
                f = host["feat"].to(dev, non_blocking=True)
                d = host["depth_logits"].to(dev, non_blocking=True)
                mats = [m.to(dev, non_blocking=True) for m in host_mats]
                ops.lift_splat(f, d, *mats, xs, ys, ds, prob["off"], prob["res"], prob["dim"], cfg.discount, out=out)
                res = {"bev": out}
            for k, t in host_out.items():
                t.copy_(res[k], non_blocking=True)

    from stp3_b200 import parallel

    def barrier():
        parallel.barrier()
        torch.cuda.synchronize()

    last = {}

    def timed(fn, steps):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        issued = [0]
        stop = None
        if os.environ.get("STP3_BENCH_MONITOR") and steps > 50:     # hang diagnosis: device progress once a second
            stop = threading.Event()

            def watch():
                torch.cuda.set_device(dev)
                while not stop.wait(1.0):
                    n = issued[0]
                    done = sum(1 for i in range(n) if evs[i][1].query())
                    _progress(f"monitor: issued {n}/{steps}, finished on device {done}")
            threading.Thread(target=watch, daemon=True).start()
        for s, e in evs:
            flush.zero_()                      # evict L2 between timed iterations (not timed)
            s.record(); last["out"] = fn(); e.record()
            issued[0] += 1
        barrier()
        if stop is not None:
            stop.set()
        return parallel.max_over_ranks(sum(s.elapsed_time(e) for s, e in evs), dev)

    def timed_pipelined(pipe, steps):
        """End-to-end throughput with the copies of neighbouring steps overlapped with compute (PipelinedPerception):
        every step still moves its inputs host->device and its results device->host inside the timed region."""
        args_h = (host["feat"], host["depth_logits"], host["intrinsics"], host["extrinsics"], host["future_egomotion"])
        pipe.between_steps = flush.zero_            # L2 eviction between steps, on the compute stream
        for _ in range(3):
            pipe.submit(*args_h); pipe.collect()
        barrier()
        t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
        t0.record()
        for k in range(steps):
            pipe.submit(*args_h)
            if k >= 1:
                pipe.collect()
        pipe.collect()
        t1.record()
        barrier()
        return parallel.max_over_ranks(t0.elapsed_time(t1), dev)

    _progress("setup done")
    for _ in range(W):
        step_resident()
    # parity gate: the step that is about to be timed must produce the reference's logits
    parity = None
    if rank == 0 and args.workload == "perceive" and args.rig == "level":
        res0 = step_resident()
        torch.cuda.synchronize()
        parity = check_parity(res0, cfg)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    if args.profiler_range:
        torch.cuda.cudart().cudaProfilerStart()
    _progress("timing resident steps")
    total_ms = timed(step_resident, K)
    _progress("timing e2e")
    if args.profiler_range:
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStop()
    if args.dump_outputs and rank == 0:
        dump_outputs(last["out"], args.dump_outputs)
    e2e_mode = "serial: H2D -> compute -> D2H per step"
    if graphed is not None and not args.no_pipeline:
        from stp3_b200.models.stp3 import PipelinedPerception
        with torch.no_grad():
            pipe = PipelinedPerception(model, b, cfg.n_cameras, depth=2, device=dev, entry="heads" if heads else "lift")
        e2e_ms = timed_pipelined(pipe, K)
        e2e_mode = "pipelined (depth 2): copies of steps i-1 / i+1 overlap the CUDA graph of step i"
    else:
        for _ in range(2):
            step_e2e()
        e2e_ms = timed(step_e2e, K)
    clocks = sampler.stop() if rank == 0 else None
    # the host link: what one pinned host->device copy of the step's inputs achieves on this box (the e2e figure cannot beat it)
    link_gbs = None
    if rank == 0:
        big = host["feat"]
        dst = torch.empty_like(big, device=dev)
        for _ in range(2):
            dst.copy_(big, non_blocking=True)
        a, c = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(5):
            dst.copy_(big, non_blocking=True)
        c.record()
        torch.cuda.synchronize()
        link_gbs = 5 * big.numel() * big.element_size() / (a.elapsed_time(c) * 1e-3) / 1e9
        del dst

    # Everything after this point is explanatory (sustained run, per-stage graphs, launch count, rooflines, CPU baseline,
    # latency mode).  The contract line exists from here on; a watchdog prints it as it stands if the rest does not come
    # back (a stuck device or collective), so a late failure never costs the headline measurement.
    if rank == 0:
        frames = b * world
        h2d = sum(host[k].numel() * host[k].element_size() for k in ("feat", "depth_logits"))
        h2d += sum(t.numel() * t.element_size() for t in host_mats)
        d2h = sum(t.numel() * 4 for t in host_out.values())
        _LINE["line"] = {
            "metric": METRIC, "value": frames / (total_ms / K * 1e-3), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 (dense layers: bf16x3 split products, fp32 accumulate)" if perceive else "f32",
            "data": "synthetic", "config": workload_config(args, cfg, world),
            "clocks": clocks,
            "e2e": {"value": frames / (e2e_ms / K * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms / K,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "mode": e2e_mode,
                    "host_link_h2d_gbs": link_gbs,
                    "h2d_ms_per_step_at_link_rate": (h2d / (link_gbs * 1e9) * 1e3) if link_gbs else None},
            "parity_checked": parity is not None, "parity": parity,
        }
    dog = extras_watchdog(float(os.environ.get("STP3_BENCH_EXTRAS_LIMIT", "600" if world == 1 else "300")), rank)

    _progress("sustained")
    # sustained figure: the same resident step back to back for >= 2 s (the 20-step region above is a ~65 ms burst)
    sustained = None
    if not args.no_extras:
        n_sus = max(K, int(2000.0 / max(total_ms / K, 1e-3)) + 1)
        sus_ms = timed(step_resident, n_sus)
        sustained = {"value": b * world / (sus_ms / n_sus * 1e-3), "unit": UNIT, "steps": n_sus,
                     "ms_per_step": sus_ms / n_sus, "seconds": sus_ms * 1e-3}

    _progress("stages")
    # per-stage device time: each stage captured as its own CUDA graph (no launch gaps), timed with CUDA events
    stage_ms = {}
    if perceive:
        stage_ms = time_stages(model, graphed.static if graphed is not None else None, d_feat, d_depth, inp, flush, dev,
                               heads=heads)
    ours, total_launches, conv_ms_prof = count_launches(step_resident, dev)

    _progress("rigs")
    # the lift-splat on both rigs (level cameras = SURVEY 8d; 1 degree of roll / pitch / yaw error per camera)
    rigs = {}
    if not args.no_extras and args.workload in ("perceive", "lift_splat"):
        for name, tdeg in (("level", 0.0), ("tilted_1deg", 1.0)):
            pr = make_problem(cfg, b, seed=rank * b, tilt_deg=tdeg)
            f, d = pr["inp"]["feat"].to(dev), pr["inp"]["depth_logits"].to(dev)
            mats = [m.to(dev) for m in pr["mats"]]
            o = torch.empty((b, cfg.receptive_field, cfg.out_channels, X, Y), dtype=torch.float32, device=dev)
            ws = ops.Workspace()

            def ls():
                ops.lift_splat(f, d, *mats, xs, ys, ds, pr["off"], pr["res"], pr["dim"], cfg.discount, out=o, workspace=ws)
            _, ranks = ops.lift_splat(f[:1], d[:1], *[m[:1] for m in mats], xs, ys, ds, pr["off"], pr["res"], pr["dim"],
                                      cfg.discount, return_ranks=True)
            fpf = fast_path_fraction(ranks)
            for _ in range(3):
                ls()
            ms = timed(ls, 10) / 10
            rigs[name] = {"ms": ms, "fast_path_fraction": fpf}
            del f, d, o

    _progress("main measurements done")
    # latency mode (north_star): global batch 1 < #GPUs, camera frames sharded, ONE all-gather of raw BEV frames
    run_latency = world > 1 and perceive and not args.no_extras

    if rank == 0:
        ms_per_step = total_ms / K
        pk = peaks()
        alg = algorithmic_bytes_lift_splat(cfg, b)
        ls_ms = stage_ms.get("lift_splat", ms_per_step)
        roof_ls = {"bound": "hbm", "kernel": "lift-splat (scatter + finalize, one C-ABI call)",
                   "achieved": alg / (ls_ms * 1e-3) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                   "frac": alg / (ls_ms * 1e-3) / 1e9 / pk["hbm_gbs"], "peak_source": pk["source"],
                   "traffic": TRAFFIC["lift_splat"]["bytes_per_sample"] * b if args.workload == "perceive" else None,
                   "traffic_source": TRAFFIC["lift_splat"]["source"],
                   "algorithmic_bytes_per_step": alg, "ms": ls_ms, "rig": args.rig}
        for name, r in rigs.items():
            r["achieved"] = alg / (r["ms"] * 1e-3) / 1e9
            r["frac"] = r["achieved"] / pk["hbm_gbs"]
        if rigs:
            roof_ls["rigs"] = rigs
        line = _LINE["line"]
        line["sustained"] = sustained
        if args.rig != "level":
            line["config"]["rig"] = "tilted: every camera 1 degree off level (timed workload)"
        # launches inside the resident + e2e timed regions (2K steps), counted by CUPTI on one step of this run
        line["gpu_launches"] = 2 * K * ours if ours is not None else None
        line["launches_per_step"] = {"ours": ours, "all_kernels": total_launches, "how": "torch.profiler (CUPTI), one replayed step of this run"}
        if perceive:
            dense_ms = stage_ms.get("temporal_model", 0.0) + stage_ms.get("decoder", 0.0) + stage_ms.get("encoder_heads", 0.0)
            # the flop count was taken on the reference modules for the perceive configuration only
            flops = (GFLOP_TEMPORAL + GFLOP_DECODER + (GFLOP_HEADS if heads else 0.0)) * 1e9 * b \
                if args.workload in ("perceive", "perceive_heads") else None
            ach = flops / (dense_ms * 1e-3) / 1e12 if flops and dense_ms > 0 else None
            line["stage_ms"] = stage_ms
            line["roofline"] = {"bound": "tensor", "kernel": "conv_igemm_kernel<BN, PAIR, STACK> + aspp_fused_kernel + block_fused_kernel (temporal model + decoder)",
                                "achieved": ach, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
                                "frac": ach / pk["bf16_tflops_sustained"] if ach else None, "peak_source": pk["source"],
                                "traffic": TRAFFIC["conv"]["bytes_per_sample"] * b if args.workload == "perceive" else None,
                                "traffic_source": TRAFFIC["conv"]["source"],
                                "algorithmic_flops_per_step": flops, "ms": dense_ms,
                                "conv_kernel_ms_cupti": conv_ms_prof,
                                "note": "algorithmic 2*MAC flops of the fp32 layers; the kernel issues 3 bf16 MMAs per product (hi*hi+hi*lo+lo*hi) to hold 1e-3 parity: "
                                        "profiles/r02_precision_plan.txt shows every 2-MMA form missing the bar"}
            line["roofline_lift_splat"] = roof_ls
        else:
            line["roofline"] = roof_ls
        if perceive and os.environ.get("STP3_TUNE_REPORT"):
            from stp3_b200 import dense
            for desc, times in dense.TUNE_LOG:
                print("TUNE", desc.ljust(44), "  ".join(f"{k}:{v * 1e3:7.1f}us" for k, v in times.items()), file=sys.stderr)
        if world == 1 and not args.no_cpu_baseline:
            arm = ReferenceArm(args.workload, cfg)
            r = arm.time(3, 1)
            line["cpu_baseline"] = {"value": r["fps"], "unit": UNIT, "cores": r["threads"], "kind": arm.kind,
                                    "sample": arm.describe(r, 3, 1)}
    # the latency mode runs LAST (under the same watchdog): whatever happens in it (a collective that never returns on
    # some topology), rank 0 still prints its ONE JSON line and every rank exits 0
    if run_latency:
        if rank == 0:
            _LINE["line"]["latency_mode"] = {"unavailable": "did not finish (watchdog)"}
        try:
            latency = time_latency_mode(model, cfg, dev, flush, rank, world)
        except Exception as e:            # never let the extra mode cost the main line
            latency = {"unavailable": f"{type(e).__name__}: {e}"[:300]}
        if rank == 0:
            _LINE["line"]["latency_mode"] = latency
    dog.cancel()
    if rank == 0:
        print(json.dumps(_LINE["line"]), flush=True)
    if world > 1:
        import torch.distributed as dist
        bye = threading.Timer(30.0, os._exit, args=(0,))      # the line is out: a stuck teardown must not keep the job alive
        bye.daemon = True
        bye.start()
        try:
            dist.destroy_process_group()
        except Exception:
            pass
        bye.cancel()


_LINE = {}


def extras_watchdog(limit_s, rank, exit_fn=os._exit, out=None):
    """Timer armed once the contract line exists (_LINE["line"] on rank 0): if the explanatory part of the run has not
    cancelled it after `limit_s` seconds, rank 0 prints the line as it stands -- marked -- and every rank exits 0."""
    def give_up():
        if rank == 0:
            _LINE["line"]["extras"] = {"unavailable": f"timed out after {limit_s:.0f} s (watchdog): the keys after "
                                                      "'parity' are missing or partial"}
            print(json.dumps(_LINE["line"]), file=out or sys.stdout, flush=True)
        exit_fn(0)
    dog = threading.Timer(limit_s, give_up)
    dog.daemon = True
    dog.start()
    return dog

# DRAM traffic (dram__bytes_read.sum + dram__bytes_write.sum) cannot be measured outside ncu: static values from the
# committed `ncu --set full` captures, per sample
TRAFFIC = {
    "lift_splat": {"bytes_per_sample": int(263.6e6 / 4), "source": "static: profiles/r02_ncu_liftsplat_v2_summary.txt (scatter 108.7 MB + finalize 155.0 MB, B=4)"},
    "conv": {"bytes_per_sample": int(2464e6 / 4), "source": "static: profiles/r02_ncu_conv_v3_summary.txt (the temporal model's 6 tensor-core launches incl. the four B2B launches + the first 10 decoder convs of 35, cold cache, B=4)"},
}


def _progress(msg):
    if os.environ.get("STP3_BENCH_PROGRESS"):
        print(f"[bench rank {os.environ.get('RANK', '0')} +{time.time() % 1000:.1f}s] {msg}", file=sys.stderr, flush=True)


def time_latency_mode(model, cfg, dev, flush, rank, world, reps=10):
    """Global batch 1 on `world` GPUs: STP3.forward_features_frame_sharded (each rank splats its share of the B*S camera
    frames, ONE NCCL all-gather of raw BEV frames, replicated temporal model + decoder) next to the unsharded forward
    of the same sample on every rank.  Eager launches on both sides (NCCL is not captured in a graph here); device
    times by CUDA events, max over ranks."""
    import torch.distributed as dist
    from stp3_b200 import parallel
    inp = syn.lift_inputs(cfg, 1, seed=0)
    a = (inp["feat"].to(dev), inp["depth_logits"].to(dev), inp["intrinsics"], inp["extrinsics"], inp["future_egomotion"])
    X, Y = cfg.bev_xy
    S, C = cfg.receptive_field, cfg.out_channels
    with torch.no_grad():
        _progress("latency: eager nccl warm-up")
        for _ in range(3):
            sh = model.forward_features_frame_sharded(*a)
            full = model.forward_features(*a)
        torch.cuda.synchronize()
        _progress("latency: eager nccl timed")
        err = max(float((sh[k] - full[k]).abs().max() / full[k].abs().max()) for k in ("segmentation", "pedestrian", "hdmap"))

        def timed(fn):
            tot = 0.0
            for _ in range(reps):
                flush.zero_()
                dist.barrier()
                torch.cuda.synchronize()
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record(); fn(); e.record()
                torch.cuda.synchronize()
                tot += s.elapsed_time(e)
            return parallel.max_over_ranks(tot / reps, dev)
        ms_sharded = timed(lambda: model.forward_features_frame_sharded(*a))
        ms_full = timed(lambda: model.forward_features(*a))
        # the all-gather fused into the finalize kernel's epilogue (peer stores over NVLink, symmetric memory)
        peer = None
        try:
            _progress("latency: peer warm-up (symmetric memory rendezvous)")
            for _ in range(3):
                shp = model.forward_features_frame_sharded(*a, gather="peer")
            torch.cuda.synchronize()
            err_p = max(float((shp[k] - full[k]).abs().max() / full[k].abs().max()) for k in ("segmentation", "pedestrian", "hdmap"))
            ms_peer = timed(lambda: model.forward_features_frame_sharded(*a, gather="peer"))
            # the lift stage alone, both ways: splat own frames + exchange + discount
            from stp3_b200 import ops
            h = {k: v.to(dev) for k, v in model.prepare_inputs(a[2], a[3], a[4]).items()}
            off, res, dim = model._bev_host()
            f0s, fcs = parallel.shard_batch(S, rank, world)
            pf = model.__dict__["_peer_frames"][1]

            def lift_nccl():
                r = ops.lift_splat_frames(a[0], a[1], h["cam_M"], h["cam_t"], h["ego_R"], h["ego_t"], *model._axes(), off, res, dim,
                                          f0s, fcs, workspace=model._ws) if fcs > 0 else torch.empty((0, X, Y, C), device=dev)
                ops.bev_discount(parallel.all_gather_frames(r, S).view(1, S, X, Y, C), float(model.discount))

            def lift_peer():
                pf.barrier()
                if fcs > 0:
                    ops.lift_splat_frames(a[0], a[1], h["cam_M"], h["cam_t"], h["ego_R"], h["ego_t"], *model._axes(), off, res, dim,
                                          f0s, fcs, workspace=model._ws, peer_ptrs=pf.ptrs)
                pf.barrier()
                ops.bev_discount(pf.buf.view(1, S, X, Y, C), float(model.discount))
            _progress("latency: lift stage both ways")
            for _ in range(2):
                lift_nccl(); lift_peer()
            # both as ONE CUDA graph (what a latency-critical deployment would run): unsharded vs frame-sharded + peer stores
            graphed = None
            _progress("latency: graph capture")
            try:
                from stp3_b200.models.stp3 import GraphedPerception
                g_full = GraphedPerception(model, 1, cfg.n_cameras, dev, entry="lift")
                g_shard = GraphedPerception(model, 1, cfg.n_cameras, dev, entry="sharded")
                for g in (g_full, g_shard):
                    g(a[0], a[1], a[2], a[3], a[4])
                torch.cuda.synchronize()
                err_g = max(float((g_shard.out[k] - g_full.out[k]).abs().max() / g_full.out[k].abs().max())
                            for k in ("segmentation", "pedestrian", "hdmap"))
                graphed = {"ms_unsharded": timed(g_full.graph.replay), "ms_frame_sharded_peer_stores": timed(g_shard.graph.replay),
                           "parity_vs_unsharded": parallel.max_over_ranks(err_g, dev) <= 1e-4}
            except Exception as e:
                graphed = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
            peer = {"ms": ms_peer, "graphed": graphed, "parity_vs_unsharded": parallel.max_over_ranks(err_p, dev) <= 1e-4,
                    "lift_stage_ms_nccl_allgather": timed(lift_nccl), "lift_stage_ms_peer_stores": timed(lift_peer),
                    "how": "finalize epilogue stores each frame into every rank's symmetric-memory buffer (st.global on peer "
                           "addresses), two device-side barriers, no collective launch"}
        except Exception as e:      # no P2P / symmetric memory on this box: report, keep the NCCL numbers
            peer = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
        f0, fc = parallel.shard_batch(S, rank, world)
        raw = torch.zeros((fc, X, Y, C), dtype=torch.float32, device=dev)
        ms_ag = timed(lambda: parallel.all_gather_frames(raw, S))
        cmax = max(parallel.shard_batch(S, r, world)[1] for r in range(world))
    err = parallel.max_over_ranks(err, dev)
    return {"global_batch": 1, "frames_per_rank": [parallel.shard_batch(S, r, world)[1] for r in range(world)],
            "ms": ms_sharded, "ms_unsharded_same_sample": ms_full, "allgather_ms": ms_ag,
            "bytes": int(world * cmax * X * Y * C * 4), "bytes_note": "all_gather_into_tensor output per rank (padded to equal shards)",
            "parity_vs_unsharded": err <= 1e-4, "max_rel_err_vs_unsharded": err, "launch": "eager (Python/ctypes launches on both sides)",
            "fused_allgather": peer}


def time_stages(model, static, d_feat, d_depth, inp, flush, dev, reps=5, heads=False):
    """GPU time of the stages of STP3.forward_device (and the encoder heads before it), each replayed as its own CUDA graph."""
    from stp3_b200 import dense, ops
    from stp3_b200.models.stp3 import STP3  # noqa: F401
    if static is None:
        h = {k: v.to(dev) for k, v in model.prepare_inputs(inp["intrinsics"], inp["extrinsics"], inp["future_egomotion"]).items()}
        static = dict(**({"r_lo": d_feat, "r_hi": d_depth} if heads else {"feat": d_feat, "depth_logits": d_depth}), **h)
    B, S = static["cam_M"].shape[:2]
    X, Y = model.bev_size
    C = model.encoder_out_channels
    off, res, dim = model._bev_host()
    planes = torch.empty((2, B, S, X, Y, C), dtype=torch.bfloat16, device=dev)
    hold = {}

    def enc_heads():
        r_lo, r_hi = static["r_lo"], static["r_hi"]
        n = r_lo.shape[2]
        f, d = model.encoder.heads_f32(r_lo.view(B * S * n, *r_lo.shape[3:]), r_hi.view(B * S * n, *r_hi.shape[3:]),
                                       channels_last=True)
        hold["feat"], hold["depth"] = f.view(B, S, n, *f.shape[1:]), d.view(B, S, n, *d.shape[1:])

    def lift():
        f = hold["feat"] if heads else static["feat"]
        d = hold["depth"] if heads else static["depth_logits"]
        r = ops.lift_splat(f, d, static["cam_M"], static["cam_t"], static["ego_R"],
                           static["ego_t"], *model._axes(), off, res, dim, float(model.discount), workspace=model._ws,
                           out_hilo=planes, pool_sum=True, feat_channels_last=heads)
        hold["sums"] = r[1].view(B * S, C)

    def temporal():
        hold["states"] = model.temporal_model.forward_hl(dense.HL(planes[0], planes[1], C), const=static["const"],
                                                         sums=hold["sums"])

    def decoder():
        hold["out"] = model.decoder.forward_hl(hold["states"])

    out = {}
    with torch.no_grad():
        stages = (("lift_splat", lift), ("temporal_model", temporal), ("decoder", decoder))
        if heads:
            stages = (("encoder_heads", enc_heads),) + stages
        for name, fn in stages:
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                fn()
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                fn()
            tot = 0.0
            for _ in range(reps):
                flush.zero_()
                a, c = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); g.replay(); c.record()
                torch.cuda.synchronize()
                tot += a.elapsed_time(c)
            out[name] = tot / reps
    return out


if __name__ == "__main__":
    main()
