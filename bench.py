#!/usr/bin/env python
"""bench.py -- DRRs/sec fwd+bwd (512^3 CT -> 256^2 detector) and achieved algorithmic HBM GB/s vs the B200 peak.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]

A "step" is one pass of the hot path over one batch of synthetic poses: Siddon forward (line integrals of
`--batch` poses through a 512^3 fp32 volume onto a 256^2 detector) + Siddon backward (gradients w.r.t. the ray
end points / ray lengths, i.e. the pose-gradient path of 2D/3D registration).  Since every pixel depends on one ray
only, the forward walk also accumulates the ray's 6 end-point sensitivities (they do not depend on the upstream
gradient) and the backward pass is an elementwise kernel: one walk per step instead of two, same outputs.
Reported on ONE JSON line:

  value      whole-job DRRs/s with the rays already resident in HBM (kernels only, CUDA-event timed)
  e2e        the same metric through the public module call `DRR(rot, xyz)` + backward, with the pose parameters
             coming from pinned HOST memory every step and the images / loss / pose gradients copied back
  roofline   algorithmic bytes of the dominant kernel / its CUDA-event duration vs the measured HBM peak
  cpu_baseline  the CPU oracle (C port of the reference algorithm, OpenMP) on a bounded sample, rank 0 only

With N > 1 (torchrun, one rank per GPU, NCCL) the poses are sharded across ranks (weak scaling: `--batch` poses per
GPU), the volume is replicated, and every step ends with ONE all_gather of the image stack.
`--impl reference` times the CPU oracle port instead (the reference is pure Python and cannot travel to the GPU
box; SURVEY.md 8c) with all host threads, on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

VOL = 512
DET = 256
METRIC = "DRRs/sec fwd+bwd (512^3 CT -> 256^2 det)"
WORKLOAD = "siddon fwd+bwd(pose), 512^3 fp32 CT -> 256^2 detector"
HBM_FALLBACK_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback
# dram__bytes_read.sum + dram__bytes_write.sum per launch from `ncu --set full` captures of the default workload
# (16 poses, 512^3 -> 256^2): profiles/r01_fwd_slab_B16_ncu_summary.txt and gpurun capture of the backward kernel.
# Only quoted when the run uses that workload; otherwise null.
NCU_TRAFFIC_SOURCE = ("not measured by this run: dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of "
                      "the same command (profiles/r02_siddon_sens_slab_ncu_summary.txt, captured 2026-09-24 on a B200 of this pool); null off the default workload")
NCU_TRAFFIC_BYTES = {"siddon_fwd_slab_kernel": 1.05e9 + 0.02e9, "siddon_bwd_slab_kernel": 2.26e9 + 0.09e9,
                     "siddon_sens_slab_kernel": 1.4126e9 + 0.1360e9}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=16, help="poses per GPU per step")
    ap.add_argument("--vol", type=int, default=VOL)
    ap.add_argument("--det", type=int, default=DET)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="report the eager end-to-end step only")
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary BASELINE configs / reference-on-GPU legs")
    ap.add_argument("--workload", default="metric", choices=["metric", "config4"],
                    help="metric = BASELINE.json's metric workload (default); config4 = 512^3 -> 1024^2, 256 poses sharded over the GPUs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (rank 0's shard) as DIR/<name>.npy, float32, at most 64 MB in all")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, arrays):
    """Saves each tensor of `arrays` as out_dir/<name>.npy in float32.  When together they exceed DUMP_BYTES, every tensor
    keeps the same fraction of its elements, flattened, at positions drawn from a fixed seed: the positions depend only on
    the tensor sizes, so two builds of the project run with the same arguments can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    total = sum(4 * t.numel() for t in arrays.values())
    keep = min(1.0, (DUMP_BYTES - 1024 * len(arrays)) / total)  # 1 KB per file for the .npy header
    for name, t in arrays.items():
        t = t.detach().float()
        if keep < 1.0:
            flat = t.reshape(-1)
            n = max(1, int(flat.numel() * keep))
            pos = torch.randint(flat.numel(), (n,), generator=torch.Generator().manual_seed(0)).sort().values
            t = flat[pos.to(flat.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples nvidia-smi SM clocks / throttle reasons in the background during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._thr = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) == 6:
                    self.rows.append(parts)
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._thr.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(self.rows)}


# ---------------------------------------------------------------------------------------------------------------
# CPU oracle legs (cpu_baseline and --impl reference)
# ---------------------------------------------------------------------------------------------------------------
def make_host_rays(vol_n, det_n, batch, seed):
    """Rays of `batch` synthetic poses in voxel coordinates, computed with the host-side geometry (CPU torch)."""
    from diffdrr_b200 import DRR, synthetic
    from diffdrr_b200.pose import convert

    subj = synthetic.make_subject(torch.zeros(1, 1, 1, 1))
    subj.volume.affine = synthetic.make_affine(vol_n)
    drr = DRR(subj, **synthetic.detector_kwargs(det_n))
    rot, xyz = synthetic.make_poses(batch, seed=seed)
    with torch.no_grad():
        src, tgt = drr.detector(convert(rot, xyz, parameterization="euler_angles", convention="ZXY"), None)
        raylen = (tgt - src).norm(dim=-1).unsqueeze(1)
        src, tgt = drr.affine_inverse(src), drr.affine_inverse(tgt)
    return src.numpy(), tgt.numpy(), raylen.numpy()


def host_threads() -> int:
    """All host cores, whatever OMP_NUM_THREADS says (torchrun exports OMP_NUM_THREADS=1 to every rank)."""
    return os.cpu_count() or 1


def cpu_model() -> str:
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def load_reference():
    """The UNMODIFIED reference renderers (pip-installed into baseline/_ref, git-ignored, travels with the snapshot).
    diffdrr/renderers.py imports only torch; returns None when the install is absent (the port is timed instead)."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "diffdrr")):
        return None
    import importlib.util

    spec = importlib.util.spec_from_file_location("_ref_diffdrr_renderers", os.path.join(ref_dir, "diffdrr", "renderers.py"))
    mod = importlib.util.module_from_spec(spec)
    try:
        spec.loader.exec_module(mod)
    except Exception:
        return None
    return mod


def cpu_oracle_time(vol_n, det_n, n_drr, repeats, threads):
    """Seconds per fwd+bwd DRR of the C oracle (reference algorithm: all planes merged/sorted per ray, fp32)."""
    from diffdrr_b200 import synthetic
    from oracle import oracle

    oracle.set_threads(threads)
    vol = synthetic.make_volume(vol_n, "rand", seed=0)
    src, tgt, raylen = make_host_rays(vol_n, det_n, max(n_drr, 2), seed=0)
    src, tgt, raylen = src[:n_drr], tgt[:n_drr], raylen[:n_drr]
    gout = np.ones_like(raylen)
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        oracle.siddon_fwd(vol, src, tgt, raylen, dtype=np.float32)
        oracle.siddon_bwd(vol, src, tgt, raylen, gout, want_vol=False, dtype=np.float32)
        times.append(time.perf_counter() - t0)
    return times


class ReferenceRun:
    """reference renderers.py:34-91 (`Siddon.forward`, unmodified) + autograd w.r.t. the ray end points, on a sample of the
    workload's rays: one pose of the synthetic batch, `n_rays` detector pixels spread evenly over the detector."""

    def __init__(self, ref_mod, vol_n, det_n, device="cpu"):
        from diffdrr_b200 import synthetic

        self.device = torch.device(device)
        self.siddon = ref_mod.Siddon().to(self.device)
        self.vol = torch.as_tensor(synthetic.make_volume(vol_n, "rand", seed=0)).to(self.device)
        src, tgt, raylen = make_host_rays(vol_n, det_n, 2, seed=0)
        self.src, self.tgt, self.raylen = (torch.as_tensor(x[:1]).to(self.device) for x in (src, tgt, raylen))
        self.n_total = self.tgt.shape[1]

    def step(self, n_rays, img_out=None):
        sel = torch.linspace(0, self.n_total - 1, n_rays, device=self.device).long()
        src = self.src.clone().requires_grad_(True)
        tgt = self.tgt[:, sel].clone().requires_grad_(True)
        raylen = self.raylen[:, :, sel]
        if self.device.type == "cuda":
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        img = self.siddon(self.vol, src, tgt, raylen)
        img.sum().backward()
        if self.device.type == "cuda":
            torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        assert torch.isfinite(tgt.grad).all()
        if img_out is not None:
            img_out.append((sel.cpu().numpy(), img.detach().cpu().numpy()))
        return dt


def best_reference_threads(run, n_rays=1024):
    """PyTorch's CPU kernels stop scaling long before 128 threads on this shape (measured on the GPU box: 128 threads are
    ~20x SLOWER than 8): time a small sample at a few thread counts and keep the fastest, so that the baseline is the
    reference at its best on these host cores."""
    best, best_t = host_threads(), float("inf")
    tried = {}
    for n in sorted({host_threads(), max(1, host_threads() // 2), max(1, host_threads() // 4), 32, 16, 8}, reverse=True):
        if n > host_threads():
            continue
        torch.set_num_threads(n)
        run.step(n_rays)
        t = min(run.step(n_rays), run.step(n_rays))
        tried[n] = t
        if t < best_t:
            best, best_t = n, t
    torch.set_num_threads(best)
    return best, tried


def cpu_reference_sample(vol_n, det_n, budget_s, min_runs=5):
    """Times the unmodified reference on the host cores within ~budget_s seconds.  Returns None without baseline/_ref."""
    ref_mod = load_reference()
    if ref_mod is None:
        return None
    run = ReferenceRun(ref_mod, vol_n, det_n)
    threads, tried = best_reference_threads(run)
    n_rays = 2048
    t = run.step(n_rays)                      # warm-up + calibration
    per_ray = run.step(n_rays) / n_rays
    n_rays = int(min(run.n_total, max(2048, budget_s / (min_runs + 1) / per_ray)))
    times = [run.step(n_rays) for _ in range(min_runs)]
    return {"n_rays": n_rays, "times": times, "n_total": run.n_total, "warmup_s": t, "threads": threads, "threads_tried": tried}


def run_reference(args, rank, world):
    """`--impl reference`: the reference's own CPU implementation of the path on the host cores (rank 0 only): the
    UNMODIFIED diffdrr.renderers.Siddon from baseline/_ref (forward + autograd to the ray end points) when that install
    is present, else the C/OpenMP port of the same algorithm (oracle/).  Each step is a bounded sample of the workload."""
    if rank != 0:
        return
    threads = host_threads()
    ref_mod = load_reference()
    if ref_mod is not None:
        run = ReferenceRun(ref_mod, args.vol, args.det)
        threads, _tried = best_reference_threads(run)
        run.step(1024)
        per_ray = run.step(2048) / 2048
        # ~3 s of CPU work per step, at most one full DRR
        n_rays = int(min(run.n_total, max(1024, 3.0 / per_ray)))
        for _ in range(args.warmup):
            run.step(n_rays)
        times = [run.step(n_rays) for _ in range(args.steps)]
        frac = n_rays / run.n_total
        kind, what = "reference", (f"unmodified diffdrr.renderers.Siddon.forward + backward (torch {torch.__version__}, "
                                   f"{threads} threads = fastest of the counts tried on {host_threads()} cores, {cpu_model()})")
        sample = f"{n_rays} of the {run.n_total} rays of one pose ({frac:.3f} DRR) fwd+bwd per step"
    else:
        from oracle import oracle  # noqa: F401

        times = cpu_oracle_time(args.vol, args.det, 1, args.warmup + args.steps, threads)[args.warmup:]
        frac, kind, what = 1.0, "port", "C/OpenMP port of reference renderers.py (oracle/); baseline/_ref is absent"
        sample = "1 DRR (pose) fwd+bwd per step"
    sec = float(np.sum(times))
    value = frac * len(times) / sec
    med = float(np.median(times))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "DRRs/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * sec / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "volume": [args.vol] * 3, "detector": [args.det] * 2, "sample": sample,
                   "renderer": "siddon"},
        "cpu_baseline": {"value": value, "unit": "DRRs/s", "cores": threads, "kind": kind, "cpu": cpu_model(),
                         "sample": f"{sample}, {len(times)} steps; {what}",
                         "median_value": frac / med, "min_step_s": float(np.min(times)), "median_step_s": med},
        "e2e": {"value": value, "unit": "DRRs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------
def _time_events(fn, steps, warmup=2):
    """Per-launch CUDA-event times (ms) of fn on the current stream."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in evs:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in evs]


def _stat(ms_list):
    return {"mean_ms": float(np.mean(ms_list)), "median_ms": float(np.median(ms_list)), "min_ms": float(np.min(ms_list))}


def _device_rays(drr, rot, xyz, dev):
    from diffdrr_b200.pose import convert

    B = rot.shape[0]
    with torch.no_grad():
        src, tgt = drr.detector(convert(rot.to(dev), xyz.to(dev), parameterization="euler_angles", convention="ZXY"), None)
        raylen = (tgt - src).norm(dim=-1).reshape(B, -1).contiguous()
        src = drr.affine_inverse(src).reshape(B, 3).contiguous()
        tgt = drr.affine_inverse(tgt).contiguous()
    return src, tgt, raylen


def extra_configs(dev, lib, peak, main):
    """Secondary, driver-visible numbers (VERDICT r1 item 4): the north star's inference forward (slab-major and brick-major
    TMA kernels), the reconstruction backward WITH the volume gradient, BASELINE config 2 (256^3 -> 256^2, B = 16, Siddon
    forward), config 3 (512^3 -> 512^2, B = 64, trilinear fwd+bwd(pose), 500 points) and config 5 (registration loop,
    1000 steps).  Every entry: CUDA-event times (mean / median / min) and the roofline fraction on ALGORITHMIC bytes."""
    from diffdrr_b200 import DRR, NormalizedCrossCorrelation2d, Registration, _lib, synthetic
    from diffdrr_b200.renderers import _get_alpha_minmax, _ptr, _stream, siddon_visits

    res = {}
    vol, src, tgt, raylen, gout = main["vol"], main["src"], main["tgt"], main["raylen"], main["gout"]
    B, D, det, N = main["B"], main["D"], main["det"], main["det"] ** 2
    tot_visits = main["tot_visits"]
    out = torch.empty(B, N, device=dev)

    def roof(bytes_, ms):
        gbs = bytes_ / (ms * 1e-3) / 1e9
        return {"achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak, "algorithmic_bytes_per_launch": bytes_}

    # ---- (a) north-star metric: Siddon FORWARD 512^3 -> 256^2, both production kernels ------------------------------
    fwd_bytes = 4 * tot_visits + 20 * B * N
    # variant 15 = the slab-major kernel (16 x 16 tiles, 32-plane slabs) by its explicit id; variant 0 = the library's choice for
    # this batch (up to 16 poses of 256^2 rays at >= 384^3: every ray cut into pieces along its own major axis)
    t_slab = _time_events(lambda: _lib.check(lib.b200drr_siddon_fwd_grid(_ptr(vol), D, D, D, _ptr(src), _ptr(tgt), _ptr(raylen),
                                                                         _ptr(out), B, det, det, 0.5, 1e-8, 15, _stream()), "fwd_grid"), 10)
    ref_img = out.clone()
    entry = {"workload": f"siddon forward, {D}^3 -> {det}^2, {B} poses", "slab_major": {**_stat(t_slab), "drr_per_s": B / np.median(t_slab) * 1e3,
                                                                                      "roofline": roof(fwd_bytes, float(np.median(t_slab)))}}
    t_def = _time_events(lambda: _lib.check(lib.b200drr_siddon_fwd_grid(_ptr(vol), D, D, D, _ptr(src), _ptr(tgt), _ptr(raylen),
                                                                        _ptr(out), B, det, det, 0.5, 1e-8, 0, _stream()), "fwd_grid"), 10)
    entry["library_default_major_axis_pieces"] = {**_stat(t_def), "drr_per_s": B / np.median(t_def) * 1e3,
                                                  "roofline": roof(fwd_bytes, float(np.median(t_def))),
                                                  "maxdiff_vs_slab_major": float((out - ref_img).abs().max() / ref_img.abs().max()),
                                                  "note": "b200drr_siddon_fwd_grid variant 0: siddon_fwd_slab_kernel<16,16,4,MAJ> with 16 pieces "
                                                          "per ray at this size (csrc/siddon.cu small_batch_pieces); the zero fill is in the time"}
    try:
        ws = torch.empty(lib.b200drr_siddon_brick_workspace_bytes(B, det, det), dtype=torch.uint8, device=dev)
        t_brick = _time_events(lambda: _lib.check(lib.b200drr_siddon_fwd_brick(
            _ptr(vol), D, D, D, _ptr(src), _ptr(tgt), _ptr(raylen), None, None, None, None, _ptr(out), _ptr(ws), ws.numel(), B, det,
            det, 0.5, 1e-8, 0, _stream()), "fwd_brick"), 10)
        entry["brick_major_tma"] = {**_stat(t_brick), "drr_per_s": B / np.median(t_brick) * 1e3,
                                    "roofline": roof(fwd_bytes, float(np.median(t_brick))),
                                    "maxdiff_vs_slab_major": float((out - ref_img).abs().max() / ref_img.abs().max()),
                                    "note": "ray table + zero fill (brick_prep_kernel) included in the time"}
        main["brick_img0"] = out[0].clone()
    except Exception as exc:  # pragma: no cover
        entry["brick_major_tma"] = {"error": f"{type(exc).__name__}: {exc}"}
    res["siddon_forward_inference"] = entry

    # ---- (b) reconstruction backward: two-walk backward WITH the volume gradient -----------------------------------
    g_src, g_tgt, g_len = torch.empty(B, 3, device=dev), torch.empty(B, N, 3, device=dev), torch.empty(B, N, device=dev)
    g_vol = torch.zeros_like(vol)
    t_gv = _time_events(lambda: _lib.check(lib.b200drr_siddon_bwd_grid(
        _ptr(vol), D, D, D, _ptr(src), _ptr(tgt), _ptr(raylen), _ptr(gout), _ptr(g_src), _ptr(g_tgt), _ptr(g_len), _ptr(g_vol), B, det,
        det, 0.5, 1e-8, 0, 0, _stream()), "bwd_grid"), 5)
    gv_bytes = 12 * tot_visits + 36 * B * N   # voxel read + 8 B read-modify-write of g_vol per visit + per-ray I/O
    res["siddon_backward_with_volume_gradient"] = {
        "workload": f"siddon backward incl. g_vol (reconstruction), {D}^3 -> {det}^2, {B} poses", **_stat(t_gv),
        "drr_per_s": B / np.median(t_gv) * 1e3, "roofline": roof(gv_bytes, float(np.median(t_gv)))}
    try:
        # the volume gradient alone (fixed poses: what a reconstruction step needs) by the brick kernel run as a scatter
        # (shared-memory accumulation, one TMA store per brick, no global atomics) vs the slab-major walk with global atomics
        g_ref = g_vol.clone()   # (accumulated over the timed launches above: compare shapes of one launch below)
        g_vol.zero_()
        one_slab = lambda: _lib.check(lib.b200drr_siddon_bwd_grid(  # noqa: E731
            _ptr(vol), D, D, D, _ptr(src), _ptr(tgt), _ptr(raylen), _ptr(gout), None, None, None, _ptr(g_vol), B, det, det, 0.5, 1e-8, 0,
            0, _stream()), "bwd_grid")
        one_slab()
        g_ref.copy_(g_vol)
        t_gs = _time_events(one_slab, 5)
        ws = torch.empty(lib.b200drr_siddon_brick_workspace_bytes(B, det, det), dtype=torch.uint8, device=dev)
        t_gb = _time_events(lambda: _lib.check(lib.b200drr_siddon_bwd_vol_brick(
            _ptr(gout), D, D, D, _ptr(src), _ptr(tgt), _ptr(raylen), None, None, None, None, _ptr(g_vol), _ptr(ws), ws.numel(), B, det,
            det, 0.5, 1e-8, _stream()), "bwd_vol_brick"), 5)
        sc_bytes = 8 * tot_visits + 4 * D ** 3 + 20 * B * N   # read-modify-write per visit + the volume store + per-ray inputs
        res["siddon_backward_with_volume_gradient"]["volume_gradient_only"] = {
            "slab_major_global_atomics": {**_stat(t_gs), "drr_per_s": B / np.median(t_gs) * 1e3, "roofline": roof(sc_bytes, float(np.median(t_gs)))},
            "brick_scatter_tma_store": {**_stat(t_gb), "drr_per_s": B / np.median(t_gb) * 1e3, "roofline": roof(sc_bytes, float(np.median(t_gb))),
                                        "maxdiff_vs_slab_major": float((g_vol - g_ref).abs().max() / g_ref.abs().max())}}
        del g_ref
    except Exception as exc:  # pragma: no cover
        res["siddon_backward_with_volume_gradient"]["volume_gradient_only"] = {"error": f"{type(exc).__name__}: {exc}"}
    del g_vol

    # ---- (c) BASELINE config 2: 256^3 -> 256^2, batch 16, Siddon forward ----------------------------------------------
    D2, B2 = 256, 16
    vol2 = torch.rand(D2, D2, D2, device=dev, generator=torch.Generator(device=dev).manual_seed(0))
    subj = synthetic.make_subject(torch.zeros(1, 1, 1, 1))
    subj.volume.affine = synthetic.make_affine(D2)
    drr2 = DRR(subj, **synthetic.detector_kwargs(256)).to(dev)
    rot, xyz = synthetic.make_poses(B2, seed=0)
    s2, t2, l2 = _device_rays(drr2, rot, xyz, dev)
    v2 = int(siddon_visits((D2, D2, D2), s2, t2).sum())
    o2 = torch.empty(B2, 256 * 256, device=dev)
    t_c2 = _time_events(lambda: _lib.check(lib.b200drr_siddon_fwd_grid(_ptr(vol2), D2, D2, D2, _ptr(s2), _ptr(t2), _ptr(l2), _ptr(o2),
                                                                       B2, 256, 256, 0.5, 1e-8, 0, _stream()), "fwd_grid c2"), 10)
    res["config2_siddon_forward_256"] = {"workload": "BASELINE config 2: 256^3 -> 256^2, 16 poses, Siddon forward (slab-major kernel)",
                                         **_stat(t_c2), "drr_per_s": B2 / np.median(t_c2) * 1e3,
                                         "roofline": roof(4 * v2 + 20 * B2 * 256 * 256, float(np.median(t_c2)))}
    del vol2, o2

    # ---- (d) BASELINE config 3: 512^3 -> 512^2, batch 64, trilinear fwd+bwd(pose), 500 points -------------------------
    try:
        H3, B3, P3 = 512, 64, 500
        N3 = H3 * H3
        subj = synthetic.make_subject(torch.zeros(1, 1, 1, 1))
        subj.volume.affine = synthetic.make_affine(D)
        drr3 = DRR(subj, **synthetic.detector_kwargs(H3)).to(dev)
        rot, xyz = synthetic.make_poses(B3, seed=0)
        s3, t3, l3 = _device_rays(drr3, rot, xyz, dev)
        with torch.no_grad():
            amin, amax = _get_alpha_minmax(s3.reshape(B3, 1, 3), t3, torch.tensor([D, D, D], device=dev, dtype=torch.float32), 0.5, 1e-8)
            ar = torch.stack([amin.min(), amax.max()]).contiguous()
            lin = torch.linspace(0, 1, P3, device=dev) * (ar[1] - ar[0]) + ar[0]
            cnt = 0
            for b in range(0, B3, 8):   # in-volume samples of every 8th pose (>= 1 corner in bounds), scaled up
                for c in range(0, N3, 65536):
                    pts = s3[b][None, None, :] + lin[None, :, None] * (t3[b, c:c + 65536][:, None, :] - s3[b][None, None, :])
                    cnt += int(((pts > -1) & (pts < D)).all(-1).sum())
            cnt *= 8
        packed = torch.empty(int(lib.b200drr_packed_volume_floats(D, D, D)), device=dev)
        _lib.check(lib.b200drr_pack_corners(_ptr(vol), D, D, D, _ptr(packed), _stream()), "pack")
        o3, sens3 = torch.empty(B3, N3, device=dev), torch.empty(B3, N3, 12, device=dev)
        go3 = torch.rand(B3, N3, device=dev)
        h_src, h_tgt, h_len, h_ar = torch.empty(B3, 3, device=dev), torch.empty(B3, N3, 3, device=dev), torch.empty(B3, N3, device=dev), torch.zeros(2, device=dev)

        def tri_step():
            _lib.check(lib.b200drr_trilinear_fwd_sens_packed(_ptr(packed), D, D, D, _ptr(s3), _ptr(t3), _ptr(l3), _ptr(o3), _ptr(sens3), B3,
                                                             H3, H3, 0.5, 1e-8, P3, _ptr(ar), 0, _stream()), "tri fwd_sens")
            _lib.check(lib.b200drr_trilinear_bwd_sens(_ptr(sens3), _ptr(go3), _ptr(h_src), _ptr(h_tgt), _ptr(h_len), _ptr(h_ar), B3, N3,
                                                      _stream()), "tri bwd_sens")

        t_c3 = _time_events(tri_step, 5, warmup=1)
        t_c3f = _time_events(lambda: _lib.check(lib.b200drr_trilinear_fwd_packed(
            _ptr(packed), D, D, D, _ptr(s3), _ptr(t3), _ptr(l3), _ptr(o3), B3, H3, H3, 0.5, 1e-8, P3, _ptr(ar), 16, _stream()), "tri fwd"), 3, warmup=1)
        tri_bytes = 32 * cnt
        res["config3_trilinear_fwd_bwd_512"] = {
            "workload": "BASELINE config 3: 512^3 -> 512^2, 64 poses, trilinear (500 points) forward + backward (pose gradients); "
                        "one march yields image + sensitivities, backward elementwise",
            **_stat(t_c3), "drr_per_s": B3 / np.median(t_c3) * 1e3, "in_volume_sample_fraction": cnt / (B3 * N3 * P3),
            "roofline": roof(tri_bytes, float(np.median(t_c3))),
            "forward_only_slab_major": {**_stat(t_c3f), "drr_per_s": B3 / np.median(t_c3f) * 1e3, "roofline": roof(tri_bytes, float(np.median(t_c3f)))}}
        del packed, sens3, h_tgt, o3
        # the same step through the module API, `DRR(rot, xyz)` + backward(): pose-in entry (rays generated in-kernel,
        # b200drr_trilinear_fwd_sens_pose) against detector.forward + the ray-tensor kernels
        import diffdrr_b200.drr as drr_mod

        drr3m = DRR(subj, **synthetic.detector_kwargs(H3), renderer="trilinear").to(dev)
        drr3m.density = vol
        rot_d, xyz_d = rot.to(dev).requires_grad_(True), xyz.to(dev).requires_grad_(True)
        w3 = go3.view(B3, 1, H3, H3)

        def mod_step():
            rot_d.grad, xyz_d.grad = None, None
            img = drr3m(rot_d, xyz_d, parameterization="euler_angles", convention="ZXY", n_points=P3)
            (img * w3).sum().backward()

        module = {}
        keep = drr_mod._TRILINEAR_POSE_IN
        for tag, flag in (("pose_in", True), ("ray_tensors", False)):
            drr_mod._TRILINEAR_POSE_IN = flag
            t_m = _time_events(mod_step, 5, warmup=2)
            module[tag] = {**_stat(t_m), "drr_per_s": B3 / np.median(t_m) * 1e3}
        drr_mod._TRILINEAR_POSE_IN = keep
        res["config3_trilinear_fwd_bwd_512"]["module_drr_rot_xyz_backward"] = module
        del drr3m, go3, w3
    except Exception as exc:  # pragma: no cover
        res.setdefault("config3_trilinear_fwd_bwd_512", {})["error"] = f"{type(exc).__name__}: {exc}"
    torch.cuda.empty_cache()

    # ---- (e) BASELINE config 5: 2D/3D registration loop, 1000 gradient steps, 512^3 CT, 256^2 target -------------------
    try:
        x = torch.linspace(-1, 1, D, device=dev)
        X, Y, Z = x[:, None, None], x[None, :, None], x[None, None, :]
        smooth = torch.exp(-((X - 0.2) ** 2 + (Y + 0.1) ** 2 + (Z - 0.05) ** 2) / 0.18)
        smooth += 0.6 * torch.exp(-((X + 0.35) ** 2 + (Y - 0.3) ** 2 + (Z + 0.25) ** 2) / 0.05)
        subj = synthetic.make_subject(torch.zeros(1, 1, 1, 1))
        subj.volume.affine = synthetic.make_affine(D)
        drr5 = DRR(subj, **synthetic.detector_kwargs(256), renderer="siddon", stop_gradients_through_grid_sample=True).to(dev)
        drr5.density = smooth.contiguous()
        true_rot, true_xyz = torch.tensor([[0.0, 0.0, 0.0]], device=dev), torch.tensor([[0.0, 850.0, 0.0]], device=dev)
        with torch.no_grad():
            target = drr5(true_rot, true_xyz, parameterization="euler_angles", convention="ZXY")
        reg = Registration(drr5, (true_rot + torch.tensor([[0.15, -0.1, 0.08]], device=dev)).clone(),
                           (true_xyz + torch.tensor([[12.0, -25.0, 9.0]], device=dev)).clone(), "euler_angles", "ZXY").to(dev)
        ncc = NormalizedCrossCorrelation2d()
        # torch's own fused (multi-tensor) Adam: 4 launches per step instead of ~25; the loss is the fused NCC (csrc/ncc.cu)
        opt = torch.optim.Adam([{"params": [reg.rotation], "lr": 5e-3}, {"params": [reg.translation], "lr": 5e-1}], capturable=True,
                               fused=True)

        def reg_step():
            opt.zero_grad(set_to_none=False)
            loss = 1.0 - ncc(target, reg()).mean()
            loss.backward()
            opt.step()
            return loss

        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(5):
                reg_step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            reg_step()
        n_it = 1000
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n_it):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        with torch.no_grad():
            final = float(1.0 - ncc(target, reg()).mean())
        res["config5_registration_loop"] = {
            "workload": "BASELINE config 5: 1000 gradient steps (Adam, NCC), 512^3 CT, 256^2 target DRR, B = 1, whole step in one CUDA graph; "
                        "renderer: forward-with-sensitivities kernel with 12 major-axis pieces per ray, loss: b200drr_ncc_fwd/_bwd, optimiser: "
                        "torch.optim.Adam(fused=True, capturable=True)",
            "it_per_s": n_it / (ms * 1e-3), "ms_per_it": ms / n_it, "final_1_minus_ncc": final,
            "rot_err_rad": float((reg.rotation.detach() - true_rot).abs().max()),
            "xyz_err_mm": float((reg.translation.detach() - true_xyz).abs().max())}
        del smooth
    except Exception as exc:  # pragma: no cover
        res["config5_registration_loop"] = {"error": f"{type(exc).__name__}: {exc}"}
    torch.cuda.empty_cache()
    return res


def reference_on_gpu(vol_n, det_n):
    """SURVEY 2b's bar: the reference's own PyTorch path (`Siddon.forward` + autograd) under .to("cuda") on this B200,
    512^3 -> 256^2, ONE pose, forward + backward (it materialises ~20 (1, 65536, 1539) tensors; B = 16 would not fit the
    comparison's spirit of a single call).  Wall clock around synchronised calls, 1 warm-up + 5 runs."""
    ref_mod = load_reference()
    if ref_mod is None:
        return {"unavailable": "baseline/_ref is absent"}
    try:
        run = ReferenceRun(ref_mod, vol_n, det_n, device="cuda")
        run.step(run.n_total)
        times = [run.step(run.n_total) for _ in range(5)]
        return {"workload": f"reference Siddon.forward + backward on the same B200, {vol_n}^3 -> {det_n}^2, 1 pose per call",
                "drr_per_s": 1.0 / float(np.median(times)), "median_s": float(np.median(times)), "min_s": float(np.min(times)),
                "peak_memory_gb": torch.cuda.max_memory_allocated() / 1e9}
    except Exception as exc:
        return {"error": f"{type(exc).__name__}: {exc}"}
    finally:
        torch.cuda.empty_cache()


def run_ours(args, rank, local_rank, world):
    import torch.distributed as dist

    from diffdrr_b200 import DRR, _lib, synthetic
    from diffdrr_b200.pose import convert
    from diffdrr_b200.renderers import _ptr, _stream, siddon_visits

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: diffdrr_b200 has no CPU path (use --impl reference for the CPU port)")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    B, N, D = args.batch, args.det * args.det, args.vol

    # synthetic volume (performance is data independent) + module with the reference surface
    gen = torch.Generator(device=dev).manual_seed(0)
    vol = torch.rand(D, D, D, device=dev, generator=gen)
    subj = synthetic.make_subject(torch.zeros(1, 1, 1, 1))
    subj.volume.affine = synthetic.make_affine(D)
    drr = DRR(subj, **synthetic.detector_kwargs(args.det), renderer="siddon").to(dev)
    drr.density = vol  # the 537 MB volume lives on the device only

    # this rank's poses (weak scaling: B per GPU); host copies live in pinned memory for the e2e leg
    rot_all, xyz_all = synthetic.make_poses(B * world, seed=0)
    mine = list(range(rank * B, (rank + 1) * B))
    balance = "contiguous slices"
    if world > 1 and os.environ.get("B200DRR_BENCH_BALANCE", "0") == "1":  # opt-in: measured 1.3 % SLOWER at N = 8 (DESIGN.md 6)
        # every rank still renders exactly B poses (weak scaling), but WHICH poses is decided by their cost (voxels visited,
        # known from a closed-form count): the step ends when the slowest rank does
        from diffdrr_b200.parallel import balanced_pose_assignment

        with torch.no_grad():
            costs = []
            for b0 in range(0, B * world, 16):
                p_ = convert(rot_all[b0:b0 + 16].to(dev), xyz_all[b0:b0 + 16].to(dev), parameterization="euler_angles", convention="ZXY")
                s_, t_ = drr.detector(p_, None)
                costs += siddon_visits((D, D, D), drr.affine_inverse(s_), drr.affine_inverse(t_)).sum(dim=1).tolist()
        mine = balanced_pose_assignment(costs, world)[rank]
        balance = "equal pose counts, groups balanced by visit count (parallel.balanced_pose_assignment)"
    rot_h = rot_all[mine].contiguous().pin_memory()
    xyz_h = xyz_all[mine].contiguous().pin_memory()
    with torch.no_grad():
        pose = convert(rot_h.to(dev), xyz_h.to(dev), parameterization="euler_angles", convention="ZXY")
        src, tgt = drr.detector(pose, None)
        raylen = (tgt - src).norm(dim=-1).unsqueeze(1).contiguous()
        src = drr.affine_inverse(src).reshape(B, 3).contiguous()
        tgt = drr.affine_inverse(tgt).contiguous()
    w = torch.rand(B, 1, args.det, args.det, device=dev, generator=gen)  # upstream gradient dLoss/dImage
    gout = w.reshape(B, N).contiguous()
    out = torch.empty(B, N, device=dev)
    g_src, g_tgt, g_len = torch.empty(B, 3, device=dev), torch.empty(B, N, 3, device=dev), torch.empty(B, N, device=dev)

    visits = siddon_visits((D, D, D), src, tgt)
    tot_visits = int(visits.sum().item())
    fwd_bytes = 4 * tot_visits + (4 + 16) * B * N            # voxels + out + (tgt, raylen)
    bwd_bytes = 4 * tot_visits + (4 + 16 + 12 + 4) * B * N   # voxels + gout + (tgt, raylen) + g_tgt + g_raylen

    stream = torch.cuda.current_stream()

    sens = torch.empty(B, N, 8, device=dev)
    sens_bytes = 4 * tot_visits + (16 + 4 + 32) * B * N      # voxels + (tgt, raylen) + out + 8 sensitivities per ray

    outs = [out, torch.empty_like(out)] if world > 1 else [out]
    gathered = [torch.empty(B * world, N, device=dev) for _ in range(2)] if world > 1 else None
    pending, state = [None, None], {"k": 0}
    # the gather of the image stack: peer copies on the copy engines (no SM), NCCL only if symmetric memory is unavailable
    peer, gather_kind = None, "none (1 GPU)"
    if world > 1:
        gather_kind = "nccl all_gather_into_tensor"
        if os.environ.get("B200DRR_BENCH_GATHER", "peer") == "peer":
            try:
                from diffdrr_b200.parallel import PeerGather

                peer = PeerGather((B, N), torch.float32, dev, slots=2)
                gather_kind = "peer copies over NVLink on the copy engines (symmetric memory), no SM"
            except Exception as exc:
                gather_kind += f" (peer gather unavailable: {type(exc).__name__}: {exc})"

    def kernel_step(ev=None):
        """One training step at kernel level: image + per-ray sensitivities in ONE walk, then the elementwise backward."""
        out = outs[state["k"] & 1] if world > 1 else outs[0]
        if ev:
            ev[0].record(stream)
        _lib.check(lib.b200drr_siddon_fwd_sens_grid(_ptr(vol), D, D, D, _ptr(src), _ptr(tgt), _ptr(raylen), _ptr(out),
                                                    _ptr(sens), B, args.det, args.det, 0.5, 1e-8, 0, _stream()),
                   "siddon_fwd_sens_grid")
        if ev:
            ev[1].record(stream)
        _lib.check(lib.b200drr_siddon_bwd_sens(_ptr(sens), _ptr(gout), _ptr(g_src), _ptr(g_tgt), _ptr(g_len), B, N, 0,
                                               _stream()), "siddon_bwd_sens")
        if ev:
            ev[2].record(stream)
        if world > 1:
            # double-buffered: the gather of this step's image stack runs on NCCL's stream while the next step walks
            # (the next step writes the other buffer); a buffer is reused only after its gather has been waited for
            slot = state["k"] & 1
            if peer is not None:
                peer.wait(slot)           # the previous gather into this slot has been consumed
                peer.push(outs[slot], slot)
            else:
                if pending[slot] is not None:
                    pending[slot].wait()
                pending[slot] = dist.all_gather_into_tensor(gathered[slot], outs[slot], async_op=True)
            state["k"] += 1

    def drain():
        for slot in (0, 1):
            if peer is not None:
                peer.wait(slot)
            elif pending[slot] is not None:
                pending[slot].wait()
                pending[slot] = None

    def two_walk_step(ev):
        """The inference forward and the backward WALK (still the path when the volume needs gradients), for the record."""
        ev[0].record(stream)
        _lib.check(lib.b200drr_siddon_fwd_grid(_ptr(vol), D, D, D, _ptr(src), _ptr(tgt), _ptr(raylen), _ptr(out), B, args.det,
                                               args.det, 0.5, 1e-8, 0, _stream()), "siddon_fwd_grid")
        ev[1].record(stream)
        _lib.check(lib.b200drr_siddon_bwd_grid(_ptr(vol), D, D, D, _ptr(src), _ptr(tgt), _ptr(raylen), _ptr(gout), _ptr(g_src),
                                               _ptr(g_tgt), _ptr(g_len), None, B, args.det, args.det, 0.5, 1e-8, 0, 0,
                                               _stream()), "siddon_bwd_grid")
        ev[2].record(stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- kernels-only leg (inputs resident in HBM) ------------------------------------------------------
    for _ in range(args.warmup):
        kernel_step()
    drain()
    events = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    with ClockSampler(local_rank) as clocks:
        t_start.record(stream)
        for k in range(args.steps):
            kernel_step(events[k])
        drain()  # the last gathers complete inside the timed region
        t_end.record(stream)
        barrier()
    ms_total = t_start.elapsed_time(t_end)
    if args.dump_outputs and rank == 0:  # the legs below overwrite these buffers
        last = outs[(state["k"] - 1) & 1] if world > 1 else outs[0]
        dump = {"image": last.reshape(B, 1, args.det, args.det).cpu(), "grad_source": g_src.cpu(),
                "grad_target": g_tgt.cpu(), "grad_raylen": g_len.cpu()}
    sens_list = [e[0].elapsed_time(e[1]) for e in events]
    sens_bwd_list = [e[1].elapsed_time(e[2]) for e in events]
    sens_ms = float(np.mean(sens_list))
    sens_bwd_ms = float(np.mean(sens_bwd_list))
    # not part of `value`: the plain forward kernel (inference) and the backward walk, timed the same way
    events2 = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    for k in range(args.steps):
        two_walk_step(events2[k])
    torch.cuda.synchronize()
    fwd_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in events2[1:] or events2]))
    bwd_ms = float(np.mean([e[1].elapsed_time(e[2]) for e in events2[1:] or events2]))

    # ---- end-to-end leg through the public module, host buffers in and out -----------------------------
    img_h = torch.empty(B, 1, args.det, args.det).pin_memory()
    grad_h = torch.empty(2, B, 3).pin_memory()
    loss_h = torch.empty(1).pin_memory()

    def e2e_step():
        rot = rot_h.to(dev, non_blocking=True).requires_grad_(True)
        xyz = xyz_h.to(dev, non_blocking=True).requires_grad_(True)
        img = drr(rot, xyz, parameterization="euler_angles", convention="ZXY")
        loss = (img * w).sum()
        loss.backward()
        if world > 1:
            if peer is not None:
                peer.push(img.detach().reshape(B, N), 0)
                peer.wait(0)
            else:
                dist.all_gather_into_tensor(gathered[0], img.detach().reshape(B, N))
        img_h.copy_(img.detach(), non_blocking=True)
        grad_h[0].copy_(rot.grad, non_blocking=True)
        grad_h[1].copy_(xyz.grad, non_blocking=True)
        loss_h.copy_(loss.detach().reshape(1), non_blocking=True)
        torch.cuda.current_stream().synchronize()  # the user reads the result every step

    for _ in range(args.warmup):
        e2e_step()
    e_start, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e_start.record(stream)
    for _ in range(args.steps):
        e2e_step()
    e_end.record(stream)
    barrier()
    e2e_eager_ms_total = e_start.elapsed_time(e_end)

    # ---- the same end-to-end step captured ONCE in a CUDA graph and replayed (streams + graphs, no tracing compiler):
    # pinned-host pose -> H2D -> DRR(rot, xyz) -> loss -> backward -> D2H of image stack / loss / pose gradients.
    # The host buffers are re-read by every replay, so each step can carry new poses.  (Single GPU only: NCCL
    # collectives are kept out of the capture.)
    e2e_ms_total, e2e_mode = e2e_eager_ms_total, "eager"
    # N > 1: the per-rank step is replayed from its graph and the gather of the image stack is issued after the replay,
    # outside the capture (B200DRR_BENCH_GRAPH_MULTI=0 switches back to the eager step).
    graph_multi = world > 1 and os.environ.get("B200DRR_BENCH_GRAPH_MULTI", "1") == "1"
    if (world == 1 or graph_multi) and not args.no_graph:
        try:
            rot_d = torch.zeros(B, 3, device=dev, requires_grad=True)
            xyz_d = torch.zeros(B, 3, device=dev, requires_grad=True)
            rot_d.grad, xyz_d.grad = torch.zeros_like(rot_d), torch.zeros_like(xyz_d)

            copy_stream = torch.cuda.Stream()

            def graph_body():
                main = torch.cuda.current_stream()
                with torch.no_grad():
                    rot_d.copy_(rot_h, non_blocking=True)
                    xyz_d.copy_(xyz_h, non_blocking=True)
                    rot_d.grad.zero_()
                    xyz_d.grad.zero_()
                img = drr(rot_d, xyz_d, parameterization="euler_angles", convention="ZXY")
                # the 4 MB image stack goes back to the host on a second stream while loss + backward run
                # (a fork/join inside the captured graph)
                copy_stream.wait_stream(main)
                with torch.cuda.stream(copy_stream):
                    img_h.copy_(img.detach(), non_blocking=True)
                loss = (img * w).sum()
                loss.backward()
                main.wait_stream(copy_stream)
                grad_h[0].copy_(rot_d.grad, non_blocking=True)
                grad_h[1].copy_(xyz_d.grad, non_blocking=True)
                loss_h.copy_(loss.detach().reshape(1), non_blocking=True)
                return img.detach()

            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(3):
                    graph_body()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            ref_img = img_h.clone()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                img_static = graph_body()

            def graph_step():
                graph.replay()
                if world > 1:
                    if peer is not None:
                        peer.push(img_static.reshape(B, N), 0)
                        peer.wait(0)
                    else:
                        dist.all_gather_into_tensor(gathered[0], img_static.reshape(B, N))
                torch.cuda.current_stream().synchronize()  # the user reads the result every step

            for _ in range(args.warmup):
                graph_step()
            assert torch.allclose(img_h, ref_img, rtol=1e-4, atol=1e-3), "graph replay changed the images"
            g_start, g_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            g_start.record(stream)
            for _ in range(args.steps):
                graph_step()
            g_end.record(stream)
            barrier()
            e2e_ms_total, e2e_mode = g_start.elapsed_time(g_end), "cuda-graph replay of the public-API step"
        except Exception as exc:  # capture is an optimisation of the launch path only; never hide the eager number
            e2e_mode = f"eager (graph capture failed: {type(exc).__name__})"
    if args.dump_outputs and rank == 0:  # + what the last end-to-end step handed back to the host
        dump.update(e2e_image=img_h, e2e_grad_rot=grad_h[0], e2e_grad_xyz=grad_h[1], e2e_loss=loss_h)
        dump_outputs(args.dump_outputs, dump)

    # ---- max over ranks -------------------------------------------------------------------------------------
    stats = torch.tensor([ms_total, e2e_ms_total, fwd_ms, bwd_ms, e2e_eager_ms_total, sens_ms, sens_bwd_ms], device=dev,
                         dtype=torch.float64)
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms_total, fwd_ms, bwd_ms, e2e_eager_ms_total, sens_ms, sens_bwd_ms = (float(x) for x in stats.tolist())
    if rank != 0:
        return

    peak, peak_src = hbm_peak()
    total_drr = B * world * args.steps
    value = total_drr / (ms_total * 1e-3)
    e2e_value = total_drr / (e2e_ms_total * 1e-3)
    fwd_gbs = fwd_bytes / (fwd_ms * 1e-3) / 1e9
    bwd_gbs = bwd_bytes / (bwd_ms * 1e-3) / 1e9
    sens_gbs = sens_bytes / (sens_ms * 1e-3) / 1e9
    dom = ("siddon_sens_slab_kernel", sens_gbs, sens_bytes, sens_ms)  # >95 % of the step
    line = {
        "metric": METRIC, "value": value, "unit": "DRRs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "volume": [D] * 3, "detector": [args.det] * 2, "batch_per_gpu": B,
                   "global_batch": B * world, "renderer": "siddon", "parallelism": f"pose-sharded dp{world}", "gather": gather_kind, "pose_assignment": balance,
                   "l2": f"inputs > L2 ({4 * D ** 3 / 1e6:.0f} MB volume vs 126 MB L2); no explicit flush",
                   "mean_visits_per_ray": tot_visits / (B * N)},
        "e2e": {"value": e2e_value, "unit": "DRRs/s", "ms_per_step": e2e_ms_total / args.steps, "mode": e2e_mode,
                "eager_value": total_drr / (e2e_eager_ms_total * 1e-3), "eager_ms_per_step": e2e_eager_ms_total / args.steps,
                "h2d_bytes_per_step": int(rot_h.numel() + xyz_h.numel()) * 4,
                "d2h_bytes_per_step": int(img_h.numel() + grad_h.numel() + loss_h.numel()) * 4,
                "path": "DRR(rot, xyz) -> (img*w).sum().backward(); pinned host pose in; image stack + loss + pose grads out"},
        "gpu_launches": 2 * args.steps,
        "roofline": {"bound": "hbm", "kernel": dom[0], "achieved": dom[1], "peak": peak, "unit": "GB/s", "frac": dom[1] / peak,
                     "traffic": NCU_TRAFFIC_BYTES.get(dom[0]) if (B, D, args.det) == (16, VOL, DET) else None,
                     "traffic_source": NCU_TRAFFIC_SOURCE, "algorithmic_bytes_per_launch": dom[2], "ms_per_launch": dom[3], "peak_source": peak_src},
        "step_breakdown_ms": {"siddon_sens_slab_kernel (image + sensitivities, one walk)": sens_ms,
                              "sens_bwd_kernel (elementwise backward)": sens_bwd_ms},
        "roofline_fwd": {"kernel": "siddon_fwd_slab_kernel (b200drr_siddon_fwd_grid's choice for this batch: rays cut into major-axis "
                                   "pieces up to 16 poses of 256^2 rays, slab-major beyond)", "achieved": fwd_gbs, "frac": fwd_gbs / peak, "ms_per_launch": fwd_ms,
                         "algorithmic_bytes_per_launch": fwd_bytes, "drr_per_s_fwd_only": B / (fwd_ms * 1e-3)},
        "roofline_bwd": {"kernel": "siddon_bwd_slab_kernel", "achieved": bwd_gbs, "frac": bwd_gbs / peak, "ms_per_launch": bwd_ms,
                         "algorithmic_bytes_per_launch": bwd_bytes,
                         "note": "two-walk backward; used when the volume needs gradients, not part of the timed step"},
        "clocks": clocks.summary(),
    }
    line["timing"] = {"siddon_sens_slab_kernel": _stat(sens_list), "sens_bwd_kernel": _stat(sens_bwd_list),
                      "note": "per-launch CUDA-event times over the timed region; roofline.achieved uses the mean"}
    if world == 1:
        # ---- parity of the TIMED output: pose 0 of this run against the fp64 oracle on the same rays ------------------
        try:
            from oracle import oracle

            oracle.set_threads(host_threads())
            a = (src[:1].cpu().numpy().reshape(1, 1, 3), tgt[:1].cpu().numpy(), raylen[:1].cpu().numpy().reshape(1, 1, N))
            ref64 = oracle.siddon_fwd(np.ascontiguousarray(vol.cpu().numpy()), *a, dtype=np.float64).reshape(-1)
            kernel_step()
            torch.cuda.synchronize()
            got = outs[0][0].cpu().numpy().astype(np.float64)
            err = float(np.abs(got - ref64).max() / np.abs(ref64).max())
            line["parity_check"] = {"sens_kernel_image_vs_fp64_oracle": err, "tolerance": 1e-4, "pose": 0,
                                    "what": "max-abs error / max-abs reference over the full 256^2 image of pose 0"}
            assert err < 1e-4, f"timed kernel output differs from the oracle: {err:.3e}"
        except ImportError:
            ref64 = None
        main_state = dict(vol=vol, src=src, tgt=tgt, raylen=raylen, gout=gout, B=B, D=D, det=args.det, tot_visits=tot_visits)
        if not args.no_extra:
            try:  # secondary legs never take the headline line down with them: a failure is reported, not hidden
                line["configs"] = extra_configs(dev, lib, peak, main_state)
            except Exception as exc:  # pragma: no cover
                line["configs"] = {"error": f"{type(exc).__name__}: {exc}"}
                torch.cuda.empty_cache()
            if ref64 is not None and "brick_img0" in main_state:
                e2 = float(np.abs(main_state["brick_img0"].cpu().numpy().astype(np.float64) - ref64).max() / np.abs(ref64).max())
                line["parity_check"]["brick_forward_image_vs_fp64_oracle"] = e2
                assert e2 < 1e-4, f"brick forward differs from the oracle: {e2:.3e}"
            try:
                line["reference_on_this_gpu"] = reference_on_gpu(D, args.det)
            except Exception as exc:  # pragma: no cover
                line["reference_on_this_gpu"] = {"error": f"{type(exc).__name__}: {exc}"}
            ref_gpu = line["reference_on_this_gpu"].get("drr_per_s")
            if ref_gpu:
                line["reference_on_this_gpu"]["ours_over_reference_fwd_bwd"] = value / ref_gpu
    if not args.no_cpu_baseline and world == 1:
        # the reference's own PyTorch-CPU path on this box's host cores (bounded sample), else the C port of it
        sample = cpu_reference_sample(D, args.det, budget_s=15.0)
        if sample is not None:
            med = float(np.median(sample["times"]))
            frac = sample["n_rays"] / sample["n_total"]
            line["cpu_baseline"] = {
                "value": frac / med, "unit": "DRRs/s", "cores": sample["threads"], "host_cores": host_threads(), "kind": "reference",
                "cpu": cpu_model(), "threads_tried_s": {str(k): v for k, v in sample["threads_tried"].items()},
                "sample": f"{sample['n_rays']} of {sample['n_total']} rays of one pose ({frac:.3f} DRR) fwd+bwd, median of "
                          f"{len(sample['times'])} runs after warm-up; unmodified diffdrr.renderers.Siddon (baseline/_ref), torch "
                          f"{torch.__version__} with {sample['threads']} threads (fastest of the counts tried on {host_threads()} cores)",
                "min_value": frac / float(np.min(sample["times"]))}
        from oracle import oracle

        threads = host_threads()
        times = cpu_oracle_time(D, args.det, 1, 6, threads)[1:]
        port = {"value": 1.0 / float(np.median(times)), "unit": "DRRs/s", "cores": threads, "kind": "port",
                "sample": f"1 DRR fwd+bwd(pose) of the same {D}^3->{args.det}^2 workload, median of {len(times)} runs after 1 warm-up; "
                          "C/OpenMP port of reference renderers.py (oracle/)"}
        if "cpu_baseline" in line:
            line["cpu_port"] = port
        else:
            line["cpu_baseline"] = port
    print(json.dumps(line), flush=True)


def run_config4(args, rank, local_rank, world):
    """BASELINE config 4: 512^3 CT -> 1024^2 detector, batch = 256 poses pose-sharded across the GPUs of the box, one gather
    of the (256, 1024, 1024) image stack per step.  Inference forward through the brick-major TMA kernel (slab-major kernel
    timed beside it on rank 0's shard); strong scaling: the global batch is fixed at 256."""
    import torch.distributed as dist

    from diffdrr_b200 import DRR, _lib, synthetic
    from diffdrr_b200.renderers import _ptr, _stream, siddon_visits

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    D, det, GB = 512, 1024, 256
    N = det * det
    if GB % world:
        raise SystemExit("config4 needs a GPU count that divides 256")
    B = GB // world
    vol = torch.rand(D, D, D, device=dev, generator=torch.Generator(device=dev).manual_seed(0))
    subj = synthetic.make_subject(torch.zeros(1, 1, 1, 1))
    subj.volume.affine = synthetic.make_affine(D)
    drr = DRR(subj, **synthetic.detector_kwargs(det)).to(dev)
    rot_all, xyz_all = synthetic.make_poses(GB, seed=0)
    src, tgt, raylen = _device_rays(drr, rot_all[rank * B:(rank + 1) * B], xyz_all[rank * B:(rank + 1) * B], dev)
    out = torch.empty(B, N, device=dev)
    ws = torch.empty(lib.b200drr_siddon_brick_workspace_bytes(B, det, det), dtype=torch.uint8, device=dev)
    visits = 0
    for b0 in range(0, B, 8):
        visits += int(siddon_visits((D, D, D), src[b0:b0 + 8].contiguous(), tgt[b0:b0 + 8].contiguous()).sum())
    peer, gather_kind = None, "none (1 GPU)"
    if world > 1:
        try:
            from diffdrr_b200.parallel import PeerGather

            peer = PeerGather((B, N), torch.float32, dev, slots=1)
            gather_kind = "peer copies over NVLink on the copy engines (symmetric memory), no SM"
        except Exception as exc:
            gather_kind = f"nccl all_gather_into_tensor ({type(exc).__name__}: {exc})"
            gathered = torch.empty(GB, N, device=dev)

    def brick():
        _lib.check(lib.b200drr_siddon_fwd_brick(_ptr(vol), D, D, D, _ptr(src), _ptr(tgt), _ptr(raylen), None, None, None, None, _ptr(out),
                                                _ptr(ws), ws.numel(), B, det, det, 0.5, 1e-8, 0, _stream()), "fwd_brick")

    def slab():
        _lib.check(lib.b200drr_siddon_fwd_grid(_ptr(vol), D, D, D, _ptr(src), _ptr(tgt), _ptr(raylen), _ptr(out), B, det, det, 0.5, 1e-8, 0,
                                               _stream()), "fwd_grid")

    # the module's own choice (renderers._brick_ok): dense ray sets (1024^2 pixels through 512^2-voxel cross-sections, rays half
    # a voxel apart) take the slab-major kernel, sparse ones the brick-major TMA kernel
    use_brick = N <= 0.5 * float(D * D)
    forward = brick if use_brick else slab

    def step():
        forward()
        if world > 1:
            if peer is not None:
                peer.push(out, 0)
                peer.wait(0)
            else:
                dist.all_gather_into_tensor(gathered, out)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    with ClockSampler(local_rank) as clocks:
        e0.record()
        for _ in range(args.steps):
            step()
        e1.record()
        barrier()
    ms_total = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:  # before the kernel timings below overwrite `out`
        dump_outputs(args.dump_outputs, {"image": out.reshape(B, 1, det, det)})
    t_brick = _time_events(brick, 3, warmup=1)
    t_slab = _time_events(slab, 3, warmup=1)
    stats = torch.tensor([ms_total, float(np.median(t_brick)), float(np.median(t_slab)), float(visits)], device=dev, dtype=torch.float64)
    if world > 1:
        mx = stats.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = stats.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        ms_total, kb, ks = float(mx[0]), float(mx[1]), float(mx[2])
        visits_all = float(sm[3])
    else:
        kb, ks, visits_all = float(stats[1]), float(stats[2]), float(visits)
    if rank != 0:
        return
    peak, peak_src = hbm_peak()
    bytes_rank = 4 * visits_all / world + 20 * B * N
    print(json.dumps({
        "metric": "DRRs/sec fwd (512^3 CT -> 1024^2 det, 256 poses), BASELINE config 4", "value": GB * args.steps / (ms_total * 1e-3),
        "unit": "DRRs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "siddon forward (inference), 512^3 fp32 CT -> 1024^2 detector, 256 poses pose-sharded + one gather of the "
                               "image stack per step", "batch_per_gpu": B, "global_batch": GB, "gather": gather_kind,
                   "mean_visits_per_ray": visits_all / (GB * N), "l2": "inputs > L2; no explicit flush"},
        "roofline": {"bound": "hbm", "kernel": ("siddon_fwd_brick_kernel" if use_brick else "siddon_fwd_slab_kernel") + " (slowest rank)",
                     "achieved": bytes_rank / ((kb if use_brick else ks) * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": bytes_rank / ((kb if use_brick else ks) * 1e-3) / 1e9 / peak, "ms_per_launch": kb if use_brick else ks,
                     "algorithmic_bytes_per_launch": bytes_rank, "peak_source": peak_src, "traffic": None,
                     "brick_major_kernel_ms_per_launch": kb, "brick_major_frac": bytes_rank / (kb * 1e-3) / 1e9 / peak,
                     "slab_major_kernel_ms_per_launch": ks, "slab_major_frac": bytes_rank / (ks * 1e-3) / 1e9 / peak,
                     "note": "rays are 0.5 voxel apart at 1024^2: algorithmic bytes exceed the DRAM bytes many times over (every "
                             "staged voxel serves ~4x more rays than at 256^2)"},
        "gather_bytes_per_step_per_rank": (world - 1) * B * N * 4, "clocks": clocks.summary()}), flush=True)


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local_rank)
        opts = None
        try:  # the only collectives left are barriers / tiny reductions: keep NCCL's kernels off the walk's SMs
            opts = dist.ProcessGroupNCCL.Options()
            opts.config.max_ctas = 2
        except Exception:
            opts = None
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), **({"pg_options": opts} if opts else {}))
    try:
        if args.workload == "config4":
            run_config4(args, rank, local_rank, world)
        else:
            run_ours(args, rank, local_rank, world)
    finally:
        if world > 1:
            import torch.distributed as dist

            dist.destroy_process_group()


if __name__ == "__main__":
    main()
