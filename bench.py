#!/usr/bin/env python3
"""
bench.py -- NH3 log-likelihood throughput (BASELINE.json metric, config 2).

Workload at every N: per GPU, 2^20 parameter vectors (3 velocity components,
18 parameters) scored against 1024 synthetic pixels (2 x 1000 channels, NH3
(1,1)+(2,2), 1024 vectors per pixel); one *step* = one pass of the fused
likelihood kernel over that batch.  `value` = evals/s with inputs resident in
HBM (CUDA-event timed), `e2e` = the same batch through the host-buffer C-ABI
call (H2D of the parameters and D2H of lnL inside the timed region).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

`--steps` sets the number of timed launches of each likelihood path (device-resident, host-buffer pinned and
pageable, Gaussian model).  `--dump-outputs DIR` writes the lnL arrays the device-resident NH3 and Gaussian
calls returned in their last timed step as DIR/nh3_lnl.npy and DIR/gauss_lnl.npy (float64, 8 MB per GPU each,
all ranks in rank order; a fixed seeded sample beyond 64 MB in all, see `dump_outputs`); the inputs are seeded,
so two builds run with the same arguments can be compared output for output.

`--impl reference` times the reference's own CPU implementation of the same path
(oracle/_ref = the unmodified reference compiled by oracle/build_ref.py; the C
oracle port if that is absent) on all host cores, on a bounded sample per step.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

NCOMP = 3
N_PIX = int(os.environ.get("NF_BENCH_NPIX", "1024"))   # profiling runs shrink the batch; the bench uses 1024
VPP = 1024
N_CHAN = 1000
DV = 0.07
NOISE = 0.1
B_TOTAL = N_PIX * VPP
N_SETUP_SFU = 40 * 2 * NCOMP      # SURVEY.md 8d: n_su = 40 * N_spec * ncomp
WORKLOAD = "nh3_loglike_microbench: 2^20 vectors x 3 comp, 1024 px x 1024 vec, 2x1000 ch (configs[1])"


# --------------------------------------------------------------------------
# CPU reference / oracle workers (checker + baseline only)
# --------------------------------------------------------------------------
_W = {}


def _worker_init(kind, xs, data, noise):
    _W["kind"] = kind
    _W["xs"], _W["data"], _W["noise"] = xs, data, noise
    if kind == "reference":
        from oracle import ref
        m = ref.load()
        _W["amm"] = m.ammonia
        _W["specs"] = {}
    else:
        from oracle import oracle as orc
        _W["orc"] = orc


def _worker_run(job):
    params, pix = job
    t0 = time.perf_counter()
    if _W["kind"] == "reference":
        amm = _W["amm"]
        out = np.empty(params.shape[0])
        for b in range(params.shape[0]):
            p = int(pix[b])
            specs = _W["specs"].get(p)
            if specs is None:
                specs = [amm.AmmoniaSpectrum(_W["xs"][t], _W["data"][p, t].copy(), float(_W["noise"][p, t]),
                                             trans_id=t + 1) for t in (0, 1)]
                _W["specs"] = {p: specs}      # keep one pixel's objects alive
            v = params[b].copy()
            lnl = 0.0
            for s in specs:
                amm.amm_predict(s, v)
                lnl += s.loglikelihood
            out[b] = lnl
    else:
        out = _W["orc"].nh3_batch(_W["xs"], [1, 2], params, NCOMP, data=_W["data"], noise=_W["noise"],
                                  pix_of_vec=pix)["lnL"]
    return out, time.perf_counter() - t0


class CpuArm:
    """All-core fan-out of the reference CPU path over a sample of vectors."""

    def __init__(self, xs, data, noise):
        from oracle import ref
        self.kind = "reference" if ref.available() else "port"
        self.cores = os.cpu_count() or 1
        import multiprocessing as mp
        ctx = mp.get_context("fork")
        self.pool = ctx.Pool(self.cores, initializer=_worker_init,
                             initargs=(self.kind, xs, np.asarray(data, dtype=np.float64),
                                       np.asarray(noise, dtype=np.float64)))

    def run(self, params, pix):
        """Score the vectors on all cores; returns (lnL, wall seconds)."""
        n = params.shape[0]
        nj = min(n, self.cores * 4)
        bounds = np.linspace(0, n, nj + 1).astype(int)
        jobs = [(params[a:b], pix[a:b]) for a, b in zip(bounds[:-1], bounds[1:]) if b > a]
        t0 = time.perf_counter()
        res = self.pool.map(_worker_run, jobs)
        wall = time.perf_counter() - t0
        return np.concatenate([r[0] for r in res]), wall

    def close(self):
        self.pool.close()
        self.pool.join()


CKMS = 299792.458
NU_NH3 = (23.6944955e9, 23.722633335e9)      # (1,1), (2,2) rest frequencies [Hz], ammonia.pyx:69-70

# Algorithmic work per evaluation of this exact (seeded) workload, counted once with the reference's FP64
# window rule by tools/count_work.py (the C oracle, test infrastructure) on the 8192-vector sample
# `default_rng(7).choice(B_TOTAL, 8192)`; tests/test_gpu_bench_work.py re-counts and pins these numbers.
WORK_N_GAUSS = 8891.77197265625      # windowed Gaussian exponentials per eval (SURVEY.md 8d: n_g)
WORK_N_RT = 2447.415283203125        # radiative-transfer exponentials per eval (n_rt)
WORK_GAUSS_MODEL = 2563.73388671875            # windowed Gaussians per eval of the 8 x 4096 Gaussian-model workload


def axes():
    """Config-2 axes: v_j = (j - (N-1)/2) dv, x = sort(nu0 (1 - v/c))  (SURVEY.md 8d)."""
    v = (np.arange(N_CHAN) - 0.5 * (N_CHAN - 1)) * DV
    return [np.sort(nu0 * (1.0 - v / CKMS)) for nu0 in NU_NH3]


# --------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(np.max(smax)) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------
def build_problem(nb, rank):
    """Synthetic config-2 problem built with the product's own kernels."""
    ut = nb.get_irdc_priors()
    xs = axes()
    rng = np.random.default_rng(1234)
    # truth per pixel: ncomp_true in {1,2,3} cyclic, drawn through the prior; the model spectra
    # come from the predict kernel (1-, 2-, 3-component launches), plus N(0, sigma^2) noise
    clean = np.zeros((N_PIX, 2, N_CHAN), dtype=np.float32)
    scratch = nb.PixelBlock("ammonia", xs, np.zeros((1, 2, N_CHAN), dtype=np.float32), NOISE, trans_ids=[1, 2])
    for nc in (1, 2, 3):
        idx = np.arange(nc - 1, N_PIX, 3)
        U = rng.uniform(size=(idx.size * 2, 6 * nc))
        T = ut.transform_batch(U, nc)
        T = T[np.isfinite(T).all(axis=1)][:idx.size]
        clean[idx] = scratch.predict(T, nc)
    scratch.close()
    data = clean + rng.normal(0.0, NOISE, size=clean.shape).astype(np.float32)
    noise = np.full((N_PIX, 2), NOISE)
    U = np.random.default_rng(4321 + rank).uniform(size=(B_TOTAL, 6 * NCOMP))
    P = ut.transform_batch(U, NCOMP)
    bad = ~np.isfinite(P).all(axis=1)
    if bad.any():       # redraw non-finite rows (SURVEY.md 8d)
        good = np.flatnonzero(~bad)
        P[bad] = P[good[: bad.sum()]]
    return xs, data, noise, P.astype(np.float32)


def run_ours(args):
    import torch
    import nestfit_b200 as nb
    from nestfit_b200 import _lib
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = _lib.load()
    dev = local_rank

    xs, data, noise, P32 = build_problem(_with_device(nb, dev), rank)
    blk = nb.PixelBlock("ammonia", xs, data, noise, trans_ids=[1, 2], device=dev)
    d_params = torch.from_numpy(P32).to(f"cuda:{dev}")
    d_lnl = torch.empty(B_TOTAL, dtype=torch.float64, device=f"cuda:{dev}")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{dev}")   # > 126 MB L2
    stream = torch.cuda.current_stream().cuda_stream

    def launch():
        _lib.check(lib.nf_nh3_loglike(blk.handle, d_params.data_ptr(), _lib.NF_F32, None, VPP, B_TOTAL, NCOMP, 0,
                                      d_lnl.data_ptr(), stream), "nf_nh3_loglike")

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        flush.zero_()
        launch()
    barrier()
    sampler = ClockSampler(dev)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for k in range(args.steps):
        flush.zero_()                     # L2 flush between timed iterations (outside the event pair)
        ev[k][0].record()
        launch()
        ev[k][1].record()
    barrier()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = float(sum(step_ms))
    lnl_dev = d_lnl.cpu().numpy()

    # ---- end to end through the host-buffer C-ABI call (pinned host memory) ----
    h_params = torch.from_numpy(P32).pin_memory()
    h_lnl = torch.empty(B_TOTAL, dtype=torch.float64).pin_memory()
    hp, hl = h_params.numpy(), h_lnl.numpy()

    def e2e_call():
        _lib.check(lib.nf_nh3_loglike_host(blk.handle, _lib.ptr(hp), _lib.NF_F32, None, VPP, B_TOTAL, NCOMP, 0,
                                           _lib.ptr(hl)), "nf_nh3_loglike_host")

    for _ in range(2):
        e2e_call()
    n_e2e = args.steps
    barrier()
    t0 = time.perf_counter()
    for _ in range(n_e2e):
        e2e_call()
    barrier()
    e2e_s = time.perf_counter() - t0
    clocks = sampler.stop()
    assert np.allclose(hl, lnl_dev, rtol=1e-12, atol=1e-9), "host-call and device-call results differ"
    # the same call with plain (pageable) numpy buffers, what a reference-side caller hands over
    pp, pl = P32.copy(), np.empty(B_TOTAL)

    def e2e_pageable():
        _lib.check(lib.nf_nh3_loglike_host(blk.handle, _lib.ptr(pp), _lib.NF_F32, None, VPP, B_TOTAL, NCOMP, 0,
                                           _lib.ptr(pl)), "nf_nh3_loglike_host")
    e2e_pageable()
    barrier()
    t0 = time.perf_counter()
    for _ in range(n_e2e):
        e2e_pageable()
    barrier()
    e2e_pg_s = time.perf_counter() - t0

    times = torch.tensor([total_ms, e2e_s, e2e_pg_s], dtype=torch.float64, device=f"cuda:{dev}")
    if dist is not None:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    total_ms, e2e_s, e2e_pg_s = float(times[0]), float(times[1]), float(times[2])

    outputs = {"nh3_lnl": d_lnl}
    gauss_result = None
    if not args.no_gauss:
        gauss_result, outputs["gauss_lnl"] = run_gauss(nb, lib, _lib, dev, rank, dist, args.steps)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs, dist, rank)
    cube_result = None
    if args.cube_size > 0 or args.scale_cube != "0x0" or args.full_cube:
        del d_params, d_lnl, flush, outputs
        torch.cuda.empty_cache()
        cube_result = run_cube_fit(nb, args, rank, world, dev, dist)
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    evals = float(B_TOTAL) * world
    value = evals * args.steps / (total_ms * 1e-3)
    cube = cube_result
    e2e_value = evals * n_e2e / e2e_s

    # ---- roofline of the dominant (only) kernel --------------------------------
    ns = 8192
    n_g, n_rt = WORK_N_GAUSS, WORK_N_RT
    sfu_per_eval = n_g + n_rt + N_SETUP_SFU
    flop_per_eval = 5 * n_g + 8 * n_rt + 3 * 2 * N_CHAN + 30 * NCOMP * (18 + 21)
    mufu = _lib.C.c_double()
    ffma = _lib.C.c_double()
    _lib.check(lib.nf_measure_peaks(dev, _lib.C.byref(mufu), _lib.C.byref(ffma)), "nf_measure_peaks")
    launch_s = (total_ms * 1e-3) / args.steps
    ach_sfu = B_TOTAL * sfu_per_eval / launch_s * 1e-9          # Gop/s, one GPU
    ach_fp32 = B_TOTAL * flop_per_eval / launch_s * 1e-9
    bound = "sfu" if sfu_per_eval / mufu.value >= flop_per_eval / ffma.value else "fp32"
    peak = mufu.value if bound == "sfu" else ffma.value
    ach = ach_sfu if bound == "sfu" else ach_fp32
    traffic = None
    tp = ROOT / "profiles" / "traffic.json"
    if tp.exists():
        try:
            traffic = json.loads(tp.read_text()).get("nf_like_kernel_dram_bytes_per_launch")
        except Exception:
            traffic = None
    roofline = {
        "bound": bound, "achieved": ach, "peak": peak, "unit": "Gop/s" if bound == "sfu" else "GFLOP/s",
        "frac": ach / peak, "traffic": traffic,
        "traffic_source": "stored figure: dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture of "
                          "this kernel on this workload (profiles/traffic.json), not measured in this run",
        "peak_source": "measured live by nf_measure_peaks (MUFU.EX2 / FFMA register loops, this box)",
        "work_per_eval": {"n_gauss": n_g, "n_rt": n_rt, "n_setup": N_SETUP_SFU, "sfu_ops": sfu_per_eval,
                          "fp32_flop": flop_per_eval, "counted_on": f"{ns}-vector host sample of this seeded workload (tools/count_work.py: reference window "
                                        "rule in FP64; pinned by tests/test_gpu_bench_work.py)"},
        "fp32": {"achieved_gflops": ach_fp32, "peak_gflops": ffma.value, "frac": ach_fp32 / ffma.value},
        "hbm": {"algorithmic_bytes_per_launch": B_TOTAL * (4 * 6 * NCOMP + 8) + N_PIX * 2 * 1024 * 4,
                "note": "80 B per eval + 8 KB per pixel staged once per CTA tile; not the bound"},
    }

    line = {
        "metric": "NH3 loglike evals/s (3-comp, 2x1000 ch)", "value": value, "unit": "evals/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32 (f64 set-up and lnL accumulation)", "data": "synthetic",
        "config": {"workload": WORKLOAD, "vectors_per_gpu": B_TOTAL, "pixels_per_gpu": N_PIX, "ncomp": NCOMP,
                   "n_chan": [N_CHAN, N_CHAN], "l2": "flushed between timed iterations (256 MB memset)",
                   "parallelism": f"replicated pixels, disjoint vector batches x{world}"},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "evals/s", "h2d_bytes_per_step": int(P32.nbytes),
                "d2h_bytes_per_step": int(B_TOTAL * 8), "steps": n_e2e,
                "api": "nf_nh3_loglike_host (pinned host buffers, chunks pipelined over a ring of 3 streams)",
                "pageable_host_buffers": {"value": evals * n_e2e / e2e_pg_s, "unit": "evals/s",
                                          "note": "same call, plain numpy arrays (what a reference-side caller passes): bounced through the "
                                                  "library's page-locked ring by 4 host threads"}},
        "gpu_launches": args.steps,
        "roofline": roofline,
    }

    # ---- CPU baseline beside it (rank 0, N = 1 only) ---------------------------
    if world == 1 and not args.no_cpu:
        arm = CpuArm(xs, data, noise)
        pilot_n = 64 * arm.cores
        pix_all = (np.arange(B_TOTAL) // VPP).astype(np.int32)
        _, w = arm.run(P32[:pilot_n].astype(np.float64), pix_all[:pilot_n])
        rate = pilot_n / w
        n_s = int(min(B_TOTAL, max(pilot_n, rate * 12.0)))
        n_s = (n_s // VPP) * VPP or VPP
        lnl_cpu, w = arm.run(P32[:n_s].astype(np.float64), pix_all[:n_s])
        arm.close()
        err = np.abs(lnl_cpu - lnl_dev[:n_s])
        # BASELINE north_star: 1e-3 absolute within 1e3 of the best attainable lnL, 1e-6 relative for the poor fits.
        # The batch is prior-drawn (no vector is near a pixel's posterior), so "best attainable" is the
        # expectation at the truth, -N_chan/2 (minus five sigma of a chi-square with N_chan degrees of freedom)
        n_ch = 2 * N_CHAN
        near = lnl_cpu >= -(0.5 * n_ch + 5.0 * math.sqrt(0.5 * n_ch)) - 1e3
        i_abs, i_rel = int(np.argmax(err)), int(np.argmax(err / np.abs(lnl_cpu)))
        line["cpu_baseline"] = {
            "value": n_s / w, "unit": "evals/s", "cores": arm.cores, "kind": arm.kind,
            "sample": f"first {n_s} vectors of the same batch ({n_s // VPP} pixels), fork pool over all cores",
            "max_abs_dlnL_vs_gpu": float(err[i_abs]), "lnL_at_max_abs_dlnL": float(lnl_cpu[i_abs]),
            "max_rel_dlnL_vs_gpu": float(err[i_rel] / abs(lnl_cpu[i_rel])), "lnL_at_max_rel_dlnL": float(lnl_cpu[i_rel]),
            "vectors_within_1e3_of_best": int(near.sum()),
            "max_abs_dlnL_within_1e3_of_best": float(err[near].max()) if near.any() else None,
            "parity_ok": bool((err[near] <= 1e-3).all() and (err[~near] <= 1e-6 * np.abs(lnl_cpu[~near])).all()),
            "parity_rule": "|dlnL| <= 1e-3 within 1e3 of the best attainable lnL (-N_chan/2), <= 1e-6 |lnL| elsewhere",
        }
    if gauss_result is not None:
        line["gauss_loglike"] = gauss_result
    if cube is not None:
        line.update(cube)
    emit(line)
    if dist is not None:
        dist.destroy_process_group()


def run_gauss(nb, lib, _lib, dev, rank, dist, n_it):
    """Secondary metric (BASELINE configs[4]): Gaussian model, 8 components over 4096 channels, 2^20 vectors per
    GPU against 256 pixels (replicated data, disjoint vector slices); device-resident evals/s over `n_it` timed
    launches, max over ranks.  Returns (result line or None off rank 0, device lnL of the last launch)."""
    import torch
    from nestfit_b200.parallel import max_over_ranks
    B, n_chan, ncomp, n_pix = 1 << 20, 4096, 8, 256
    rng = np.random.default_rng(5 + rank)
    v = (np.arange(n_chan) - 2047.5) * 0.05
    x = np.sort(NU_NH3[0] * (1 - v / CKMS))
    P = np.concatenate([np.sort(rng.uniform(-90, 90, (B, ncomp)), axis=1), rng.uniform(0.2, 3, (B, ncomp)),
                        rng.uniform(0.1, 5, (B, ncomp))], axis=1).astype(np.float32)
    scratch = nb.PixelBlock("gaussian", [x], np.zeros((1, 1, n_chan), np.float32), 0.1, rest_freq=NU_NH3[0], device=dev)
    clean = scratch.predict(P[:n_pix], ncomp)
    scratch.close()
    data = clean + np.random.default_rng(6).normal(0, 0.1, clean.shape).astype(np.float32)
    blk = nb.PixelBlock("gaussian", [x], data, 0.1, rest_freq=NU_NH3[0], device=dev)
    d_p = torch.from_numpy(P).to(f"cuda:{dev}")
    d_l = torch.empty(B, dtype=torch.float64, device=f"cuda:{dev}")
    st = torch.cuda.current_stream().cuda_stream

    def launch():
        _lib.check(lib.nf_gauss_loglike(blk.handle, d_p.data_ptr(), _lib.NF_F32, None, B // n_pix, B, ncomp,
                                        d_l.data_ptr(), st), "nf_gauss_loglike")
    for _ in range(3):
        launch()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n_it):
        launch()
    e1.record()
    torch.cuda.synchronize()
    ms = max_over_ranks(e0.elapsed_time(e1) / n_it, dist, device=f"cuda:{dev}")
    blk.close()
    if rank != 0:
        return None, d_l
    world = 1 if dist is None else dist.get_world_size()
    return {"metric": "Gaussian loglike evals/s (8-comp, 4096 ch)", "value": world * B / (ms * 1e-3), "unit": "evals/s",
            "ms_per_launch": ms, "launches": n_it, "vectors_per_gpu": B, "windowed_gaussians_per_eval": WORK_GAUSS_MODEL,
            "scaling": "weak"}, d_l


def _shared_cube(nb, shape, ncomp_max, noise_grad, seed, dev, rank, dist, tag):
    """The synthetic cube of a cube-fit leg (SURVEY.md 8d configs 3/4): truth ncomp 0..ncomp_max in spatial blocks,
    sigma = 0.1 K or a smooth 0.05..0.3 K gradient through `NoiseMap`.  Built once on rank 0 with the predict
    kernel and shared with the other ranks through /dev/shm (memory-mapped), outside every timed region."""
    import torch
    from nestfit_b200.synth import make_synth_stack, velocity_axis_hz
    ut = nb.get_irdc_priors()
    port = os.environ.get("MASTER_PORT", "0")
    shm = Path("/dev/shm" if Path("/dev/shm").is_dir() else "/tmp") / f"nf_bench_{port}_{tag}"
    lon, lat = np.indices(shape)
    b = max(1, min(shape) // 4)
    ncomp_map = ((lon // b) + (lat // b)) % (ncomp_max + 1)
    noise = 0.05 + 0.25 * (lon + lat) / float(shape[0] + shape[1] - 2) if noise_grad else NOISE
    if rank == 0:
        shm.mkdir(parents=True, exist_ok=True)
        stack = make_synth_stack(shape, ut, ncomp_map=ncomp_map, n_chan=N_CHAN, dv=DV, noise=noise, seed=seed, device=dev)
        for t, c in enumerate(stack.cubes):
            np.save(shm / f"cube{t}.npy", c.data)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    xs = [velocity_axis_hz(1, N_CHAN, DV), velocity_axis_hz(2, N_CHAN, DV)]
    nm = nb.NoiseMap(np.asarray(noise).T.copy()) if noise_grad else NOISE
    cubes = [nb.DataCube.from_arrays(np.load(shm / f"cube{t}.npy", mmap_mode="r"), xs[t], nm, trans_id=t + 1,
                                     header={'CTYPE1': 'RA---SIN', 'CTYPE2': 'DEC--SIN', 'NAXIS1': shape[0],
                                             'NAXIS2': shape[1]}) for t in (0, 1)]
    return nb.CubeStack(cubes), ut, ncomp_map, shm


def _cube_leg(nb, shape, ncomp_max, noise_grad, seed, rank, world, dev, dist, tag, blocks_per_gpu, posteriors=True,
              concurrent_blocks=2, n_streams=1, pixels_per_stream=1024):
    """One cube-fit leg through the public API: `CubeFitter.fit_cube` at N = 1, its SPMD form `fit_cube_rank` (one
    existing process per GPU, blocks claimed dynamically, one store chunk per rank) at N > 1.  The timed region
    holds everything the call does: store creation, uploads, the fit, the posterior products, the chunk writes."""
    import shutil
    import torch
    from nestfit_b200.models import ammonia
    stack, ut, ncomp_map, shm = _shared_cube(nb, shape, ncomp_max, noise_grad, seed, dev, rank, dist, tag)
    fitter = nb.CubeFitter(stack, ut, ammonia.AmmoniaRunner, ncomp_max=ncomp_max, lnZ_thresh=11,
                           mn_kwargs={'nlive': 100, 'tol': 1.0, 'efr': 0.3}, nlive_snr_fact=5, n_prop=32,
                           store_posteriors=posteriors, n_streams=n_streams if world == 1 else 1,
                           pixels_per_stream=pixels_per_stream)
    store_root = Path(os.environ.get("NF_BENCH_STORE", "/tmp")) / f"nf_bench_store_{os.environ.get('MASTER_PORT', '0')}_{tag}"
    if rank == 0:
        shutil.rmtree(store_root, ignore_errors=True)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    barrier()
    t0 = time.perf_counter()
    if world == 1:
        results = fitter.fit_cube(str(store_root / "cube"), nproc=1, devices=[dev])
    else:
        results = fitter.fit_cube_rank(str(store_root / "cube"), rank, world, blocks_per_gpu=blocks_per_gpu, device=dev,
                                       barrier=barrier, concurrent_blocks=concurrent_blocks)
    barrier()
    wall = time.perf_counter() - t0
    # per-rank bookkeeping -> rank 0
    mine = {"busy_s": float(fitter.stats.get("rank_fit_seconds", sum(r["seconds"] for r in results))), "n_evals": int(sum(r["n_evals"] for r in results)),
            "n_pix": int(sum(np.asarray(r["nbest"]).size for r in results)),
            "blocks": int(sum(len(r.get("blocks", [0])) for r in results)),
            "store_s": float(sum(r.get("store_seconds", 0.0) for r in results)),
            "store_wait_s": float(sum(r.get("store_wait_seconds", 0.0) for r in results)),
            "n_truncated": int(sum(r.get("n_truncated", 0) for r in results)), "wall_s": wall,
            "evals_by_ncomp": np.sum([r["evals_by_ncomp"] for r in results], axis=0).tolist() if results else []}
    nbest_local = np.full(shape, -9, dtype=np.int64)
    for r in results:
        nbest_local[r["i_lon"], r["i_lat"]] = r["nbest"]
    per_rank = [mine]
    if dist is not None:
        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine)
        t = torch.from_numpy(nbest_local).to(f"cuda:{dev}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        nbest_local = t.cpu().numpy()
    out = None
    if rank == 0:
        wall = max(p["wall_s"] for p in per_rank)
        n_pix = shape[0] * shape[1]
        assert sum(p["n_pix"] for p in per_rank) == n_pix and (nbest_local >= 0).all()
        du = subprocess.run(["du", "-sb", str(store_root)], capture_output=True, text=True).stdout.split()
        store = nb.HdfStore(str(store_root / "cube"))
        n_groups = sum(1 for _ in store.iter_pix_groups())
        store.close()
        out = {"value": n_pix / wall, "unit": "pixels/s", "seconds": wall, "cube": [shape[0], shape[1], 2, N_CHAN],
               "ncomp_max": ncomp_max, "noise": "0.05..0.3 K gradient (NoiseMap)" if noise_grad else "0.1 K uniform",
               "nlive": "100 + 5*SNR", "tol": 1.0, "lnZ_thresh": 11, "blocks_per_gpu": blocks_per_gpu if world > 1 else 1,
               "api": f"CubeFitter(n_streams={n_streams}, pixels_per_stream={pixels_per_stream}).fit_cube(store, nproc=1)"
                      if world == 1 else
                      f"CubeFitter.fit_cube_rank(store, rank, {world}, blocks_per_gpu={blocks_per_gpu}, "
                      f"concurrent_blocks={concurrent_blocks})",
               "likelihood_evals_per_pixel": sum(p["n_evals"] for p in per_rank) / n_pix,
               "likelihood_evals_by_ncomp": np.sum([p["evals_by_ncomp"] for p in per_rank], axis=0).tolist(),
               "nbest_matches_truth": float((np.minimum(nbest_local, ncomp_max) == ncomp_map).mean()),
               "rank_busy_fraction": [p["busy_s"] / wall for p in per_rank],
               "rank_blocks": [p["blocks"] for p in per_rank], "rank_pixels": [p["n_pix"] for p in per_rank],
               "store": {"bytes": int(du[0]) if du else None, "pixel_groups": n_groups, "posteriors": bool(posteriors),
                         "writer_seconds_sum": sum(p["store_s"] for p in per_rank),
                         "exposed_wait_seconds_max_rank": max(p["store_wait_s"] for p in per_rank),
                         "exposed_fraction_of_wall": max(p["store_wait_s"] for p in per_rank) / wall},
               "runs_repeated_after_truncation": sum(p["n_truncated"] for p in per_rank)}
        shutil.rmtree(store_root, ignore_errors=True)
    barrier()
    if rank == 0:
        shutil.rmtree(shm, ignore_errors=True)
    return out, (stack, ut, nbest_local)


def run_cube_fit(nb, args, rank, world, dev, dist):
    """BASELINE metric M2, cube pixels/s with full evidence model selection, through CubeFitter with the store on:
      * N = 1: configs[2] (size x size, ncomp <= 3, uniform noise) -> `cube_fit_config2`
      * every N: ONE fixed configs[3]-shaped cube (ncomp <= 4, noise gradient) cut into blocks over the N GPUs
        -> `cube_fit` (strong scaling)
      * N = 8 (or --full-cube): the full 512 x 512 configs[3] cube -> `cube_fit_full`."""
    legs = {}
    sx, sy = (int(v) for v in args.scale_cube.lower().split("x"))

    def leg(key, *a, **kw):
        """One leg.  On a single process a failing leg (a full disk under the 55 GB store, say) is reported under
        its key and the line with the headline metric is still printed; with several ranks the error propagates
        (the ranks meet in collectives)."""
        try:
            return _cube_leg(nb, *a, **kw)
        except Exception as exc:
            if world > 1:
                raise
            import traceback
            traceback.print_exc(file=sys.stderr)
            legs[key] = {"error": f"{type(exc).__name__}: {exc}"}
            import shutil
            port = os.environ.get("MASTER_PORT", "0")       # what the leg left behind must not starve the next one
            for root in (Path(os.environ.get("NF_BENCH_STORE", "/tmp")), Path("/dev/shm"), Path("/tmp")):
                for left in list(root.glob(f"nf_bench_store_{port}_*")) + list(root.glob(f"nf_bench_{port}_*")):
                    shutil.rmtree(left, ignore_errors=True)
            return None, None

    if world == 1 and args.cube_size > 0:
        out, aux = leg("cube_fit_config2", (args.cube_size, args.cube_size), 3, False, 77, rank, world, dev, dist, "c2", 1,
                       n_streams=args.cube_streams, pixels_per_stream=args.cube_pps)
        if rank == 0 and out is not None:
            out["metric"] = "cube pixels/s fit (configs[2]: ncomp 1-3 evidence model selection, 1 GPU)"
            out["scaling"] = "n/a (single GPU)"
            if not args.no_cpu:
                out["cpu_baseline"] = cube_cpu_baseline(aux[0], aux[1], (args.cube_size, args.cube_size), aux[2])
            legs["cube_fit_config2"] = out
    if sx > 0:
        out, _ = leg("cube_fit", (sx, sy), 4, True, 78, rank, world, dev, dist, "c3", args.blocks_per_gpu,
                     concurrent_blocks=args.concurrent_blocks, n_streams=args.cube_streams,
                     pixels_per_stream=args.cube_pps)
        if rank == 0 and out is not None:
            out["metric"] = "cube pixels/s fit (configs[3] shape: ncomp <= 4, noise map; one fixed cube over N GPUs)"
            out["scaling"] = "strong"
            legs["cube_fit"] = out
    if args.full_cube or world == 8:
        # the posterior rows of 262 144 pixels are ~400 GB: this leg stores everything but them (attributes,
        # marginals, best-fit / MAP vectors); the two smaller legs store the posteriors as well
        out, _ = leg("cube_fit_full", (512, 512), 4, True, 79, rank, world, dev, dist, "c3full", args.blocks_per_gpu,
                     posteriors=False, concurrent_blocks=args.concurrent_blocks, n_streams=args.cube_streams,
                     pixels_per_stream=args.cube_pps)
        if rank == 0 and out is not None:
            out["metric"] = "cube pixels/s fit (configs[3]: 512x512, ncomp <= 4, noise map)"
            out["scaling"] = "strong"
            legs["cube_fit_full"] = out
    return legs if rank == 0 else None


def _cube_cpu_worker(ix):
    from oracle import ns_port
    xs, packed, data, noise = _W["cube"]
    t0 = time.perf_counter()
    r = ns_port.fit_pixel(xs, [1, 2], data[ix], noise[ix], packed, ncomp_max=3, lnZ_thresh=11, nlive=100,
                          nlive_snr_fact=5, tol=1.0, efr=0.3, n_prop=32, seed=1000 + ix)
    return r["nbest"], r["n_evals"], time.perf_counter() - t0


CUBE_CPU_CAP_S = 90.0      # wall-time cap of the cube-fit CPU baseline: keeps the default run within a few minutes


def _cube_cpu_worker_ix(ix):
    return ix, _cube_cpu_worker(ix)


def cube_cpu_baseline(stack, ut, shape, nbest_gpu):
    """CPU baseline of the cube-fit metric (SURVEY.md 8d): the same batched nested-sampling scheme and ncomp
    escalation as a numpy port (oracle/ns_port.py) scored with the C oracle likelihood, one pixel per host core
    (MultiNest, the reference's sampler, is an external Fortran library that is not available)."""
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    n_tot = shape[0] * shape[1]
    # one pixel per core, spread over the cube so that every true ncomp (0..3, in blocks) is represented
    flat = (np.arange(cores) * (n_tot / cores) + 0.37 * n_tot / cores).astype(int) % n_tot
    lon, lat = np.unravel_index(flat, shape)
    data, noise, _ = stack.block_arrays(lon, lat)
    _W["cube"] = ([np.asarray(c.xarr, dtype=np.float64) for c in stack.cubes], ut.pack(),
                  np.asarray(data, dtype=np.float64), np.asarray(noise, dtype=np.float64))
    t0 = time.perf_counter()
    res, done_ix = [], []
    cap_s = CUBE_CPU_CAP_S
    with mp.get_context("fork").Pool(cores) as pool:
        it = pool.imap_unordered(_cube_cpu_worker_ix, range(cores), chunksize=1)
        try:
            for _ in range(cores):
                ix, r = it.next(timeout=max(1.0, cap_s - (time.perf_counter() - t0)))
                done_ix.append(ix)
                res.append(r)
        except mp.TimeoutError:
            pool.terminate()          # the most expensive pixels did not finish within the cap
    wall = time.perf_counter() - t0
    if not res:
        return {"value": None, "unit": "pixels/s", "cores": cores, "kind": "port",
                "sample": f"no pixel finished within {cap_s:.0f} s"}
    lon, lat = lon[done_ix], lat[done_ix]
    nb_cpu = np.array([r[0] for r in res])
    # throughput of a cube of many such pixels with every core kept busy (the wall time of this small sample is
    # set by its slowest pixel and would understate the CPU)
    # (pixels cut off by the wall-time cap count with the core time they used up but not as fitted pixels)
    busy = float(np.sum([r[2] for r in res])) + (cores - len(res)) * wall
    return {"value": len(res) * cores / busy, "unit": "pixels/s", "cores": cores, "kind": "port",
            "truncated": len(res) < cores,
            "sample": f"{len(res)} of {cores} pixels spread over the cube, one per core (numpy port of the sampler + C "
                      "oracle likelihood, same nlive/tol/efr/escalation)",
            "wall_seconds": wall, "likelihood_evals_per_pixel": float(np.mean([r[1] for r in res])),
            "cpu_seconds_per_pixel": float(np.mean([r[2] for r in res])),
            "nbest_agrees_with_gpu": float((nb_cpu == nbest_gpu[lon, lat]).mean())}


DUMP_LIMIT_BYTES = 64_000_000 - 4096      # 64 MB of files in all, npy headers included


def dump_outputs(dirname, tensors, dist, rank):
    """Write each device output as DIR/<name>.npy in float64 from rank 0: the slices of all ranks in rank order,
    i.e. everything the callers of the multi-GPU path receive.  An array that would take the files past 64 MB
    is replaced by a fixed sample of it: the entries at the sorted indices `default_rng(0).choice(n, k)`."""
    import torch
    arrays = {}
    for name, t in tensors.items():
        if dist is not None:
            parts = [torch.empty_like(t) for _ in range(dist.get_world_size())]
            dist.all_gather(parts, t)
            t = torch.cat(parts)
        arrays[name] = t.double().cpu().numpy()
    if rank != 0:
        return
    k = DUMP_LIMIT_BYTES // (8 * len(arrays))
    out = Path(dirname)
    out.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        if a.size > k:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, k, replace=False))]
        np.save(out / f"{name}.npy", a)


def _with_device(nb, dev):
    """PixelBlock / PriorTransformer helpers default to device 0; bind to `dev`."""
    if dev == 0:
        return nb

    class _NB:
        pass
    o = _NB()
    o.get_irdc_priors = lambda: _DevPriors(nb.get_irdc_priors(), dev)
    o.PixelBlock = lambda *a, **k: nb.PixelBlock(*a, **{**k, "device": dev})
    return o


class _DevPriors:
    def __init__(self, ut, dev):
        self.ut, self.dev = ut, dev

    def transform_batch(self, u, ncomp):
        return self.ut.transform_batch(u, ncomp, device=self.dev)


# --------------------------------------------------------------------------
# reference arm
# --------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    from oracle import ref
    from oracle import oracle as orc
    xs = axes()
    rng = np.random.default_rng(1234)
    n_pix = 64                                   # bounded sample of the workload's pixels
    if ref.available():
        m = ref.load()
        ut = ref.make_irdc_priors(m.core)

        def transform(U, nc):
            P = U.copy()
            for row in P:
                ut.transform(row, nc)
            return P
    else:
        import nestfit_b200.prior_constructors as pc
        packed = pc.get_irdc_priors().pack()

        def transform(U, nc):
            return orc.prior_transform(packed, U, nc)
    clean = np.zeros((n_pix, 2, N_CHAN))
    for nc in (1, 2, 3):
        idx = np.arange(nc - 1, n_pix, 3)
        T = transform(rng.uniform(size=(idx.size * 2, 6 * nc)), nc)
        T = T[np.isfinite(T).all(axis=1)][:idx.size]
        clean[idx] = orc.nh3_batch(xs, [1, 2], T, nc, want_pred=True)["pred"]
    data = (clean + rng.normal(0.0, NOISE, size=clean.shape)).astype(np.float32).astype(np.float64)
    noise = np.full((n_pix, 2), NOISE)
    arm = CpuArm(xs, data, noise)
    # per-step sample sized from a pilot so K + W steps finish within a few minutes
    pilot = 32 * arm.cores
    Ppil = transform(np.random.default_rng(4321).uniform(size=(pilot * 2, 6 * NCOMP)), NCOMP)
    Ppil = Ppil[np.isfinite(Ppil).all(axis=1)][:pilot].astype(np.float32).astype(np.float64)
    _, w = arm.run(Ppil, (np.arange(pilot) % n_pix).astype(np.int32))
    rate = pilot / w
    budget_s = 150.0 / float(args.steps + max(args.warmup, 1))
    n_s = int(max(pilot, min(rate * min(budget_s, 15.0), 1 << 18)))
    n_s = max(n_pix, (n_s // n_pix) * n_pix)
    U = np.random.default_rng(4321).uniform(size=(int(n_s * 1.05) + 64, 6 * NCOMP))
    P = transform(U, NCOMP)
    P = P[np.isfinite(P).all(axis=1)][:n_s].astype(np.float32).astype(np.float64)
    pix = np.sort(np.arange(P.shape[0]) % n_pix).astype(np.int32)
    for _ in range(max(args.warmup, 1)):
        arm.run(P, pix)
    t_tot = 0.0
    for _ in range(args.steps):
        _, w = arm.run(P, pix)
        t_tot += w
    arm.close()
    value = P.shape[0] * args.steps / t_tot
    sample = f"{P.shape[0]} vectors per step over {n_pix} pixels (bounded sample of the 2^20-vector batch)"
    line = {
        "impl": "reference", "metric": "NH3 loglike evals/s (3-comp, 2x1000 ch)", "value": value,
        "unit": "evals/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 1),
        "ms_per_step": 1e3 * t_tot / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "ncomp": NCOMP, "n_chan": [N_CHAN, N_CHAN], "sample": sample},
        "cpu_baseline": {"value": value, "unit": "evals/s", "cores": arm.cores, "kind": arm.kind, "sample": sample},
        "e2e": {"value": value, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


_REAL_STDOUT = None


def quiet_stdout():
    """Libraries (NCCL's version banner, ...) write to fd 1; the contract is ONE JSON line on stdout.
    Point fd 1 at stderr for the duration of the run and keep the real stdout for `emit`."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-gauss", action="store_true", help="skip the secondary Gaussian-model metric")
    ap.add_argument("--cube-size", type=int, default=128,
                    help="side of the configs[2] cube fitted at N = 1 (0 = skip)")
    ap.add_argument("--scale-cube", default="256x128",
                    help="LONxLAT of the fixed configs[3]-shaped cube fitted at every N (strong scaling; 0x0 = skip)")
    ap.add_argument("--full-cube", action="store_true", help="also fit the full 512x512 configs[3] cube (default at N = 8)")
    ap.add_argument("--cube-streams", type=int, default=1,
                    help="N = 1 cube legs: host threads / CUDA streams that escalate sub-blocks of a wave concurrently")
    ap.add_argument("--cube-pps", type=int, default=1024, help="pixels per sub-block when --cube-streams > 1")
    ap.add_argument("--blocks-per-gpu", type=int, default=8, help="over-decomposition of the multi-GPU cube fit")
    ap.add_argument("--concurrent-blocks", type=int, default=2,
                    help="groups of blocks a rank keeps in flight (host threads / streams)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the lnL arrays of the last timed step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed: not available with --impl reference")
    if args.gpus > 1 and "RANK" not in os.environ:
        # convenience: re-launch one process per GPU (the driver does this itself)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 2000), __file__] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    quiet_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
