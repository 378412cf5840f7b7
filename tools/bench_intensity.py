"""Cost of the intensity credible intervals (PixelBlock.moments, nf_ns_intensity, CubeFitter(intensity_marginals=True))
on one GPU.

  python tools/bench_intensity.py [--vectors 1048576] [--host-vectors 131072] [--reps 3] [--cube-size 128]
                                  [--cube-reps 2] [--skip-moments] [--out FILE]

(a) vectors/s of the moments mode of the hyperfine kernel at the bench axis (NH3 (1,1)+(2,2), 2 x 1000 channels of
    0.07 km/s), single-component vectors drawn from the priors: the device-resident call timed with CUDA events,
    and, alternated in the same run, the host-buffer calls PixelBlock.moments against PixelBlock.predict followed
    by numpy's max and float64 sum over the channels (the peaks must agree bit for bit).
(b) rows/s of nf_ns_intensity on one cube wave: the 2-component runs of a 64 x 64 patch of the configs[2] cube.
(c) pixels/s of CubeFitter.fit_cube on the configs[2] cube (ncomp <= 3, 2 x 1000 channels, 0.1 K, store with
    posteriors), intensity_marginals off and on, alternated, with the writer-thread time of the intensity pass.
Prints one JSON object, with the device name and power limit read in the same run."""
import argparse
import json
import shutil
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import nestfit_b200 as nb  # noqa: E402
from nestfit_b200 import _lib  # noqa: E402
from oracle import oracle as orc  # noqa: E402

N_CHAN, DV, NOISE = 1000, 0.07, 0.1          # bench.py's axis and noise


def device_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        power = q.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def single_vectors(rng, n):
    ut = nb.get_irdc_priors()
    P = orc.prior_transform(ut.pack(), rng.uniform(size=(2 * n, 6)), 1)
    return np.ascontiguousarray(P[np.isfinite(P).all(axis=1)][:n])


def moments_rates(n_vec, n_host, reps, steps=5, seed=0):
    import torch
    rng = np.random.default_rng(seed)
    xs = [orc.bench_axis(1, N_CHAN, DV), orc.bench_axis(2, N_CHAN, DV)]
    blk = nb.PixelBlock("ammonia", xs, np.zeros((1, 2, N_CHAN), np.float32), NOISE, trans_ids=[1, 2])
    P = single_vectors(rng, n_vec)
    lib = _lib.load()
    dev = torch.device("cuda:0")
    Pd = torch.from_numpy(P).to(dev)
    pk = torch.empty((n_vec, 2), dtype=torch.float32, device=dev)
    sm = torch.empty((n_vec, 2), dtype=torch.float64, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    def launch():
        _lib.check(lib.nf_predict_moments(blk.handle, Pd.data_ptr(), _lib.NF_F64, None, n_vec, 0, pk.data_ptr(),
                                          sm.data_ptr(), stream), "nf_predict_moments")

    launch()
    torch.cuda.synchronize()
    dev_t = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            launch()
        e1.record()
        e1.synchronize()
        dev_t.append(e0.elapsed_time(e1) / 1e3 / steps)
    Ph = P[:n_host]
    blk.moments(Ph[:4096])
    blk.predict(Ph[:4096], 1)
    host = {"moments": [], "predict_then_host_reduce": []}
    same = True
    for _ in range(reps):               # A/B alternated
        t0 = time.perf_counter()
        a_pk, a_sm = blk.moments(Ph)
        t1 = time.perf_counter()
        pred = blk.predict(Ph, 1)
        b_pk, b_sm = pred.max(axis=2), pred.sum(axis=2, dtype=np.float64)
        t2 = time.perf_counter()
        host["moments"].append(t1 - t0)
        host["predict_then_host_reduce"].append(t2 - t1)
        same = same and np.array_equal(a_pk, b_pk)
        rel = float(np.max(np.abs(a_sm - b_sm) / np.maximum(np.abs(pred).sum(axis=2, dtype=np.float64), 1e-300)))
        del pred
    res = {"vectors_device": n_vec, "vectors_host": n_host, "n_chan": [N_CHAN, N_CHAN], "reps": reps,
           "device_moments_vectors_per_s_median": n_vec / float(np.median(dev_t)),
           "device_call_ms": [round(1e3 * t, 3) for t in dev_t],
           "peak_bit_identical_to_predict": bool(same), "sum_max_rel_diff": rel}
    for k, t in host.items():
        res[f"host_{k}_vectors_per_s_median"] = n_host / float(np.median(t))
        res[f"host_{k}_s"] = [round(x, 3) for x in t]
    res["host_moments_over_predict"] = (res["host_moments_vectors_per_s_median"] /
                                        res["host_predict_then_host_reduce_vectors_per_s_median"])
    blk.close()
    return res


def config2_stack(size, seed=77):
    """The configs[2] cube of bench.py: truth ncomp 0..3 in spatial blocks, 2 x 1000 channels, 0.1 K."""
    from nestfit_b200.synth import make_synth_stack
    lon, lat = np.indices((size, size))
    b = max(1, size // 4)
    ncomp_map = ((lon // b) + (lat // b)) % 4
    return make_synth_stack((size, size), nb.get_irdc_priors(), ncomp_map=ncomp_map, n_chan=N_CHAN, dv=DV,
                            noise=NOISE, seed=seed)


def wave_rate(stack, side=64, reps=3):
    """nf_ns_intensity on the 2-component runs of a side x side patch of the cube (one sampler = one wave)."""
    from nestfit_b200.sampler import NestedSamplingBatch
    lon, lat = (a.ravel() for a in np.indices((side, side)))
    data, noise, _ = stack.block_arrays(lon, lat)
    blk = nb.PixelBlock("ammonia", [c.xarr for c in stack.cubes], data, noise, trans_ids=[1, 2])
    snr = np.maximum(np.max(data.max(axis=2) / noise, axis=1), 0.0)
    ns = NestedSamplingBatch(blk, nb.get_irdc_priors(), 2, nlive=100 + (5 * snr).astype(int), tol=1.0, seed=3)
    t0 = time.perf_counter()
    ns.run()
    t_fit = time.perf_counter() - t0
    prod = ns.products_all(marginals=True, posteriors=False)
    rows = int(prod["row_offsets"][-1])
    ns.intensity_marginals()                      # warm-up
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        ns.intensity_marginals()
        ts.append(time.perf_counter() - t0)
    ns.close()
    blk.close()
    t = float(np.median(ts))
    return {"runs": side * side, "ncomp": 2, "rows": rows, "vectors": 2 * rows, "sampler_s": round(t_fit, 3),
            "intensity_s": [round(x, 4) for x in ts], "rows_per_s_median": rows / t,
            "fraction_of_sampler_time": t / t_fit}


def cube_ab(stack, reps):
    from nestfit_b200.models import ammonia
    root = Path(tempfile.mkdtemp(prefix="nf_bench_intensity_"))
    n_pix = stack.spatial_shape[0] * stack.spatial_shape[1]
    out = {"off": [], "on": []}
    extra = {"on_intensity_s": [], "on_store_s": [], "off_store_s": []}
    nbest = {}
    try:
        for k in range(reps):
            for mode in ("off", "on"):            # alternated
                fitter = nb.CubeFitter(stack, nb.get_irdc_priors(), ammonia.AmmoniaRunner, ncomp_max=3, lnZ_thresh=11,
                                       mn_kwargs={'nlive': 100, 'tol': 1.0, 'efr': 0.3}, nlive_snr_fact=5, n_prop=32,
                                       store_posteriors=True, intensity_marginals=mode == "on")
                t0 = time.perf_counter()
                res = fitter.fit_cube(str(root / f"{mode}{k}"), nproc=1)[0]
                wall = time.perf_counter() - t0
                out[mode].append(wall)
                print(f"cube fit {mode} {k}: {wall:.2f} s, intensity pass {res.get('intensity_seconds', 0.0):.2f} s",
                      file=sys.stderr, flush=True)
                extra[f"{mode}_store_s"].append(round(res.get("store_seconds", 0.0), 3))
                if mode == "on":
                    extra["on_intensity_s"].append(round(res.get("intensity_seconds", 0.0), 3))
                nbest[mode] = res["nbest"]
                shutil.rmtree(root / f"{mode}{k}.store", ignore_errors=True)
    finally:
        shutil.rmtree(root, ignore_errors=True)
    r = {"cube": [stack.spatial_shape[0], stack.spatial_shape[1], 2, N_CHAN], "ncomp_max": 3, "reps": reps,
         "store_posteriors": True, "nbest_identical": bool(np.array_equal(nbest["off"], nbest["on"]))}
    for mode, t in out.items():
        r[f"{mode}_pixels_per_s_median"] = n_pix / float(np.median(t))
        r[f"{mode}_seconds"] = [round(x, 3) for x in t]
    r.update(extra)
    r["on_over_off"] = r["on_pixels_per_s_median"] / r["off_pixels_per_s_median"]
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--vectors", type=int, default=1 << 20)
    ap.add_argument("--host-vectors", type=int, default=1 << 17)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cube-size", type=int, default=128, help="side of the configs[2] cube (0 = skip the cube legs)")
    ap.add_argument("--cube-reps", type=int, default=2, help="alternated off/on pairs of the cube fit (0 = skip it)")
    ap.add_argument("--skip-moments", action="store_true")
    ap.add_argument("--out", default=None, help="also write the JSON here")
    args = ap.parse_args()
    name, power = device_info()
    res = {"device": name, "power_limit": power}
    if not args.skip_moments:
        res["moments"] = moments_rates(args.vectors, args.host_vectors, args.reps)
    if args.cube_size > 0:
        stack = config2_stack(args.cube_size)
        res["ns_intensity_wave"] = wave_rate(stack, min(64, args.cube_size), args.reps)
        if args.cube_reps > 0:
            res["cube_fit"] = cube_ab(stack, args.cube_reps)
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
