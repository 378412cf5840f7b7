"""Throughput of spectra on axes of their own (PixelBlock.from_spectra, run_multinest_batch) on one GPU.

  python tools/bench_spectra.py [--vectors 1048576] [--reps 5] [--sources 4096] [--serial 16] [--out FILE]

(a) evals/s of the device-resident NH3 likelihood at the bench shape (3 components, 2 x 1000 channels), on the same
    seeded data held once as a shared-axis block and once as a per-pixel-axes block whose pixels all carry that
    axis; the two are timed alternately, and their lnL must agree bit for bit.
(b) spectra/s for a synthetic catalogue of NH3 (1,1)+(2,2) sources, each on axes of its own (velocity centre,
    channel width, 300-1100 channels, the two spectra of a source often of different lengths) with 1 or 2 true
    components: run_multinest_batch over all sources at ncomp 1 and at ncomp 2, against a serial run_multinest
    loop over the first --serial of the same sources.
Prints one JSON object, with the device name and power limit read in the same run."""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import nestfit_b200 as nb  # noqa: E402
from nestfit_b200 import _lib  # noqa: E402
from oracle import oracle as orc  # noqa: E402

CKMS = 299792.458


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


def likelihood_ab(n_vec, reps, steps, seed=0):
    import torch
    rng = np.random.default_rng(seed)
    ncomp, n_pix = 3, 1024
    vpp = n_vec // n_pix
    ut = nb.get_irdc_priors()
    xs = [orc.bench_axis(1, 1000, 0.07), orc.bench_axis(2, 1000, 0.07)]
    T = orc.prior_transform(ut.pack(), rng.uniform(0.15, 0.85, size=(4 * n_pix, 6 * ncomp)), ncomp)
    T = T[np.isfinite(T).all(axis=1)][:n_pix]
    clean = orc.nh3_batch(xs, [1, 2], T, ncomp, want_pred=True)["pred"]
    data = (clean + rng.normal(0.0, 0.1, clean.shape)).astype(np.float32)
    P = orc.prior_transform(ut.pack(), rng.uniform(size=(n_pix * vpp, 6 * ncomp)), ncomp)
    bad = ~np.isfinite(P).all(axis=1)
    P[bad] = np.repeat(T, vpp, axis=0)[bad]
    shared = nb.PixelBlock("ammonia", xs, data, 0.1, trans_ids=[1, 2])
    spectra = [[nb.AmmoniaSpectrum(xs[s], data[p, s].astype(np.float64), 0.1, s + 1) for s in range(2)]
               for p in range(n_pix)]
    perpix = nb.PixelBlock.from_spectra("ammonia", spectra)
    lib = _lib.load()
    dev = torch.device("cuda:0")
    Pd = torch.from_numpy(P).to(dev)
    out = {k: torch.empty(P.shape[0], dtype=torch.float64, device=dev) for k in ("shared", "per_pixel")}
    blocks = {"shared": shared, "per_pixel": perpix}
    stream = torch.cuda.current_stream().cuda_stream

    def launch(name):
        _lib.check(lib.nf_nh3_loglike(blocks[name].handle, Pd.data_ptr(), _lib.NF_F64, None, vpp, P.shape[0], ncomp,
                                      0, out[name].data_ptr(), stream), "nf_nh3_loglike")

    for name in blocks:            # warm-up
        launch(name)
    torch.cuda.synchronize()
    times = {k: [] for k in blocks}
    for _ in range(reps):
        for name in blocks:        # A/B alternated
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                launch(name)
            e1.record()
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1) / 1e3 / steps)
    identical = bool(torch.equal(out["shared"], out["per_pixel"]))
    res = {"vectors": int(P.shape[0]), "pixels": n_pix, "ncomp": ncomp, "n_chan": [1000, 1000], "steps": steps,
           "reps": reps, "lnL_bit_identical": identical}
    for name, t in times.items():
        res[f"{name}_evals_per_s_median"] = P.shape[0] / float(np.median(t))
        res[f"{name}_call_ms"] = [round(1e3 * x, 4) for x in t]
    res["per_pixel_over_shared"] = res["per_pixel_evals_per_s_median"] / res["shared_evals_per_s_median"]
    shared.close()
    perpix.close()
    return res


def axis(nu0, n, dv, v0):
    v = v0 + (np.arange(n) - 0.5 * (n - 1)) * dv
    return np.sort(nu0 * (1.0 - v / CKMS))


def catalogue(n_src, seed=1, noise=0.12):
    """Sources with distinct velocity centres and channel widths, 300-1100 channels per spectrum (the two spectra
    of a source usually of different lengths), and 1 or 2 true components."""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n_src):
        vsrc = rng.uniform(-1.5, 1.5)
        if i % 3 == 0:
            ncomp, truth = 2, np.array([vsrc - 1.3, vsrc + 1.3, 10, 15, 5, 6, 14.6, 14.9, 0.3, 0.5, 0, 0], float)
        else:
            ncomp, truth = 1, np.array([vsrc, rng.uniform(11, 16), rng.uniform(5, 7), rng.uniform(14.4, 14.8),
                                        rng.uniform(0.3, 0.6), 0.0])
        n = rng.integers(300, 1101, size=2)
        if i % 4 == 0:
            n[1] = n[0]
        spec = []
        for s in range(2):
            x = axis(orc.NU[s], int(n[s]), rng.uniform(0.08, 0.2), vsrc + rng.uniform(-3, 3))
            clean = orc.nh3_batch([x], [s + 1], truth[None], ncomp, want_pred=True)["pred"][0, 0]
            spec.append([x, clean + rng.normal(0, noise, x.size), noise, s + 1])
        out.append(spec)
    return out


def catalogue_rates(n_src, n_serial, nlive, tol):
    ut = nb.get_irdc_priors()
    t0 = time.perf_counter()
    cat = catalogue(n_src)
    t_gen = time.perf_counter() - t0
    res = {"sources": n_src, "nlive": nlive, "tol": tol, "synth_s": round(t_gen, 2),
           "unequal_length_sources": int(sum(len(s[0][0]) != len(s[1][0]) for s in cat))}
    fit_s = runners_s = 0.0
    for ncomp in (1, 2):
        t0 = time.perf_counter()
        runners = [nb.AmmoniaRunner.from_data(s, ut, ncomp=ncomp) for s in cat]
        t1 = time.perf_counter()
        out = nb.run_multinest_batch(runners, nlive=nlive, tol=tol, seed=ncomp)
        t2 = time.perf_counter()
        fit_s += t2 - t1
        runners_s += t1 - t0
        res[f"batch_ncomp{ncomp}"] = {"runners_s": round(t1 - t0, 2), "fit_s": round(t2 - t1, 2),
                                      "truncated": int(out["truncated"].sum()), "launches": int(out["launches"]),
                                      "mean_lnZ_minus_null": float(np.mean([r.run_lnZ - r.null_lnZ for r in runners]))}
        for r in runners:
            r._block.close()
    res["batch_spectra_per_s"] = n_src / fit_s
    res["batch_spectra_per_s_incl_runners"] = n_src / (fit_s + runners_s)     # the serial figure includes them
    t0 = time.perf_counter()
    for s in cat[:n_serial]:
        for ncomp in (1, 2):
            r = nb.AmmoniaRunner.from_data(s, ut, ncomp=ncomp)
            nb.run_multinest(r, None, nlive=nlive, tol=tol, seed=ncomp)
            r._block.close()
    t_serial = time.perf_counter() - t0
    res["serial_sources"] = n_serial
    res["serial_s"] = round(t_serial, 2)
    res["serial_spectra_per_s"] = n_serial / t_serial
    res["batch_over_serial"] = res["batch_spectra_per_s"] / res["serial_spectra_per_s"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--vectors", type=int, default=1 << 20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--sources", type=int, default=4096)
    ap.add_argument("--serial", type=int, default=16)
    ap.add_argument("--nlive", type=int, default=100)
    ap.add_argument("--tol", type=float, default=1.0)
    ap.add_argument("--skip-catalogue", action="store_true")
    ap.add_argument("--out", default=None, help="also write the JSON here")
    args = ap.parse_args()
    name, power = device_info()
    res = {"device": name, "power_limit": power, "likelihood": likelihood_ab(args.vectors, args.reps, args.steps)}
    if args.out:              # the likelihood figures stand on their own if the catalogue leg does not finish
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res) + "\n")
    if not args.skip_catalogue:
        res["catalogue"] = catalogue_rates(args.sources, args.serial, args.nlive, args.tol)
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
