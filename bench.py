#!/usr/bin/env python
"""bench.py — headline benchmark of the BISIP MCMC likelihood hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Metric (BASELINE.json): log-prob evals/sec = spectra x walkers x steps / time.
Workload: BASELINE config 5 — Debye polynomial decomposition (poly_deg 4, 64 taus) of synthetic
64-frequency spectra, 256 walkers x 2000 steps — with a FIXED per-GPU shard of 12,500 spectra
(weak scaling: N=8 is the full 100,000-spectra config).  One "step" = one full inversion of the
shard: on-device ensemble sampling, kept-chain write (discard 1000, thin 10), device percentile /
mean / std summary, and for N>1 the NCCL all-gather of the summaries.

`value`  : inputs (zn, zn_err, p0) already resident in HBM; timed with CUDA events, max over ranks.
`e2e`    : the same job through the public API (BatchInversion.fit_gathered) from pinned HOST buffers, with the
           host->device copies of the inputs, for N>1 the NCCL gather of the summaries, and the device->host read
           of the complete result inside the timed region.
`roofline`: ensemble_decomp kernel (the dominant launch): algorithmic flops (17,792 per eval,
           SURVEY.md §8d) / its CUDA-event duration, against the FP64 DMMA peak measured on this
           box by tools/peaks (MEASURED_PEAKS.json has no FP64 figure).
`variants`: the collapsed FP64 kernel (precision='fp64-collapsed') and the TF32 / 3xTF32 tcgen05 kernels on the same
           shard (kernel alone on a slice, and the whole shard end to end), next to the default FP64 DMMA numbers.
`configs` : BASELINE configs 2-4 on one GPU (N=1 only): Cole-Cole(2) on the bundled spectrum, Dias / Shin on 1,024 synthetic
           spectra, and the 256-tau decomposition on 10,000 spectra in FP64 DMMA / 3xTF32 / TF32 / collapsed FP64 — kernel
           alone, end to end, and a roofline fraction each.
`strong_scaling`: the fixed 100,000-spectra survey through ONE `bisip_b200.fit_sharded` call on the N ranks.
`cpu_baseline`: the reference's own Cython + NumPy log-probability (oracle/_ref) under the emcee
           restatement, on all host cores, on a bounded sample of the same spectra.  Where the reference package is not
           built, the C restatement oracle/bisip_oracle.c runs instead; `note` says which of the two was timed.
`--impl reference`: that CPU arm alone, as its own JSON line.
`--dump-outputs DIR`: after the timed steps, what the last timed step computed goes to DIR/<name>.npy (float64): the
           per-spectrum summaries and the kept chains of a fixed, seeded sample of spectra (see `dump_outputs`).  The
           inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# This script prints exactly ONE line to stdout, the JSON result (its own progress goes to stderr).  File descriptor 1
# itself is left alone: whatever the driver's instrumentation makes native libraries print there (NCCL's banner under
# NCCL_DEBUG, ...) stays visible to the driver, and no environment variable of the driver is rewritten.
def emit(line):
    sys.stdout.write(json.dumps(line) + "\n")
    sys.stdout.flush()

# ---- workload (BASELINE config 5 shard) ------------------------------------------------------
N_FREQ, N_TAU, POLY_DEG, WALKERS, NSTEPS = 64, 64, 4, 256, 2000
SPECTRA_PER_GPU = int(os.environ.get("BISIP_BENCH_SPECTRA", 12500))
DISCARD, THIN = 1000, 10
PCT = (2.5, 50, 97.5)
SEED = 0xB151B
FLOP_PER_EVAL = 2 * (POLY_DEG + 1) * N_TAU + 2 * N_TAU * 2 * N_FREQ + 6 * 2 * N_FREQ   # 17,792
WORKLOAD = (f"C5 shard: {SPECTRA_PER_GPU} synthetic {N_FREQ}-frequency spectra per GPU, Debye decomposition "
            f"poly_deg={POLY_DEG}, {N_TAU} taus, {WALKERS} walkers x {NSTEPS} steps (8 GPUs = the 100,000-spectra config)")


def env_int(name, default):
    return int(os.environ.get(name, default))


# ---- reference CPU arm ---------------------------------------------------------------------------
def _ref_worker(args):
    """One process = one synthetic spectrum through the UNMODIFIED reference fit()
    (models.py:84-119 -> emcee restatement -> _log_probability -> Cython Decomp_cyth)."""
    b, zn, zn_err, w, walkers, nsteps = args
    from oracle import refload
    bisip = refload.load()
    np.random.seed(1000 + b)
    m = bisip.PolynomialDecomposition(refload.data_file(), nwalkers=walkers, nsteps=nsteps, poly_deg=POLY_DEG)
    # inject the synthetic spectrum and the 64-tau grid through the reference's public attributes
    # (models.py:204-209 are plain attributes users may reassign)
    m._data.update(w=w, zn=zn, zn_err=zn_err, N=len(w))
    lo = np.floor(min(np.log10(1. / w)) - 1)
    hi = np.floor(max(np.log10(1. / w)) + 1)
    m.log_tau = np.linspace(lo, hi, N_TAU)
    m.log_taus = np.array([m.log_tau ** i for i in range(POLY_DEG + 1)])
    m.taus = 10 ** m.log_tau
    t0 = time.perf_counter()
    m.fit()
    dt = time.perf_counter() - t0
    return dt, m.get_param_mean(discard=nsteps // 2)


def _restatement_worker(args):
    """One process = one synthetic spectrum through the C restatement of the reference's log-probability and of
    emcee's stretch move (oracle/bisip_oracle.c): the same posterior, walkers and steps as `_ref_worker`."""
    b, zn, zn_err, w, walkers, nsteps = args
    from bisip_b200.batch import default_bounds, tau_grid
    from oracle import oracle
    _, taus, log_taus = tau_grid(w, N_TAU, POLY_DEG)
    _, bounds = default_bounds('decomp', POLY_DEG)
    prob = oracle.Problem('decomp', w, zn, zn_err, bounds, taus=taus, log_taus=log_taus, c_exp=1.0)
    p0 = np.random.default_rng(1000 + b).uniform(bounds[0], bounds[1], (walkers, bounds.shape[1]))
    t0 = time.perf_counter()
    prob.run(p0, nsteps, seed=SEED, spectrum=b)
    return time.perf_counter() - t0


def reference_impl():
    """(worker, description) of the CPU arm.  The reference package is used where oracle/build_ref.sh built it into
    oracle/_ref (that needs the reference's sources, which this repository does not hold); otherwise the repository's
    own C restatement of it runs, so that the CPU arm works from a plain checkout."""
    from oracle import refload
    if refload.available():
        return _ref_worker, "reference models.py + Cython (oracle/_ref) under oracle/emcee_restatement.py"
    return _restatement_worker, ("C restatement of the reference's log-probability and emcee's stretch move "
                                 "(oracle/bisip_oracle.c); the reference package (oracle/_ref) is not built")


def reference_sample(zn, zn_err, w, cores, walkers=WALKERS, nsteps=None, pool=None):
    """Bounded sample: `cores` spectra (one per process) x walkers x nsteps.  Returns evals/s."""
    import multiprocessing as mp
    nsteps = nsteps or env_int("BISIP_BENCH_REF_STEPS", 300)
    jobs = [(b, zn[b], zn_err[b], w, walkers, nsteps) for b in range(cores)]
    own = pool is None
    if own:
        pool = mp.get_context("fork").Pool(cores)
    t0 = time.perf_counter()
    pool.map(reference_impl()[0], jobs)
    wall = time.perf_counter() - t0
    if own:
        pool.close()
    evals = cores * walkers * nsteps
    return evals / wall, wall, f"{cores} spectra x {walkers} walkers x {nsteps} steps, one process per core"


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def synthetic_cpu(n):
    """The benchmark spectra b in [0, n) built with the oracle forward (no GPU): used by the
    reference arm, which must not touch the product path."""
    from bisip_b200 import synthetic
    from bisip_b200.batch import tau_grid
    from oracle import oracle
    _, w = synthetic.frequencies(N_FREQ)
    _, taus, log_taus = tau_grid(w, N_TAU, POLY_DEG)

    def fwd(theta, ww):
        prob = oracle.Problem('decomp', ww, np.zeros((2, len(ww))), np.ones((2, len(ww))),
                              np.zeros((2, theta.shape[1])), taus=taus, log_taus=log_taus, c_exp=1.0)
        return prob.forward(theta)
    return synthetic.make('decomp', 0, n, fwd, N=N_FREQ, poly_deg=POLY_DEG, n_tau=N_TAU)


def run_reference(args):
    rank = env_int("RANK", 0)
    if rank != 0:
        return
    cores = host_cores()
    syn = synthetic_cpu(cores)
    import multiprocessing as mp
    pool = mp.get_context("fork").Pool(cores)
    for _ in range(args.warmup):
        reference_sample(syn['zn'], syn['zn_err'], syn['w'], cores, nsteps=2, pool=pool)
    rates, walls, sample = [], [], ""
    for _ in range(args.steps):
        r, wall, sample = reference_sample(syn['zn'], syn['zn_err'], syn['w'], cores, pool=pool)
        rates.append(r)
        walls.append(wall)
    pool.close()
    val = float(np.mean(rates))
    kind = "reference"
    emit(({
        "impl": "reference", "metric": "log-prob evals/sec", "value": val, "unit": "evals/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean(walls)),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample_per_step": sample},
        "cpu_baseline": {"value": val, "unit": "evals/s", "cores": cores, "kind": kind, "sample": sample,
                         "note": reference_impl()[1]},
        "e2e": {"value": val, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ---- GPU arm -----------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([c.strip() for c in out.strip().split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace('.', '').isdigit()]
        reasons = []
        for name, col in (("hw_slowdown", 4), ("hw_thermal_slowdown", 5), ("sw_thermal_slowdown", 6), ("sw_power_cap", 7)):
            if any(len(r) >= 8 and r[col] == "Active" for r in self.rows):
                reasons.append(name)
        busy = [v for v in sm if v > 0.5 * max(sm)] if sm else []
        return {"sm_mhz": float(np.median(busy)) if busy else None,
                "sm_max_mhz": float(self.rows[0][2]) if self.rows and len(self.rows[0]) >= 8 else None,
                "reasons": reasons, "samples": len(self.rows)}


def dmma_peak():
    """FP64 tensor (DMMA) peak of this GPU, measured now by tools/peaks (sustained 2 s loop)."""
    exe = os.path.join(ROOT, "tools", "peaks")
    try:
        out = subprocess.run([exe, "--sustain", "2"], capture_output=True, text=True, timeout=120).stdout
        j = json.loads(out.strip().splitlines()[-1])
        return j["dmma_tflops_sustained"], j["dmma_tflops_burst"], "measured live: tools/peaks --sustain 2 (mma.sync m16n8k16 f64)"
    except Exception as e:          # nominal: 148 SMs x 64 DFMA/clk x 2 x 1.965 GHz
        return 37.2, 37.2, f"nominal (tools/peaks failed: {e})"


def kernel_sources_sha():
    """Hash of the sources that define the dominant kernel (ensemble_wp_kernel<DecompMmaWarpEvaluator>): the committed ncu
    DRAM figure is only quoted while they are unchanged."""
    import hashlib
    h = hashlib.sha256()
    for f in ("sampler_wp.cuh", "sampler.cuh", "decomp_eval.cuh", "common.cuh"):
        with open(os.path.join(ROOT, "bisip_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def dfma_peak():
    """FP64 vector (DFMA) peak of this GPU from tools/peaks (register-resident FMA loop)."""
    exe = os.path.join(ROOT, "tools", "peaks")
    try:
        out = subprocess.run([exe], capture_output=True, text=True, timeout=180).stdout
        return float(json.loads(out.strip().splitlines()[-1])["dfma_tflops"]), "measured live: tools/peaks (DFMA loop)"
    except Exception as e:
        return 36.8, f"round-1 measurement (tools/peaks failed: {e})"


def ncu_flops_per_eval():
    """Executed FP64 flops per log-prob evaluation of the vector-model kernels, counted once by ncu
    (smsp__sass_thread_inst_executed_op_d{fma,mul,add}_pred_on) and committed in profiles/ncu_summary.json."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "ncu_summary.json"))).get("fp64_flop_per_eval", {})
    except Exception:
        return {}


def measure_config(torch, engine, inv, p0_h, discard, thin, reps=2, warm=True):
    """One BASELINE config on this GPU: the ensemble kernel alone (device-resident inputs, CUDA events) and the whole
    job end to end through BatchInversion.fit (pinned host inputs in, host summaries out)."""
    dev = inv.device
    B, W, T = inv.n_spectra, inv.nwalkers, inv.nsteps
    spec = inv._spec()
    w_d = _dev(torch, inv.w, dev)
    y_d, ye_d, p0_d = inv._zn.to(dev), inv._zn_err.to(dev), p0_h.to(dev)
    bounds_d = _dev(torch, inv.param_bounds, dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best, res = 1e30, None
    for rep in range(reps + (1 if warm else 0)):
        c = p0_d.clone()
        del res
        e0.record()
        res = engine.ensemble_run(spec, c, w_d, y_d, ye_d, bounds_d, nsteps=T, seed=inv.seed, spectrum0=0,
                                  discard=discard, thin=thin, store_chain=True, store_logp=False)
        e1.record()
        torch.cuda.synchronize()
        if rep or not warm:
            best = min(best, e0.elapsed_time(e1))
    acc = float(res['accepted'].double().mean().item() / T)
    nan = int((res['flags'] != 0).sum().item())
    del res, c
    torch.cuda.empty_cache()
    e2e = 1e30
    for rep in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = inv.fit(p0=p0_h, discard=discard, thin=thin, percentiles=PCT)
        torch.cuda.synchronize()
        e2e = min(e2e, time.perf_counter() - t0)
    evals = float(B) * W * T
    out = {"spectra": B, "walkers": W, "nsteps": T, "kernel_ms": best, "evals_per_s": evals * (T + 1) / T / (best * 1e-3),
           "e2e_ms": 1e3 * e2e, "e2e_evals_per_s": evals / e2e, "e2e_spectra_per_s": B / e2e,
           "acceptance_fraction": acc, "nan_flags": nan,
           "h2d_bytes": int(inv._zn.numel() * 16 + p0_h.numel() * 8), "d2h_bytes": int(sum(v.nbytes for v in r.values()))}
    del r
    torch.cuda.empty_cache()
    return out


def _dev(torch, a, dev):
    return torch.from_numpy(np.ascontiguousarray(np.asarray(a, dtype=np.float64))).to(dev)


def vec_roofline(fl, name, evals_per_s, peak_dfma):
    """FP64-pipe roofline of a vector-model kernel from the executed FP64 instruction counts ncu measured once
    (profiles/ncu_summary.json: fp64_flop_per_eval).  `frac` = executed FP64 thread instructions per second over the
    pipe's instruction rate (peak DFMA flops / 2: a DMUL or DADD occupies the same slot as a DFMA) — the utilisation
    figure north_star's 50 % bar is about; `achieved` (flops, FMA = 2) is given next to it."""
    d = fl.get("detail", {}).get(name)
    if not d:
        return None
    inst_rate = evals_per_s * d["fp64_inst_per_eval"]
    return {"bound": "fp64 pipe", "fp64_flop_per_eval": d["flop_per_eval"], "fp64_inst_per_eval": d["fp64_inst_per_eval"],
            "achieved": evals_per_s * d["flop_per_eval"] / 1e12, "peak": peak_dfma, "unit": "TFLOP/s",
            "frac": inst_rate / (peak_dfma * 1e12 / 2.0), "frac_in_flops": evals_per_s * d["flop_per_eval"] / 1e12 / peak_dfma,
            "ncu_fp64_pipe_pct_of_active_cycles": d.get("fp64_pipe_pct_active"), "flop_source": fl.get("source"),
            "peak_note": "nominal DFMA peak; a DFMA reading three distinct register pairs runs at 2/3 of it on B200, the model loops "
                         "alone (no sampler) reach 62-78 % of it (profiles/r02c_vec_analysis.md)"}


def run_other_configs(torch, engine, synthetic, BatchInversion, _lib, dev, peak_dmma, peak_dfma):
    """BASELINE configs 2-4 on one GPU (config 1 is the reference's own CPU-sized case; config 5 is the headline)."""
    out = {}
    fl = ncu_flops_per_eval()
    f, w = synthetic.frequencies(N_FREQ)

    def fwd_for(model, **kw):
        probe = BatchInversion(model, w, np.zeros((1, 2, N_FREQ)), np.ones((1, 2, N_FREQ)), device=dev, **kw)
        return lambda th, ww: engine.forward(probe._spec(), _dev(torch, th[:, None, :], dev), _dev(torch, ww, dev))[:, 0].cpu().numpy()

    def pin(a):
        return torch.from_numpy(np.ascontiguousarray(a)).pin_memory()

    # ---- C3: Dias2000 and Shin2015, 1,024 synthetic 64-frequency spectra, 128 walkers x 2000 steps
    for model in ("dias", "shin"):
        syn = synthetic.make(model, 0, 1024, fwd_for(model), N=N_FREQ)
        inv = BatchInversion(model, w, pin(syn['zn']), pin(syn['zn_err']), nwalkers=128, nsteps=2000, seed=SEED, device=dev)
        r = measure_config(torch, engine, inv, pin(inv.draw_p0(0, 1024)), DISCARD, THIN)
        r["roofline"] = vec_roofline(fl, f"ensemble_{model}", r["evals_per_s"], peak_dfma)
        out[f"C3_{model}"] = dict(workload=f"{model}: 1,024 synthetic {N_FREQ}-frequency spectra, 128 walkers x 2000 steps", **r)
    # ---- C2: ColeCole n_modes=2 on the bundled example spectrum, 64 walkers x 2000 steps, batched x 1,024 streams
    from bisip_b200.data import example_tables
    from bisip_b200.utils import prepare_data
    d = prepare_data(example_tables()['SIP-K389175'], 'mrad')
    inv = BatchInversion('colecole', d['w'], pin(np.repeat(d['zn'][None], 1024, 0)), pin(np.repeat(d['zn_err'][None], 1024, 0)),
                         nwalkers=64, nsteps=2000, n_modes=2, seed=SEED, device=dev)
    r = measure_config(torch, engine, inv, pin(inv.draw_p0(0, 1024)), DISCARD, THIN)
    r["roofline"] = vec_roofline(fl, "ensemble_colecole2_n20", r["evals_per_s"], peak_dfma)
    out["C2_colecole2"] = dict(workload="ColeCole n_modes=2, bundled SIP-K389175 (20 frequencies), 64 walkers x 2000 steps, "
                                        "1,024 independent streams of the same spectrum in one launch", **r)
    # ---- C4: decomposition with 256 taus, 10,000 synthetic spectra, 256 walkers x 2000 steps: FP64 DMMA vs TF32 / 3xTF32 / collapsed
    n4 = env_int("BISIP_BENCH_C4_SPECTRA", 10000)
    syn = synthetic.make('decomp', 0, n4, fwd_for('decomp', poly_deg=POLY_DEG, n_tau=256), N=N_FREQ, poly_deg=POLY_DEG, n_tau=256)
    zn_h, ze_h = pin(syn['zn']), pin(syn['zn_err'])
    flop4 = 2 * (POLY_DEG + 1) * 256 + 2 * 256 * 2 * N_FREQ + 6 * 2 * N_FREQ          # 68,864
    c4, p0_h, ref_pct = {}, None, None
    th_chk = None
    for prec in ("fp64", "3xtf32", "tf32", "fp64-collapsed"):
        inv = BatchInversion('decomp', w, zn_h, ze_h, nwalkers=WALKERS, nsteps=NSTEPS, poly_deg=POLY_DEG, n_tau=256,
                             precision=prec, seed=SEED, device=dev)
        if p0_h is None:
            p0_h = pin(inv.draw_p0(0, n4))
        r = measure_config(torch, engine, inv, p0_h, DISCARD, THIN, reps=1, warm=(prec != "fp64"))
        r["kernel"] = engine.decomp_kernel_kind(inv._spec(), N_FREQ, WALKERS)
        if prec == "fp64":
            r["roofline"] = {"bound": "tensor", "algorithmic_flop_per_eval": flop4, "achieved": r["evals_per_s"] * flop4 / 1e12,
                             "peak": peak_dmma, "unit": "TFLOP/s", "frac": r["evals_per_s"] * flop4 / 1e12 / peak_dmma}
            ref_pct = inv.results['percentiles'].copy()
            ref_sd = inv.results['std'].copy()
            th_chk = _dev(torch, inv.results['percentiles'][:64, 1][:, None, :], dev)          # posterior medians of 64 spectra
            z_ref = engine.forward(inv._spec(), th_chk, _dev(torch, w, dev))
        else:
            z = engine.forward(inv._spec(), th_chk, _dev(torch, w, dev))
            r["forward_rel_error_vs_fp64"] = float(((z - z_ref).abs().amax((2, 3)) / z_ref.abs().amax((2, 3))).max().item())
            r["max_median_shift_in_posterior_sd"] = float(np.max(np.abs(inv.results['percentiles'][:, 1] - ref_pct[:, 1]) / ref_sd))
            r["speedup_vs_fp64"] = r["evals_per_s"] / c4["fp64"]["evals_per_s"]
        c4[prec] = r
        del inv
        torch.cuda.empty_cache()
    out["C4_decomp_256taus"] = {"workload": f"Debye decomposition poly_deg={POLY_DEG}, 256 taus, {n4} synthetic {N_FREQ}-frequency spectra, "
                                            f"{WALKERS} walkers x {NSTEPS} steps; kernel alone + end to end per precision", **c4}
    return out


DUMP_MAX_SPECTRA = 100_000     # per-spectrum summaries: 32 float64 each, 25.6 MB at most
DUMP_CHAINS = 16               # kept chains of 16 spectra: 100 x 256 x 6 float64 each, 19.7 MB at the default shape
DUMP_LIMIT = 64 << 20


def dump_outputs(torch, path, out, res):
    """Write what the last timed step computed, as float64 .npy files in `path`: the per-spectrum summaries of
    `step_resident` (percentiles, mean, std, acceptance_fraction) and, for DUMP_CHAINS spectra, the kept chain and the
    per-walker accepted counts of `engine.ensemble_run`.  Row sets are fixed by SEED (`spectra`, `chain_spectra` hold
    the indices), so that runs with the same arguments write the same rows."""
    rng = np.random.default_rng(SEED)
    n = out['mean'].shape[0]
    rows = np.arange(n) if n <= DUMP_MAX_SPECTRA else np.sort(rng.choice(n, DUMP_MAX_SPECTRA, replace=False))
    crow = np.sort(rng.choice(res['chain'].shape[0], min(DUMP_CHAINS, res['chain'].shape[0]), replace=False))
    arrays = {k: v[torch.from_numpy(rows).to(v.device)] for k, v in out.items()}
    arrays["spectra"] = rows
    sel = torch.from_numpy(crow).to(res['chain'].device)
    arrays["chain"] = res['chain'][sel]
    arrays["accepted"] = res['accepted'][sel]
    arrays["chain_spectra"] = crow
    arrays = {k: np.ascontiguousarray((v.cpu().numpy() if torch.is_tensor(v) else v), dtype=np.float64)
              for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)
    print(f"bench: wrote {len(arrays)} arrays ({total / 2**20:.1f} MiB) to {path}", file=sys.stderr)


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from bisip_b200 import _lib, engine, synthetic
    from bisip_b200.batch import BatchInversion, fit_sharded, gather_packed

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = SPECTRA_PER_GPU
    b0 = rank * B                                      # weak scaling: rank r owns spectra [rB, (r+1)B)
    nk = engine.n_keep(NSTEPS, DISCARD, THIN)

    peak_sust, peak_burst, peak_src = dmma_peak() if rank == 0 else (None, None, None)

    # ---- synthetic shard: truth through the CUDA forward, noise / normalisation on the host -------
    probe = BatchInversion('decomp', synthetic.frequencies(N_FREQ)[1], np.zeros((1, 2, N_FREQ)), np.ones((1, 2, N_FREQ)),
                           poly_deg=POLY_DEG, n_tau=N_TAU, device=dev)

    def cuda_forward(theta, w):
        th = _lib.dev_f64(theta[:, None, :], dev)
        return engine.forward(probe._spec(), th, _lib.dev_f64(w, dev))[:, 0].cpu().numpy()
    syn = synthetic.make('decomp', b0, b0 + B, cuda_forward, N=N_FREQ, poly_deg=POLY_DEG, n_tau=N_TAU)
    zn_h = torch.from_numpy(syn['zn']).pin_memory()
    ze_h = torch.from_numpy(syn['zn_err']).pin_memory()
    inv = BatchInversion('decomp', syn['w'], zn_h, ze_h, nwalkers=WALKERS, nsteps=NSTEPS, poly_deg=POLY_DEG,
                         n_tau=N_TAU, seed=SEED, spectrum_offset=b0, device=dev)
    p0_h = torch.from_numpy(inv.draw_p0(0, B)).pin_memory()

    # ---- device-resident arm ---------------------------------------------------------------------
    spec = inv._spec()
    w_d = _lib.dev_f64(syn['w'], dev)
    y_d, ye_d, p0_d = zn_h.to(dev), ze_h.to(dev), p0_h.to(dev)
    bounds_d = _lib.dev_f64(inv.param_bounds, dev)
    coords = torch.empty_like(p0_d)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
    kern_ms, stats_ms = [], []

    def step_resident(timed):
        coords.copy_(p0_d)
        ev[0].record()
        res = engine.ensemble_run(spec, coords, w_d, y_d, ye_d, bounds_d, nsteps=NSTEPS, seed=SEED, spectrum0=b0,
                                  discard=DISCARD, thin=THIN, store_chain=True, store_logp=False)
        ev[1].record()
        st = engine.column_stats(res['chain'].reshape(B, nk * WALKERS, inv.ndim), p=list(PCT), want_mean=True, want_std=True)
        ev[2].record()
        out = {'percentiles': st['pct'], 'mean': st['mean'], 'std': st['std'],
               'acceptance_fraction': res['accepted'].to(torch.float64).mean(1) / NSTEPS}
        if world > 1:
            out = gather_packed(out, B * world, rank, world)
        if timed:
            torch.cuda.synchronize()
            kern_ms.append(ev[0].elapsed_time(ev[1]))
            stats_ms.append(ev[1].elapsed_time(ev[2]))
        return out, res

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        out, res = step_resident(False)
        del res
    barrier()
    clocks = ClockSampler(local)
    clocks.start()
    launches0 = _lib.launch_count()
    t_ev0, t_ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_ev0.record()
    for _ in range(args.steps):
        res = None                  # the previous step's 15 GB chain is freed before the next one is allocated
        out, res = step_resident(True)
    t_ev1.record()
    barrier()
    launches = _lib.launch_count() - launches0
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(torch, args.dump_outputs, out, res)
    del res
    ms_total = t_ev0.elapsed_time(t_ev1)
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    evals_step = B * world * WALKERS * NSTEPS
    value = evals_step / (ms_step * 1e-3)
    acc = float(out['acceptance_fraction'].mean().item())
    flags_bad = 0
    del out
    torch.cuda.empty_cache()

    # ---- end-to-end arm: public API, pinned host inputs in, COMPLETE host result out on every rank (for N > 1 the NCCL
    #      gather of the summaries is inside the timed region: BatchInversion.fit_gathered = fit + gather_packed) ---------
    h2d = zn_h.numel() * 8 + ze_h.numel() * 8 + p0_h.numel() * 8 + syn['w'].nbytes
    e2e_ms = []
    d2h = 0
    for i in range(args.steps):
        barrier()
        t0 = time.perf_counter()
        r = inv.fit_gathered(B * world, p0=p0_h, discard=DISCARD, thin=THIN, percentiles=PCT)
        torch.cuda.synchronize()
        e2e_ms.append(1e3 * (time.perf_counter() - t0))
        d2h = sum(v.nbytes for v in r.values())
        flags_bad += int((r['flags'] != 0).sum())
        assert r['mean'].shape[0] == B * world
    te = torch.tensor([float(np.mean(e2e_ms))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = evals_step / (float(te.item()) * 1e-3)
    r_local = {k: v[b0:b0 + B] for k, v in r.items()}

    # ---- the collapsed FP64 path end to end on EVERY rank (weak scaling of the fast path: at N=8 this is the whole
    #      100,000-spectra survey, summaries gathered), max over ranks like `e2e`
    alt = BatchInversion('decomp', syn['w'], zn_h, ze_h, nwalkers=WALKERS, nsteps=NSTEPS, poly_deg=POLY_DEG,
                         n_tau=N_TAU, seed=SEED, spectrum_offset=b0, device=dev, precision='fp64-collapsed')
    col_best = 1e30
    for rep in range(3):
        barrier()
        t0 = time.perf_counter()
        r_col = alt.fit_gathered(B * world, p0=p0_h, discard=DISCARD, thin=THIN, percentiles=PCT)
        torch.cuda.synchronize()
        tc = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tc, op=dist.ReduceOp.MAX)
        col_best = min(col_best, float(tc.item()))
    r_col = {k: v[b0:b0 + B] for k, v in r_col.items()}
    del alt

    # ---- strong scaling: the FIXED 100,000-spectra survey through ONE sharded product call (fit_sharded: full-size host
    #      arrays in on every rank, complete result out on every rank), default FP64 DMMA path.  The survey is this rank's
    #      12,500 synthetic spectra tiled to 100,000 (each copy samples its own Philox stream); fit_sharded reads only the
    #      rank's block of it.
    strong = None
    n_strong = env_int("BISIP_BENCH_STRONG_SPECTRA", 100000)
    if n_strong > 0:
        reps = -(-n_strong // B)                        # the survey = this rank's shard data tiled (Philox streams differ per index)
        zn_s = zn_h.repeat(reps, 1, 1)[:n_strong]
        ze_s = ze_h.repeat(reps, 1, 1)[:n_strong]
        prec_s = os.environ.get("BISIP_BENCH_STRONG_PRECISION", "fp64")
        barrier()
        t0 = time.perf_counter()
        rs = fit_sharded('decomp', syn['w'], zn_s, ze_s, discard=DISCARD, thin=THIN, percentiles=PCT, nwalkers=WALKERS,
                         nsteps=NSTEPS, poly_deg=POLY_DEG, n_tau=N_TAU, seed=SEED, device=dev, precision=prec_s)
        torch.cuda.synchronize()
        ts = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        strong = {"spectra": n_strong, "n_gpus": world, "precision": prec_s, "seconds": float(ts.item()),
                  "evals_per_s": n_strong * WALKERS * NSTEPS / float(ts.item()), "spectra_per_s": n_strong / float(ts.item()),
                  "api": "bisip_b200.fit_sharded (full host arrays in, shard_range per rank, p0 drawn per spectrum, NCCL gather "
                         "of the summaries, complete host result on every rank); scaling = strong",
                  "complete_on_this_rank": bool(rs['mean'].shape[0] == n_strong), "nan_flags": int((rs['flags'] != 0).sum())}
        del rs, zn_s, ze_s
        torch.cuda.empty_cache()

    variants = {}
    if rank == 0:
        for prec in ("fp64-collapsed", "3xtf32", "tf32"):
            nv = min(B, 2368 if prec == "fp64-collapsed" else 592)       # one full wave of resident CTAs
            alt = BatchInversion('decomp', syn['w'], zn_h[:nv], ze_h[:nv], nwalkers=WALKERS, nsteps=NSTEPS, poly_deg=POLY_DEG,
                                 n_tau=N_TAU, seed=SEED, spectrum_offset=b0, device=dev, precision=prec)
            aspec = alt._spec()
            best = 1e30
            for rep in range(3):
                c = p0_d[:nv].clone()
                ev[3].record()
                r_alt = engine.ensemble_run(aspec, c, w_d, y_d[:nv], ye_d[:nv], bounds_d, nsteps=500, seed=SEED, spectrum0=b0,
                                            discard=250, thin=10, store_chain=True, store_logp=False)
                ev[4].record()
                torch.cuda.synchronize()
                if rep:
                    best = min(best, ev[3].elapsed_time(ev[4]))
            variants[prec] = {"kernel": engine.decomp_kernel_kind(aspec, N_FREQ, WALKERS), "evals_per_s": nv * WALKERS * 501 / (best * 1e-3),
                              "spectra": nv, "steps": 500, "kernel_ms": best,
                              "acceptance_fraction": float(r_alt['accepted'].double().mean().item() / 500),
                              "nan_flags": int((r_alt['flags'] != 0).sum().item())}
            del r_alt
        # the whole shard end to end through the public API (pinned host inputs, host summaries), like `e2e`
        alt = BatchInversion('decomp', syn['w'], zn_h, ze_h, nwalkers=WALKERS, nsteps=NSTEPS, poly_deg=POLY_DEG,
                             n_tau=N_TAU, seed=SEED, spectrum_offset=b0, device=dev, precision='3xtf32')
        best = 1e30
        for rep in range(2):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r_alt = alt.fit(p0=p0_h, discard=DISCARD, thin=THIN, percentiles=PCT)
            torch.cuda.synchronize()
            best = min(best, time.perf_counter() - t0)
        variants['3xtf32'].update({"e2e_evals_per_s": B * WALKERS * NSTEPS / best, "e2e_spectra_per_s": B / best,
                                   "e2e_ms_per_step": 1e3 * best, "e2e_nan_flags": int((r_alt['flags'] != 0).sum()),
                                   "e2e_gpus": 1})
        del r_alt, alt
        # FP64 to rounding: the collapsed sampler takes the same decisions as the two-stage DMMA path (`r_local` = last e2e
        # result of this rank) unless a ~1e-13 log-prob rounding difference flips one of the shard's 1.3e10 accept tests
        # (expected: a fraction of one spectrum per shard); from there on that spectrum's chain is a different, equally
        # valid draw
        same = np.all(r_col['percentiles'] == r_local['percentiles'], axis=(1, 2))
        shift = np.abs(r_col['percentiles'][:, 1] - r_local['percentiles'][:, 1]) / r_local['std']
        variants['fp64-collapsed'].update({
            "e2e_evals_per_s": B * world * WALKERS * NSTEPS / col_best, "e2e_spectra_per_s": B * world / col_best,
            "e2e_ms_per_step": 1e3 * col_best, "e2e_nan_flags": int((r_col['flags'] != 0).sum()), "e2e_gpus": world,
            "e2e_spectra": B * world, "spectra_with_percentiles_identical_to_fp64": int(same.sum()),
            "spectra_compared": B, "max_median_shift_in_posterior_sd": float(shift.max()),
            "algorithmic_flop_per_eval": 2 * 2 * N_FREQ * (POLY_DEG + 1 + 2)})
    del y_d, ye_d, p0_d, coords
    torch.cuda.empty_cache()
    if rank == 0:
        k_ms = float(np.mean(kern_ms))
        flops_launch = FLOP_PER_EVAL * float(B) * WALKERS * (NSTEPS + 1)       # +1: log-prob of p0
        achieved = flops_launch / (k_ms * 1e-3) / 1e12
        traffic = traffic_src = None
        summ = os.path.join(ROOT, "profiles", "ncu_summary.json")
        if os.path.exists(summ) and B == 12500:          # the committed ncu figure is for the default shard size
            try:
                e = json.load(open(summ)).get("ensemble_decomp", {})
                if e.get("kernel_sources_sha") == kernel_sources_sha():
                    traffic, traffic_src = e.get("dram_bytes_per_launch_at_bench_size"), e.get("dram_bytes_source")
                else:
                    traffic_src = ("not quoted: the kernel sources changed since the committed ncu capture "
                                   f"({e.get('kernel_sources_sha')} -> {kernel_sources_sha()}); re-run tools/ncu_summary.py")
            except Exception:
                traffic = None
        # CPU baseline (bounded sample of the same spectra, all host cores) and BASELINE configs 2-4: N=1 only
        cores = host_cores()
        other = None
        if world == 1:
            cpu_v, cpu_wall, cpu_sample = reference_sample(syn['zn'], syn['zn_err'], syn['w'], min(cores, B))
            cpu_baseline = {"value": cpu_v, "unit": "evals/s", "cores": min(cores, B), "kind": "reference", "sample": cpu_sample,
                            "wall_s": cpu_wall, "evals_per_s_per_core": cpu_v / min(cores, B),
                            "extrapolated_days_for_full_config_on_these_cores": 1e5 * WALKERS * NSTEPS / cpu_v / 86400.0,
                            "note": reference_impl()[1]}
            if env_int("BISIP_BENCH_CONFIGS", 1):
                peak_dfma, _ = dfma_peak()
                other = run_other_configs(torch, engine, synthetic, BatchInversion, _lib, dev, peak_sust, peak_dfma)
                other["fp64_vector_peak_tflops"] = peak_dfma
        else:       # the host-core baseline is a property of the box, not of N: timed at N=1 only (the other ranks would wait)
            cpu_baseline = {"value": None, "unit": "evals/s", "cores": cores, "kind": "reference",
                            "sample": "not run at N>1: see the N=1 line"}
        line = {
            "metric": "log-prob evals/sec", "value": value, "unit": "evals/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "spectra_per_gpu": B, "walkers": WALKERS, "nsteps": NSTEPS, "n_freq": N_FREQ,
                       "n_tau": N_TAU, "poly_deg": POLY_DEG, "discard": DISCARD, "thin": THIN, "percentiles": list(PCT),
                       "l2": "per-step inputs (p0 154 MB) and outputs (kept chain 15 GB) exceed the 126 MB L2; no flush needed",
                       "parallelism": f"{world} x independent shards, one NCCL all-gather of the packed summaries"},
            "spectra_per_s": B * world / (ms_step * 1e-3),
            "e2e": {"value": e2e_value, "unit": "evals/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": float(te.item()), "spectra_per_s": B * world / (float(te.item()) * 1e-3),
                    "api": "bisip_b200.BatchInversion.fit_gathered (pinned host zn/zn_err/p0 of the shard in; for N>1 the NCCL "
                           "gather of the summaries is inside the timed region; the complete host result on every rank)"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "kernel": "ensemble_wp_kernel<DecompMmaWarpEvaluator<4>, 2, 256> (bisip_ensemble_run)",
                         "achieved": achieved, "peak": peak_sust, "unit": "TFLOP/s", "frac": achieved / peak_sust,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "algorithmic_bytes": float(B) * (nk * WALKERS * inv.ndim * 8 + 2 * WALKERS * inv.ndim * 8
                                                          + WALKERS * 12 + 4 * N_FREQ * 8 + 4),
                         "peak_source": peak_src, "peak_burst": peak_burst,
                         "kernel_ms": k_ms, "kernel_share_of_step": k_ms / ms_step,
                         "stats_kernel_ms": float(np.mean(stats_ms)),
                         "stats_kernel_GBps": float(B) * nk * WALKERS * inv.ndim * 8 / (float(np.mean(stats_ms)) * 1e-3) / 1e9,
                         "algorithmic_flop_per_eval": FLOP_PER_EVAL},
            "cpu_baseline": cpu_baseline,
            "clocks": clk, "acceptance_fraction": acc, "nan_flags": flags_bad,
            "strong_scaling": strong,
            "configs": other,
            "variants": {"note": "other decomposition kernels on the same shard: evals_per_s = ensemble kernel alone on a slice (CUDA "
                                 "events), e2e_* = the whole shard through BatchInversion.fit like `e2e`.  fp64-collapsed is FP64 "
                                 "(same 1e-12 parity, z = (L K) a); tf32 / 3xtf32 tolerances in profiles/r01f_tf32_study.md.  "
                                 "value / e2e / roofline above are the default two-stage FP64 DMMA path",
                         "fp64_evals_per_s_kernel": evals_step / world * (NSTEPS + 1) / NSTEPS / (k_ms * 1e-3), **variants},
        }
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="graft", choices=["graft", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's results to DIR/<name>.npy (GPU arm)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # convenience: `python bench.py --gpus N` re-launches itself one rank per GPU
        os.execvp(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                                   f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
                                   "--master-port", str(29500 + os.getpid() % 1000), os.path.abspath(__file__)] + sys.argv[1:])
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
