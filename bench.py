#!/usr/bin/env python
"""bench.py -- chain-iterations/s of the fused Hill log-target + adaptive-Metropolis path on B200.

    python bench.py --gpus N --steps K --warmup W            (under torchrun for N > 1)
    python bench.py --impl reference ...                      (CPU arm: the reference's algorithm on host cores)

Headline workload (BASELINE.json configs[1]): every Crumb (drug, channel) pair (210) x single-level models {1, 2} x 64
chains = 26 880 chains per GPU, PyHillFit-variant adaptive Metropolis (python/PyHillFit.py:828-856), thinning 5.
One step = `--iters-per-step` iterations of every chain (two kernel launches, one per model, on two streams; inside
the timed run the two streams are joined with the main stream only before the first and after the last step),
thinned samples written to HBM.  N > 1: every rank runs the same workload with disjoint Philox chain ids (weak
scaling, no collective on the data path); the value is chains x iterations over all ranks / max-over-ranks time.

The JSON line carries: value (device-timed, inputs resident), e2e (through phf_am_single_run_host with pinned
host buffers, H2D of state+data and D2H of samples+state inside the timed region), roofline (FP64: algorithmic
flops W per chain-iteration from SURVEY.md section 8d / the live DFMA probe), cpu_baseline (the oracle's numpy/scipy
restatement of the reference loop on all host cores, bounded sample, with ESS/s by the same estimator), clocks,
gpu_launches, ess_per_s, and `other_configs`:
  * at every N, the north-star's STRONG-scaling workloads, sharded over the N ranks (python/PyHillTemp.py:151-161,
    python/compute_bayes_factors.py:77-100): the reference's whole thermodynamic-integration sweep (41 temperatures x
    210 pairs x 2 models x 500 000 iterations), BASELINE config 4 (64 temperatures) -- NCCL all-gather of the per-chain
    mean log-likelihoods and the trapezium rule INSIDE the timed region -- and BASELINE config 5 (10^6 synthetic
    datasets x 4 chains); each with its own FP64 roofline entry;
  * at N = 1 also BASELINE config 3 (hierarchical).
"""
import argparse
import hashlib
import json
import math
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

# stdout carries exactly ONE line, the JSON result: everything else that writes to file descriptor 1 (NCCL prints its
# version there from C) is sent to stderr for the life of the process.
_RESULT_FD = os.dup(1)
os.dup2(2, 1)
sys.stdout = os.fdopen(os.dup(2), "w", buffering=1)


def emit(line):
    os.write(_RESULT_FD, (json.dumps(line) + "\n").encode())


METRIC = "chain-iterations/sec (all chains, device-timed)"
UNIT = "chain-iterations/s"
WORKLOAD = "Crumb: 210 drug-channel pairs x single-level models {1,2} x %d chains, PyHillFit AM, thinning %d"
DATA = ("real: the Crumb et al. dose-response table the reference ships (data/crumb_data.csv, packaged as "
        "tests/golden/datasets.npz); chains start at the least-squares fit (chains 1..63 of a pair jittered by 2 %); "
        "config 5 in other_configs is synthetic (pyhillfit_b200/synthetic.py)")


# ----------------------------------------------------------------------------------------------
# algorithmic FP64 work per chain-iteration (SURVEY.md section 8d cost table; FMA = 2 flops)
# ----------------------------------------------------------------------------------------------
def flops_per_iteration(model, groups, prior_only=False):
    d = 2 if model == 1 else 3
    D = len(groups)
    d_other = int(np.count_nonzero(groups["n_other"] > 0))
    d_cens = int(np.count_nonzero(groups["n0"] > 0) + np.count_nonzero(groups["n100"] > 0))
    per_dose = 53 if model == 2 else 52
    lik = 0 if prior_only else 40 + 58 + D * per_dose + d_other * 5 + d_cens * 133 + 6   # t == 0: doseresponse.py:204-205
    prior = 56
    proposal = math.ceil(d / 2) * 118 + d * (d + 1) + d + 40
    accept = 53
    adapt = 3 * d * d + 16 * d + 4 * d + 3
    return lik + prior + proposal + accept + adapt


def hier_flops_per_iteration(n_expts, n_points):
    """SURVEY.md section 8d, hierarchical: per point Hill curve + 2 erfc + log = 271, per experiment ~330 (logistic +
    log-logistic terms), 5 Gamma hyper-priors, proposal / accept / adapt as for the single-level loop at dimension d
    (6.1 kflops at Ne = 3, N = 12)."""
    d = 5 + 2 * n_expts
    return (271 * n_points + 330 * n_expts + 5 * 56 + math.ceil(d / 2) * 118 + d * (d + 1) + d + 40 + 53 +
            3 * d * d + 16 * d + 4 * d + 3)


def pack_flops(model, pack):
    return np.array([flops_per_iteration(model, pack.groups[b:b + n]) for b, n in
                     zip(pack.datasets["group_begin"], pack.datasets["n_groups"])], dtype=float)


# ----------------------------------------------------------------------------------------------
# workload
# ----------------------------------------------------------------------------------------------
def build_workload(chains_per_pair):
    from _data import Table
    from pyhillfit_b200.initial_fit import best_fit_batch
    from pyhillfit_b200.packing import SinglePack
    table = Table("crumb_data")
    pairs = table.pairs()
    data = [table.concat(d, c) for d, c in pairs]
    pack = SinglePack(data)
    rng = np.random.default_rng(25)
    out = {"data": data}
    for model in (1, 2):
        d = 2 if model == 1 else 3
        fits = best_fit_batch(model, data)[0]
        theta0 = np.repeat(fits, chains_per_pair, axis=0)
        jitter = 1.0 + 0.02 * rng.standard_normal(theta0.shape)
        jitter[::chains_per_pair] = 1.0  # chain 0 of every pair starts exactly at the least-squares fit
        theta0 = theta0 * jitter
        theta0[:, -1] = np.maximum(theta0[:, -1], 2e-3)
        if model == 2:
            theta0[:, 1] = np.clip(theta0[:, 1], 1e-6, 10.0)
        theta0[:, 0] = np.maximum(theta0[:, 0], -3.0)
        ids = np.repeat(np.arange(len(pairs), dtype=np.int32), chains_per_pair)
        w = pack_flops(model, pack)
        out[model] = dict(theta0=theta0, ids=ids, d=d, flops=float(np.repeat(w, chains_per_pair).mean()),
                          flops_per_dataset=w)
    return pack, out


DUMP_CHAINS = 256          # chains per model in a --dump-outputs sample
DUMP_BYTES = 64 << 20      # bound on everything --dump-outputs writes


def dump_outputs(out_dir, samples, states, row_major):
    """Write what the last timed step returned as float64 .npy files, so two builds run with the same arguments can be
    compared file by file.  samples: {model: the rows run() returned}, states: {model: [n, state_size] chain state}.
    Per model: `model<m>_samples` [chains, rows, d+1] for a fixed seeded sample of DUMP_CHAINS chains (every row while
    they fit an equal share of DUMP_BYTES, else evenly spaced rows), `model<m>_state` of the same chains, and the
    indices `model<m>_chains` and `model<m>_rows` the sample was taken at."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(0)
    budget = DUMP_BYTES // len(samples) - (1 << 20)    # 1 MB per model left for the state and the index files
    for model in sorted(samples):
        by_chain = samples[model].transpose(0, 1) if row_major else samples[model]    # [n, rows, d+1]
        n, rows, width = by_chain.shape
        chains = np.sort(rng.choice(n, size=min(DUMP_CHAINS, n), replace=False))
        keep = min(rows, budget // (len(chains) * width * 8))
        picked = np.unique(np.linspace(0, rows - 1, keep).round().astype(np.int64))
        ci = torch.as_tensor(chains, device=by_chain.device)
        out = {"samples": by_chain.index_select(0, ci).index_select(1, torch.as_tensor(picked, device=by_chain.device)),
               "state": states[model].index_select(0, ci), "chains": chains, "rows": picked}
        for name, a in out.items():
            a = a.cpu().numpy() if torch.is_tensor(a) else a
            np.save(os.path.join(out_dir, "model%d_%s.npy" % (model, name)), np.ascontiguousarray(a, dtype=np.float64))


# ----------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ----------------------------------------------------------------------------------------------
class Clocks:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t_begin, t_end):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons, power = [], None, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.lines:
            if ts < t_begin or ts > t_end + 0.1:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0]))
                smax = float(f[1])
                power.append(float(f[2]))
            except Exception:
                continue
            for nme, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None}


# ----------------------------------------------------------------------------------------------
# CPU arms
# ----------------------------------------------------------------------------------------------
def _cpu_worker(args):
    """One chain of the reference loop (numpy/scipy restatement, numpy RNG) -- returns (seconds for `iters`, the
    min-over-parameters Geyer ESS of the run's post-burn rows: the same estimator as the GPU arm's ess_per_s)."""
    model, concs, y, theta0, warm, iters, seed = args
    import numpy.random as npr
    import hill_oracle as ho
    from pyhillfit_b200.ess import ess_min
    w0, w100, wo = ho.masks(y)
    pb = ho.compute_pi_bit_of_log_likelihood(wo)

    def target(th):
        return ho.log_target(model, y, w0, w100, wo, concs, th, 1, pb)

    npr.seed(seed)
    with np.errstate(all="ignore"):
        ho.adaptive_metropolis(target, theta0, warm, 5, "fit", rng="numpy")
        t0 = time.perf_counter()
        chain, _ = ho.adaptive_metropolis(target, theta0, iters, 5, "fit", rng="numpy")
        dt = time.perf_counter() - t0
    d = len(theta0)
    post = chain[len(chain) // 4:, :d]            # burn-in removed as PyHillFit.py:861-864 does
    return dt, ess_min(post) * len(chain) / max(len(post), 1)   # ESS of the post-burn rows scaled to the whole run


def cpu_reference_rate(iters, warm=500, cores=None, spread=False):
    """chain-iterations/s and ESS/s of the reference algorithm (oracle port) with one chain per host core.
    spread=False: every core runs Amiodarone/hERG model 2 (BASELINE configs[0]); spread=True: core k runs pair
    17k mod 210 and models alternate, a sample of the config-2 workload."""
    from _data import Table
    from pyhillfit_b200.initial_fit import best_fit
    cores = cores or mp.cpu_count()
    table = Table("crumb_data")
    pairs = table.pairs()
    jobs = []
    for k in range(cores):
        drug, channel = pairs[(17 * k) % len(pairs)] if spread else ("Amiodarone", "hERG")
        model = 1 + (k + 1) % 2 if spread else 2
        concs, y = table.concat(drug, channel)
        theta0, _ = best_fit(model, concs, y)
        jobs.append((model, concs, y, theta0, warm, iters, 25 + k))
    ctx = mp.get_context("fork")
    t0 = time.perf_counter()
    with ctx.Pool(cores) as pool:
        res = pool.map(_cpu_worker, jobs)
    wall = time.perf_counter() - t0
    slowest = max(r[0] for r in res)
    return cores * iters / slowest, cores, wall, float(sum(r[1] for r in res)) / slowest


def cpu_c_port_rate(seconds=2.0):
    """The C restatement (oracle/hill_oracle.c) on all cores: context for how much of the gap is Python."""
    import c_oracle
    import hill_oracle as ho
    from _data import Table
    table = Table("crumb_data")
    concs, y = table.concat("Amiodarone", "hERG")
    cores = mp.cpu_count()
    n = cores * 4
    pb = ho.compute_pi_bit_of_log_likelihood(y)
    theta0 = np.array([6.0, 0.6, 7.7])
    lt0, l10 = c_oracle.log_target_batch(2, concs, y, theta0[None], 1.0, pb)
    st = np.tile(c_oracle.make_state(theta0, lt0[0], l10[0], 0.05 * np.diag(theta0)), (n, 1))
    cls = c_oracle.classify(y)
    iters = 20000
    args = (n, np.full(n, 2, np.int32), np.full(n, len(y), np.int32), np.zeros(n, np.int64), concs, y, cls,
            np.ones(n), np.full(n, pb), st, np.arange(n, dtype=np.int64) * st.shape[1], 0, iters, 5,
            np.full(n, 3000, np.uint32), 0, 25, np.arange(n, dtype=np.uint64), cores)
    t0 = time.perf_counter()
    c_oracle.lib().phf_oracle_am_single_many(*args)
    dt = time.perf_counter() - t0
    return n * iters / dt, cores


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    per_step = max(200, args.ref_iters_per_step)
    rates, ess = [], []
    cores = mp.cpu_count()
    for _ in range(args.warmup):
        cpu_reference_rate(max(100, per_step // 10), warm=50, spread=True)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        r, cores, _, e = cpu_reference_rate(per_step, warm=100, spread=True)
        rates.append(r)
        ess.append(e)
    wall = time.perf_counter() - t0
    value = float(np.mean(rates))
    sample = ("%d chains (one per host core) x %d iterations per step of the PyHillFit single-level AM loop "
              "(numpy/scipy restatement of python/PyHillFit.py:828-856 + doseresponse.py:187-248, numpy MT19937); "
              "core k runs Crumb pair 17k mod 210, models 1 and 2 alternate" % (cores, per_step))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(args.steps, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": DATA,
            "config": {"workload": WORKLOAD % (args.chains_per_pair, 5), "chains_per_pair": args.chains_per_pair, "thinning": 5},
            "config_detail": {"sample": sample},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                             "ess_per_s": float(np.mean(ess))},
            "ess_per_s": float(np.mean(ess)),
            "ess_note": "Geyer initial-positive-sequence ESS (pyhillfit_b200/ess.py), min over parameters, post-burn rows "
                        "of each step's chains, summed over chains / seconds -- the estimator of the GPU arm's ess_per_s; "
                        "a %d-iteration chain has barely started adapting (adaptation begins at 1000 d), so this is an "
                        "early-chain figure" % per_step,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)
    return 0


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
class Ctx:
    """what the sections below share"""
    pass


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--iters-per-step", type=int, default=10000)
    ap.add_argument("--chains-per-pair", type=int, default=64)
    ap.add_argument("--thinning", type=int, default=5)
    ap.add_argument("--ref-iters-per-step", type=int, default=4000)
    ap.add_argument("--e2e-steps", type=int, default=12)
    ap.add_argument("--e2e-segments", type=int, default=64)
    ap.add_argument("--e2e-threads-per-model", type=int, default=2,
                    help="host threads making complete runs of one model concurrently (the library holds two workspaces per model)")
    ap.add_argument("--layout", default="row", choices=["row", "chain"],
                    help="sample layout of the device-timed step AND of the end-to-end call: row = [row][chain][d+1] "
                         "(coalesced write-out, contiguous transfers)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--block-threads", type=int, default=0)
    ap.add_argument("--no-stage", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the sharded TI sweeps / config 5")
    ap.add_argument("--ti-iterations", type=int, default=500000, help="iterations of the TI sweeps (reference default)")
    ap.add_argument("--config5-datasets", type=int, default=1000000)
    ap.add_argument("--config5-iters", type=int, default=1000)
    ap.add_argument("--lanes", type=int, default=0, help="lanes per chain (0: library default)")
    ap.add_argument("--occupancy-hint", type=int, default=0, help="developer knob: min CTAs/SM variant")
    ap.add_argument("--cta-order", type=int, default=0, help="developer knob: 0 chain blocks by decreasing cost, 1 index order")
    ap.add_argument("--serial-models", action="store_true", help="run the two models back to back on one stream")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a fixed sample of the rows and chain state the last timed step "
                         "produced (rank 0) as DIR/<name>.npy, float64, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference_arm(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    from pyhillfit_b200 import _lib
    from pyhillfit_b200.sampler import SingleLevelSampler

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        # each rank's host threads (the end-to-end calls, the pinned-buffer copies) stay on their own slice of the cores
        try:
            cores = sorted(os.sched_getaffinity(0))
            per = max(len(cores) // world, 1)
            os.sched_setaffinity(0, cores[local * per:(local + 1) * per] or cores)
        except Exception:
            pass

    pack, wl = build_workload(args.chains_per_pair)
    thin = args.thinning
    K = args.iters_per_step
    rows_per_step = K // thin
    row_major = args.layout == "row"
    samplers, buffers, streams = {}, {}, {}
    n_chains = 0
    for model in (1, 2):
        w = wl[model]
        n = len(w["ids"])
        # disjoint Philox streams per rank: global chain id = rank * n_total + local index
        s = SingleLevelSampler(model, pack, w["ids"], 1.0, w["theta0"], variant="fit", seed=25,
                               chain_id_base=(rank * 2 + (model - 1)) * (1 << 32), thinning=thin, device=dev,
                               stage=not args.no_stage, block_threads=args.block_threads, lanes=args.lanes,
                               co_resident_chains=0 if args.serial_models else len(wl[3 - model]["ids"]))
        s.occupancy_hint = args.occupancy_hint
        s.cta_order = args.cta_order
        samplers[model] = s
        buffers[model] = torch.empty((rows_per_step + 1, n, w["d"] + 1) if row_major else
                                     (n, rows_per_step + 1, w["d"] + 1), dtype=torch.float64, device=dev)
        streams[model] = torch.cuda.Stream(device=dev)
        n_chains += n
    flops_iter = sum(wl[m]["flops"] * len(wl[m]["ids"]) for m in (1, 2)) / n_chains
    bytes_iter = sum((wl[m]["d"] + 1) * 8.0 / thin * len(wl[m]["ids"]) for m in (1, 2)) / n_chains
    e2e_state0 = {m: samplers[m].state.cpu() for m in (1, 2)}    # the start state of a complete run (for run_e2e)

    main_stream = torch.cuda.current_stream(dev)
    stream_events = None
    returned = {}     # the rows each model's latest run() returned

    def step(first=True, last=True):
        """one step = one launch per model; the two models' launches go to two streams.  Inside a run of steps the
        streams are not joined between steps (each stream's launches are ordered among themselves and share nothing
        with the other stream): `first` makes the streams wait for the main stream, `last` makes the main stream wait
        for them."""
        if args.serial_models:
            for model in (2, 1):
                returned[model] = samplers[model].run(K, samples=buffers[model], row_major=row_major)
            return
        if first:
            ev = torch.cuda.Event()
            ev.record(main_stream)
        for model in (1, 2):
            st = streams[model]
            if first:
                st.wait_event(ev)
            with torch.cuda.stream(st):
                if stream_events is not None:   # per-launch duration on the launching stream
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record(st)
                returned[model] = samplers[model].run(K, samples=buffers[model], row_major=row_major)
                if stream_events is not None:
                    b.record(st)
                    stream_events[model].append((a, b))
        if last:
            for model in (1, 2):
                main_stream.wait_stream(streams[model])

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        if world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(args.warmup):
        step()
    barrier()
    clocks = Clocks(local)
    if rank == 0:
        clocks.start()
        time.sleep(0.3)
    launches0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_begin = time.time()
    stream_events = {1: [], 2: []}
    e0.record(main_stream)
    for k in range(args.steps):
        step(first=k == 0, last=k == args.steps - 1)
    e1.record(main_stream)
    barrier()
    t_end = time.time()
    ms = e0.elapsed_time(e1)
    launch_ms_timed = {m: float(np.mean([a.elapsed_time(b) for a, b in stream_events[m]])) if stream_events[m] else None
                       for m in (1, 2)}
    stream_events = None
    launches = _lib.launch_count() - launches0
    clk = clocks.stop(t_begin, t_end) if rank == 0 else None
    ms = max_over_ranks(ms)
    total_iters = float(n_chains) * K * args.steps * world
    value = total_iters / (ms * 1e-3)
    if args.dump_outputs and rank == 0:     # before the launches below overwrite the buffers and advance the chains
        dump_outputs(args.dump_outputs, returned, {m: samplers[m].state for m in (1, 2)}, row_major)

    # ---- per-kernel launch durations (each model's kernel alone on the device), for the roofline ----
    kern_ms = {}
    for model in (1, 2):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        a.record(main_stream)
        samplers[model].run(K, samples=buffers[model], row_major=row_major)
        b.record(main_stream)
        torch.cuda.synchronize(dev)
        kern_ms[model] = a.elapsed_time(b)

    # ---- ESS/s from the last written step (256 chains per model sampled, min over parameters, Geyer IPS) ----
    ess_per_s = None
    acc = None
    if rank == 0:
        from pyhillfit_b200.ess import ess_min
        rng = np.random.default_rng(0)
        per_row = []
        for model in (1, 2):
            n = samplers[model].n
            pick = rng.choice(n, size=min(256, n), replace=False)
            by_chain = buffers[model].transpose(0, 1) if row_major else buffers[model]
            smp = by_chain[torch.as_tensor(pick, device=dev)][:, :rows_per_step, :wl[model]["d"]].cpu().numpy()
            per_row.append(np.mean([ess_min(c) for c in smp]) / rows_per_step)
        rows_per_s = value / thin
        ess_per_s = float(np.mean(per_row) * rows_per_s)
        acc = float(np.mean([samplers[m].acceptance().mean() for m in (1, 2)]))

    cx = Ctx()
    cx.args, cx.torch, cx.dist, cx.dev, cx.pack, cx.wl, cx.rank, cx.world, cx.local = args, torch, dist, dev, pack, wl, rank, world, local
    cx.barrier, cx.max_over_ranks, cx.samplers = barrier, max_over_ranks, samplers

    # ---- end to end through the host-buffer C ABI (pinned host memory) ----
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(cx, e2e_state0)
    del buffers

    # ---- the north-star's strong-scaling workloads, sharded over the ranks ----
    strong = None
    if not args.no_strong and not args.no_other_configs:
        strong = strong_configs(cx)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    peak_tf, _ = _lib.fp64_peak_tflops(5)
    # The hot path is ONE kernel template, am_single_kernel<MODEL, LANES>, launched once per model per step; the two
    # launches run on two streams and share the SMs for the whole step (each lasts ~ the step).  Its roofline entry
    # is therefore taken over the timed region itself: algorithmic flops of both launches / (their common duration
    # = mean step time).  The model-2 launch timed alone (under-occupied at 13 440 chains) is reported beside it.
    n2 = samplers[2].n
    step_flops = sum(samplers[m].n * K * wl[m]["flops"] for m in (1, 2))
    ach_tf = step_flops / (ms / args.steps * 1e-3) / 1e12
    alone_tf = n2 * K * wl[2]["flops"] / (kern_ms[2] * 1e-3) / 1e12
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    traffic = None
    try:   # dram__bytes_read.sum + dram__bytes_write.sum of this kernel from the committed `ncu --set full` capture
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["am_single_kernel<2>"]
        traffic = tr["dram_bytes_per_chain_iteration"] * n_chains * K * (bytes_iter / 6.4)
    except Exception:
        pass
    ncu_util = None
    try:   # FP64-pipe and issue-slot utilisation of this kernel from the committed `ncu --set full` captures
        ncu_util = json.load(open(os.path.join(ROOT, "profiles", "pipe_utilisation.json")))
    except Exception:
        pass
    roofline = {"bound": "fp64", "achieved": ach_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach_tf / peak_tf,
                "traffic": traffic, "ncu": ncu_util,
                "kernel": "am_single_kernel<model 1 | model 2, %d lanes per chain> (two co-resident launches per step)"
                          % samplers[2].lanes,
                "launch_ms": ms / args.steps, "launch_ms_on_stream": launch_ms_timed,
                "flops_per_chain_iteration": flops_iter,
                "peak_source": "phf_fp64_peak_probe (live DFMA microbenchmark; MEASURED_PEAKS.json has no FP64 entry; "
                               "ncu FP64-pipe page of the probe kernel: profiles/r02_fp64_peak_probe_ncu.txt)",
                "algorithmic_bytes": n_chains * K * bytes_iter,
                "model2_launch_alone": {"launch_ms": kern_ms[2], "achieved": alone_tf, "frac": alone_tf / peak_tf,
                                        "flops_per_chain_iteration": wl[2]["flops"]},
                "hbm": {"achieved_gbs": n_chains * K * bytes_iter / (ms / args.steps * 1e-3) / 1e9, "peak_gbs": hbm_peak,
                        "peak_source": "MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback",
                        "algorithmic_bytes_per_chain_iteration": bytes_iter}}
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        r, cores, wall, cpu_ess = cpu_reference_rate(6000, warm=300)
        rc, _ = cpu_c_port_rate()
        cpu_baseline = {"value": r, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": "%d chains (one per host core) x 6000 iterations of the reference's single-level AM "
                                  "loop, numpy/scipy restatement (oracle/hill_oracle.py), Amiodarone/hERG model 2; "
                                  "%.1f s wall" % (cores, wall),
                        "ess_per_s": cpu_ess,
                        "ess_note": "same Geyer estimator as the GPU arm's ess_per_s (pyhillfit_b200/ess.py), min over "
                                    "parameters, post-burn rows, summed over the chains / seconds",
                        "c_port_value": rc,
                        "c_port_note": "same loop in plain C (oracle/hill_oracle.c, Philox RNG) on all cores"}
    other = {}
    if strong:
        for k, v in strong.items():
            if "flops_per_chain_iteration" in v:
                tf = v["value"] * v["flops_per_chain_iteration"] / 1e12
                v["roofline"] = {"bound": "fp64", "achieved": tf, "peak": peak_tf * world, "unit": "TFLOP/s",
                                 "frac": tf / (peak_tf * world), "flops_per_chain_iteration": v["flops_per_chain_iteration"]}
            other[k] = v
    if world == 1 and not args.no_other_configs:
        c3 = config3(cx)
        for k, v in c3.items():
            tf = v["value"] * v["flops_per_chain_iteration"] / 1e12
            v["roofline"] = {"bound": "fp64", "achieved": tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": tf / peak_tf,
                             "flops_per_chain_iteration": v["flops_per_chain_iteration"]}
            other[k] = v
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": DATA,
            "config": {"workload": WORKLOAD % (args.chains_per_pair, thin), "chains_per_pair": args.chains_per_pair, "thinning": thin,
                       "l2": "no flush needed: each step writes %.2f GB of thinned samples (> 126 MB L2); chain state is "
                             "register-resident, packed data (54 KB) is staged in shared memory" %
                             (n_chains * K * bytes_iter / 1e9)},
            "config_detail": {"chains_per_gpu": n_chains,
                              "iters_per_step": K, "sample_layout": args.layout + "-major (value and e2e alike)",
                              "theta0": "host least-squares fit; chains 1..63 of a pair jittered by 2%",
                              "target_1e10_frac": value / world / 1e10},
            "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "gpu_launches": int(launches),
            "clocks": clk, "ess_per_s": ess_per_s, "mean_acceptance": acc,
            "hbm_bytes_per_chain_iteration": bytes_iter, "flops_per_chain_iteration": flops_iter,
            "kernel_ms": {"am_single_kernel<1>": kern_ms[1], "am_single_kernel<2>": kern_ms[2]},
            "other_configs": other or None}
    emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


def _timed(torch, fn, reps=3):
    fn()
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        best = min(best, a.elapsed_time(b))
    return best * 1e-3


# ----------------------------------------------------------------------------------------------
# strong scaling: the whole job is fixed, the ranks shard it
# ----------------------------------------------------------------------------------------------
def strong_configs(cx):
    """The north-star's multi-GPU workloads, each a FIXED total job sharded over the ranks (`scaling: strong`):
      * the reference's thermodynamic-integration sweep -- 41 temperatures (python/PyHillTemp.py:151) x 210 pairs x
        models {1, 2} x `--ti-iterations` iterations -- and BASELINE config 4 (64 temperatures), through ti.run_ti: chains
        sharded contiguously by cost, no collective while sampling, then ONE all-gather per model of the per-chain mean
        temperature-1 log-likelihoods (NCCL) and the trapezium rule (compute_bayes_factors.py:77-100).  The timed region
        (CUDA events on the launching stream, max over ranks) covers sampling + all-gather + integration; the NCCL
        communicator is brought up by the warm-up call;
      * BASELINE config 5: 10^6 synthetic datasets x 4 chains, model 2, samples written to HBM."""
    torch, dist, dev, world, rank = cx.torch, cx.dist, cx.dev, cx.world, cx.rank
    from pyhillfit_b200 import synthetic, ti
    from pyhillfit_b200.packing import SinglePack
    from pyhillfit_b200.sampler import SingleLevelSampler
    args, pack, data = cx.args, cx.pack, cx.wl["data"]
    out = {}
    main_stream = torch.cuda.current_stream(dev)
    w = {m: cx.wl[m]["flops_per_dataset"] for m in (1, 2)}
    w0 = {m: np.array([flops_per_iteration(m, pack.groups[b:b + n], prior_only=True) for b, n in
                       zip(pack.datasets["group_begin"], pack.datasets["n_groups"])], dtype=float) for m in (1, 2)}
    for tag, temps in (("config4_ti_41_temperatures_reference_sweep", ti.temperature_ladder(40, 3)),
                       ("config4_ti_64_temperatures", ti.temperature_ladder(63, 3))):
        T = len(temps)
        chains = 2 * 210 * T
        iters = args.ti_iterations
        # warm-up: the same call, short (brings up the NCCL communicator and the all-gather path, loads the kernels)
        ti.run_ti(data, temps=temps, iterations=10000, segment=10000, seed=1, device=dev, pack=pack)
        # rank-count independence: with a fixed lane count the result is bit-identical for every N (the digest)
        chk = ti.run_ti(data, temps=temps, iterations=20000, segment=20000, seed=1, device=dev, pack=pack, lanes=2)
        digest = hashlib.sha256(np.ascontiguousarray(chk["B12"]).tobytes()).hexdigest()[:16]
        cx.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(main_stream)
        res = ti.run_ti(data, temps=temps, iterations=iters, segment=iters, seed=1, device=dev, pack=pack)
        e1.record(main_stream)
        torch.cuda.synchronize(dev)
        wall = time.perf_counter() - t0
        sec = cx.max_over_ranks(e0.elapsed_time(e1) * 1e-3)
        sample_s = cx.max_over_ranks(res.get("sample_seconds", 0.0))
        gather_s = cx.max_over_ranks(res["gather_seconds"])
        lb = np.log(res["B12"])
        flops = sum((w[m].sum() * (T - 1) + w0[m].sum()) for m in (1, 2)) / chains    # t = 0 chains: prior only
        out[tag] = {"scaling": "strong", "chains": chains, "chains_per_gpu_rank0": res["chains_local"], "iters": iters,
                    "value": chains * iters / sec, "unit": UNIT, "seconds": sec, "wall_seconds": cx.max_over_ranks(wall),
                    "phase_seconds": {"sampling_max_over_ranks": sample_s, "all_gather_and_trapezium": gather_s},
                    "lanes_rank0": res["lanes"], "speculation_rank0": res["speculation"],
                    "flops_per_chain_iteration": float(flops),
                    "ln_B12": {"mean_over_pairs": float(lb.mean()), "min": float(lb.min()), "max": float(lb.max()),
                               "Amiodarone_hERG": float(lb[0])},
                    "rank_count_independence": {"lanes": 2, "iterations": 20000, "B12_sha256_16": digest,
                                                "note": "same digest at every N: sharding changes no bit"},
                    "timing": "CUDA events on the launching stream around ti.run_ti (sampling on two streams ordered after "
                              "it, NCCL all-gather of per-chain means, trapezium), barrier before, max over ranks",
                    "reference": "python/PyHillTemp.py:151-161, python/compute_bayes_factors.py:77-100"}
    # ---- config 5 ----
    n_total = args.config5_datasets
    lo, hi = rank * n_total // world, (rank + 1) * n_total // world
    t0 = time.perf_counter()
    concs, Y, truth = synthetic.generate(hi - lo, offset=lo)
    sp = SinglePack.from_uniform(concs, Y)
    t_pack = time.perf_counter() - t0
    ids5 = np.repeat(np.arange(sp.n_datasets, dtype=np.int32), 4)
    s5 = SingleLevelSampler(2, sp, ids5, 1.0, np.tile([6.0, 1.0, 6.0], (len(ids5), 1)), variant="fit", seed=9,
                            chain_id_base=4 * lo, thinning=5, device=dev)
    K5 = args.config5_iters
    buf5 = torch.empty((K5 // 5, s5.n, 4), dtype=torch.float64, device=dev)
    s5.run(K5, samples=buf5, row_major=True)
    cx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 3
    e0.record(main_stream)
    for _ in range(reps):
        s5.run(K5, samples=buf5, row_major=True)
    e1.record(main_stream)
    torch.cuda.synchronize(dev)
    sec5 = cx.max_over_ranks(e0.elapsed_time(e1) * 1e-3)
    pick = np.arange(0, sp.n_datasets, max(sp.n_datasets // 2000, 1))
    w5 = float(np.mean([flops_per_iteration(2, sp.groups[b:b + n]) for b, n in
                        zip(sp.datasets["group_begin"][pick], sp.datasets["n_groups"][pick])]))
    out["config5_synthetic_1M_datasets"] = {
        "scaling": "strong", "chains": 4 * n_total, "chains_per_gpu": s5.n, "iters": K5 * reps,
        "value": 4.0 * n_total * K5 * reps / sec5, "unit": UNIT, "seconds": sec5, "lanes": s5.lanes,
        "flops_per_chain_iteration": w5, "generate_and_pack_s_per_rank": round(t_pack, 2),
        "note": "%d synthetic datasets x 4 chains, model 2, datasets sharded over the ranks (dataset k is the same for "
                "every N), row-major samples written to HBM (%.1f GB per %d iterations per GPU); no collective"
                % (n_total, buf5.numel() * 8 / 1e9, K5)}
    del buf5, s5
    return out


def config3(cx):
    """Device-timed throughput of BASELINE config 3 (hierarchical; context, not the headline): four launches on four
    streams, samples written, best of 3; the same through phf_am_hier_run_host."""
    torch, dev = cx.torch, cx.dev
    from _data import Table
    from pyhillfit_b200.packing import HierPack
    from pyhillfit_b200.sampler import HierarchicalSampler, hier_priors
    out = {}
    table = Table("crumb_data")
    pr, shapes, scales, locs = hier_priors()
    pairs = table.pairs()
    by_ne = {}
    for ip, (dg, ch) in enumerate(pairs):
        by_ne.setdefault(len(table.experiments(dg, ch)), []).append(ip)
    K3 = 1000
    hier, tot_n, tot_flops = [], 0, 0.0
    n_all = 256 * len(pairs)
    for ne, idxs in sorted(by_ne.items()):
        exs = [table.experiments(*pairs[i]) for i in idxs]
        hp = HierPack(exs)
        hid = np.repeat(np.arange(len(idxs), dtype=np.int32), 256)
        th0 = np.tile(np.concatenate(([1.0, 4.0, 6.0, 0.3], np.tile([5.5, 1.0], ne), [8.0])), (len(hid), 1))
        hs = HierarchicalSampler(hp, hid, th0, pr, seed=ne, thinning=5, device=dev, co_resident_chains=n_all - len(hid))
        hb = torch.empty((hs.n, K3 // 5, hs.d + 1), dtype=torch.float64, device=dev)
        hier.append((hs, hb, torch.cuda.Stream(device=dev)))
        tot_n += hs.n
        tot_flops += 256.0 * sum(hier_flops_per_iteration(ne, sum(len(e) for e in ex)) for ex in exs)
    from pyhillfit_b200 import _lib as _l
    _lib_hier_lanes = _l.load().phf_am_hier_lanes
    per_ne = {}
    serial_t = 0.0
    for hs, hb, _ in hier:
        t = _timed(torch, lambda hs=hs, hb=hb: hs.run(K3, samples=hb))
        serial_t += t
        with torch.cuda.device(dev):
            form = hs.lanes or int(_lib_hier_lanes(hs.n_expts, hs.n))
        per_ne["Ne=%d" % hs.n_expts] = {"chains": hs.n, "value_alone": hs.n * K3 / t, "lanes_per_chain": form}

    def all_at_once():   # the four launches are independent: one stream each, the small ones fill the big one's gaps
        ev = torch.cuda.Event()
        ev.record()
        for hs, hb, st in hier:
            st.wait_event(ev)
            with torch.cuda.stream(st):
                hs.run(K3, samples=hb)
            done = torch.cuda.Event()
            done.record(st)
            torch.cuda.current_stream().wait_event(done)
    tot_t = _timed(torch, all_at_once)
    # the same through phf_am_hier_run_host: pinned host buffers in and out, row-major samples, one host thread per Ne
    import ctypes as C
    from pyhillfit_b200 import _lib
    L = _lib.load()
    jobs = []
    for hs, _, _ in hier:
        st = torch.empty((hs.n, _lib.state_size(hs.d)), dtype=torch.float64).pin_memory()
        st.copy_(hs.state.cpu())
        smp = torch.empty((K3 // 5, hs.n, hs.d + 1), dtype=torch.float64).pin_memory()
        jobs.append(dict(hs=hs, state=st, samples=smp, ids=np.ascontiguousarray(hs.dataset_id.cpu().numpy()), t0=hs.t))

    def host_call(j):
        hs = j["hs"]
        cfg = _lib.AmConfig(model=0, reset_mean_at_adapt=0, t0=j["t0"], n_iters=K3, thinning=5, adapt_when=hs.adapt_when,
                            burn_rows=0xFFFFFFFF, rows_capacity=K3 // 5, seed=hs.seed, chain_id_base=0, stage_groups=0,
                            block_threads=0, lanes_per_chain=0, sample_layout=_lib.SAMPLES_ROW_MAJOR)
        _lib.check(L.phf_am_hier_run_host(C.byref(cfg), hs.n_expts, hs.n, j["state"].data_ptr(), j["ids"].ctypes.data,
                                          hs.pack.n_datasets, hs.pack.datasets.ctypes.data, len(hs.pack.points),
                                          hs.pack.points.ctypes.data, C.byref(pr), j["samples"].data_ptr(), 8,
                                          dev.index), "phf_am_hier_run_host")
        j["t0"] += K3

    def host_step():
        th = [threading.Thread(target=host_call, args=(j,)) for j in jobs]
        for t in th:
            t.start()
        for t in th:
            t.join()
    host_step()
    torch.cuda.synchronize(dev)
    e2e_t = []
    for _ in range(3):
        t0 = time.perf_counter()
        host_step()
        e2e_t.append(time.perf_counter() - t0)
    e2e3 = {"value": tot_n * K3 / min(e2e_t), "unit": UNIT,
            "h2d_bytes_per_step": int(sum(j["state"].numel() * 8 + j["ids"].nbytes + j["hs"].pack.points.nbytes +
                                          j["hs"].pack.datasets.nbytes for j in jobs)),
            "d2h_bytes_per_step": int(sum((j["samples"].numel() + j["state"].numel()) * 8 for j in jobs)),
            "api": "phf_am_hier_run_host (pinned host buffers, row-major samples, 8 overlapped segments/call, one host "
                   "thread per number of experiments; the hierarchical loop keeps its burn-in rows: PyHillFit.py:514-515), "
                   "best of 3"}
    del jobs
    out["config3_hierarchical"] = {"chains": tot_n, "iters": K3, "value": tot_n * K3 / tot_t, "unit": UNIT,
                                   "value_back_to_back": tot_n * K3 / serial_t, "e2e": e2e3, "per_n_expts": per_ne,
                                   "flops_per_chain_iteration": tot_flops / tot_n,
                                   "note": "dim 11..17, four launches (Ne = 3, 4, 5, 6) on four streams; lanes_per_chain: 1 = one "
                                           "thread per chain, 4 = four lanes per chain, 16 / 32 = one lane per parameter"}
    return out


def run_e2e(cx, state0):
    """The same metric through the reference-facing call, phf_am_single_run_host, with pinned HOST buffers.  One step =
    one complete PyHillFit run of `--iters-per-step` iterations of every chain: start state and packed data copied in
    (H2D), K iterations, the rows the reference SAVES copied back -- it drops the first quarter of the saved rows
    before np.savetxt (python/PyHillFit.py:861-864), so those are neither written nor transferred
    (cfg.discard_burn_rows) -- plus the final state (D2H).  Each model is driven by `--e2e-threads-per-model` host threads
    (the library keeps two workspaces per model), each making its share of the `--e2e-steps` runs back to back (a call
    returns when its results are on the host), so one run's transfers fall into another's burn-in phase, when a run has
    nothing to copy; the timed region is the wall clock from the barrier to the last call's return."""
    import ctypes as C
    from pyhillfit_b200 import _lib
    args, torch, dev, pack, wl, rank, world = cx.args, cx.torch, cx.dev, cx.pack, cx.wl, cx.rank, cx.world
    L = _lib.load()
    thin, K = args.thinning, args.iters_per_step
    saved = K // thin + 1
    burn = saved // 4                       # burn_in_fraction = 4 (PyHillFit.py:37)
    rows = saved - burn                     # rows burn .. saved-1 are kept
    row_major = args.layout == "row"
    jobs = {}
    h2d = d2h = 0
    T = args.e2e_threads_per_model
    for model in (1, 2):
        w = wl[model]
        n, d = len(w["ids"]), w["d"]
        st0 = state0[model].pin_memory()
        ids = np.ascontiguousarray(w["ids"])
        temps = np.ones(n)
        for k in range(T):      # every host thread owns its result buffers
            st = torch.empty_like(st0).pin_memory()
            # row-major samples: [row][chain][d+1], every segment is one contiguous device -> host transfer
            smp = torch.empty((rows, n, d + 1) if row_major else (n, rows, d + 1), dtype=torch.float64).pin_memory()
            jobs[(model, k)] = dict(n=n, state0=st0, state=st, samples=smp, ids=ids, temps=temps)
        h2d += st.numel() * 8 + ids.nbytes + temps.nbytes + pack.datasets.nbytes + pack.groups.nbytes
        d2h += smp.numel() * 8 + st.numel() * 8

    def call(model, k):
        j = jobs[(model, k)]
        j["state"].copy_(j["state0"])       # a complete run starts from the start state (host copy, inside the timed region)
        cfg = _lib.AmConfig(model=model, reset_mean_at_adapt=0, t0=0, n_iters=K, thinning=thin,
                            adapt_when=1000 * wl[model]["d"], burn_rows=burn, discard_burn_rows=1, rows_capacity=rows,
                            seed=25, chain_id_base=(rank * 2 + (model - 1)) * (1 << 32),
                            stage_groups=cx.samplers[model].stage_groups, block_threads=cx.samplers[model].block_threads,
                            lanes_per_chain=cx.samplers[model].lanes,
                            sample_layout=_lib.SAMPLES_ROW_MAJOR if row_major else _lib.SAMPLES_CHAIN_MAJOR)
        rc = L.phf_am_single_run_host(C.byref(cfg), j["n"], j["state"].data_ptr(), j["ids"].ctypes.data,
                                      j["temps"].ctypes.data, pack.n_datasets, pack.datasets.ctypes.data,
                                      len(pack.groups), pack.groups.ctypes.data, j["samples"].data_ptr(),
                                      args.e2e_segments, dev.index)
        _lib.check(rc, "phf_am_single_run_host")

    def run(steps):
        errs = []

        def loop(model, k):
            try:
                for _ in range(steps // T):
                    call(model, k)
            except Exception as e:      # surface a failure of a worker thread
                errs.append(e)
        th = [threading.Thread(target=loop, args=(m, k)) for m in (1, 2) for k in range(T)]
        for t in th:
            t.start()
        for t in th:
            t.join()
        if errs:
            raise errs[0]

    assert args.e2e_steps % T == 0
    run(2 * T)
    cx.barrier()
    t0 = time.perf_counter()
    run(args.e2e_steps)
    torch.cuda.synchronize(dev)
    dt = cx.max_over_ranks(time.perf_counter() - t0)
    total = float(sum(len(wl[m]["ids"]) for m in (1, 2))) * K * args.e2e_steps * world
    finite = bool(all(np.isfinite(j["samples"][-1].numpy()).all() for j in jobs.values()))
    return {"value": total / dt, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
            "steps": args.e2e_steps, "rows_kept_per_chain": rows, "rows_discarded_as_burn_in": burn - 1,
            "last_row_finite": finite,
            "api": "phf_am_single_run_host (pinned host buffers, %s-major samples, %d overlapped segments/call, "
                   "cfg.discard_burn_rows = 1: the burn-in rows PyHillFit.py:861-864 drops are not transferred; %d host "
                   "thread(s) per model, each making its calls back to back)" % (args.layout, args.e2e_segments, T),
            "timing": "host wall clock from the barrier to the return of the last call (each call ends with a stream "
                      "synchronise); max over ranks"}


if __name__ == "__main__":
    sys.exit(main())
