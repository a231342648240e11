#!/usr/bin/env python
"""bench.py — spans/sec of the span-assignment hot path (TraceWeaverV3.FindAssignments,
BASELINE.json north_star) on synthetic span streams of the shapes BASELINE.json names.

    python bench.py --gpus N --steps K --warmup W                     # ours (CUDA engine via the C ABI)
    python bench.py --impl reference --gpus N --steps K --warmup W    # CPU arm: the reference's algorithm
                                                                      # (oracle/ C port, host cores)
    --workload {hotel,media,alibaba}   stream shape of the headline line (default hotel = configs[1] shape)
    --scaling {weak,strong}            weak: 8192 services per GPU; strong: ONE fixed list (--spans, default 100 M)
    --no-extra                         skip the extra_workloads legs (media-shaped, alibaba-shaped, shipped traces)
    --dump-outputs DIR                 after the timed steps, write the arrays the last step returned (rank 0;
                                       the reference arm's inputs scale with the host's core count)

One "step" = one pass of the whole path (both iterations + GMM refit) over the service list.  The
list is ONE global list partitioned across the ranks by span count (traceweaver_b200.shard); every
step ends with the path's single collective, an all-gather of the per-service assignment arrays
(NCCL), inside the timed region.  value = spans of the whole list / max-over-ranks time.  Prints ONE
JSON line on rank 0.

  value      device-timed throughput with the span arrays already resident in HBM
  e2e        the same metric through the public batch API with HOST buffers: every step copies the
             caller's arrays into pinned staging (host memcpy), H2D, solves, D2H of assignments /
             top-K / counters — all inside the timed region; inputs are rewritten in place between
             steps so nothing can be cached
  roofline   scoring kernel (k_score3, GMM pass = the final top-K lists): algorithmic bytes /
             CUDA-event time / measured HBM peak
  cpu_baseline   oracle/ (C restatement of the reference, kind "port") on a bounded sample of the
             same services, one thread per physical core, rank 0 at N=1
  extra_workloads (N=1): the same measurements on the media-shaped and alibaba-shaped streams and on
             the shipped Jaeger directories (the problems of tests/golden, hotel x12 / media / nodejs)
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

METRIC = "spans/sec reconstructed (in+out spans of all solved services)"
UNIT = "spans/s"
WORKLOAD_TEXT = {
    "hotel": "hotel_reservation-shaped synthetic span stream (BASELINE configs[1] shape: frontend E=3 chain+"
             "transitive edge, search E=2 chain; six load levels 25..150; log-normal delays calibrated on the "
             "reference traces)",
    "media": "media_microservices-shaped synthetic span stream (BASELINE configs[2] shape: nginx E=4 parallel, "
             "movie-id E=2 parallel, four one-callee services; loads 25..150; calibrated on media_load100)",
    "alibaba": "alibaba-shaped synthetic window (BASELINE configs[3]; the trace is not shipped): 1..4 callees, "
               "millisecond clocks, exps/exp5 time compression as load",
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="hotel", choices=["hotel", "media", "alibaba"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--services", type=int, default=8192, help="services per GPU (weak scaling)")
    ap.add_argument("--spans", type=int, default=100_000_000, help="total spans of the list (strong scaling)")
    ap.add_argument("--n-in", type=int, default=1000, help="incoming spans per service")
    ap.add_argument("--cpu-sample", type=int, default=1536, help="services in the CPU-baseline sample")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--seed", type=int, default=10)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path returned in its last step as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


DUMP_BYTES = 63_000_000       # all files of --dump-outputs together, .npy headers included, stay under 64 MB


def host_outputs(res):
    """One step's result as host arrays: tensors copied out, distribution Params as their table."""
    import torch
    out = {}
    for name, v in res.items():
        v = getattr(v, "table", v)
        out[name] = v.cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)
    return out


def topk_rows(flat, hb):
    """topk_idx, laid out [in-span][rank][callee] with each service's own callee count
    (include/traceweaver_b200.h), as one row of TW_K candidate indices per (in-span, callee) tuple, in
    the tuple order of `assign`."""
    from traceweaver_b200 import _abi
    per = np.diff(hb.prob_tuple_off).astype(np.int64)
    E = np.repeat(np.diff(hb.prob_ep_off).astype(np.int64), per)
    t = np.arange(len(E), dtype=np.int64)
    e = (t - np.repeat(np.asarray(hb.prob_tuple_off[:-1], np.int64), per)) % E
    base = _abi.TW_K * (t - e) + e
    flat = np.asarray(flat)
    return np.stack([flat[base + r * E] for r in range(_abi.TW_K)], axis=1)


def dump_outputs(directory, arrays, hb=None):
    """Writes every array as DIR/<name>.npy in float64 (the integer outputs convert exactly).  topk_idx
    is written as one top-K row per tuple (topk_rows; `hb` is the batch that was solved).  The top-K
    score lists are NaN-padded past topk_cnt (include/traceweaver_b200.h); those empty slots are written
    as 0, and any other non-finite value is an error.  An array larger than an equal share of DUMP_BYTES
    keeps a fixed, seeded sample of its rows (whole rows), so that two builds run with the same
    arguments can be compared file by file."""
    arrays = dict(arrays)
    if "topk_idx" in arrays:
        arrays["topk_idx"] = topk_rows(arrays["topk_idx"], hb)
    if "topk_score" in arrays:
        s = np.array(arrays["topk_score"], np.float64)
        s[np.arange(s.shape[1]) >= np.asarray(arrays["topk_cnt"])[:, None]] = 0.0
        arrays["topk_score"] = s
    os.makedirs(directory, exist_ok=True)
    share = DUMP_BYTES // max(len(arrays), 1)
    for name, a in arrays.items():
        a = np.asarray(a)
        if a.ndim and 8 * a.size > share:
            keep = share // (8 * (a.size // len(a)))
            a = a[np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))]
        a = a.astype(np.float64)
        if not np.all(np.isfinite(a)):
            raise ValueError(f"--dump-outputs: {name} holds non-finite values")
        np.save(os.path.join(directory, name + ".npy"), a)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index):
        self.rows, self.stop = [], threading.Event()
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        self.cmd = ["nvidia-smi", f"--id={index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"]
        self.th = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(self.cmd, capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.05)

    def start(self):
        self.th.start()
        return self

    def finish(self):
        self.stop.set()
        self.th.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


def accuracy(eng, assign, truth, hb):
    """Fraction of incoming spans whose children are all assigned correctly (AccuracyForService,
    helpers/utils.py:62-79, on index arrays), computed on the device by tw_accuracy (csrc/tw_truth.cu)."""
    from traceweaver_b200 import truth as dev_truth
    tl = dev_truth.TraceLists.from_host_batch(hb, None, 0)
    a = dev_truth.accuracy(eng, tl, truth, assign, resident=eng.d)
    return float(a["correct"].sum()) / max(int(a["n_in"].sum()), 1)


def physical_cores():
    """One hardware thread per physical core, from the kernel's topology files (sched affinity aware)."""
    try:
        allowed = sorted(os.sched_getaffinity(0))
    except AttributeError:
        return list(range(os.cpu_count() or 1))
    seen, pick = set(), []
    for c in allowed:
        try:
            sib = open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list").read().strip()
        except OSError:
            sib = str(c)
        if sib not in seen:
            seen.add(sib)
            pick.append(c)
    return pick or allowed


def run_oracle_pinned(hb, seed, want_topk=True):
    """The CPU port on one thread per physical core (pinned): oversubscribed hyper-threads made the
    round-1 CPU arm swing 4.5x between hosts."""
    from oracle import tw_oracle
    cores = physical_cores()
    old = None
    try:
        old = os.sched_getaffinity(0)
        os.sched_setaffinity(0, cores)
    except (AttributeError, OSError):
        pass
    try:
        t0 = time.perf_counter()
        res = tw_oracle.find_assignments(hb, seed, len(cores), want_topk=want_topk)
        dt = time.perf_counter() - t0
    finally:
        if old is not None:
            try:
                os.sched_setaffinity(0, old)
            except OSError:
                pass
    return res, dt, len(cores)


def sample_blocks(blocks, per):
    from traceweaver_b200.batch import ServiceBlock
    out = []
    for b in blocks:
        k = min(per, b.in_start.shape[0])
        out.append(ServiceBlock(in_start=b.in_start[:k], in_end=b.in_end[:k], out_start=[o[:k] for o in b.out_start],
                                out_end=[o[:k] for o in b.out_end], preds=b.preds, truth=b.truth[:, :k], name=b.name))
    return out


def cpu_baseline(blocks, gpu_assign, n_services_sample, seed, gpu_assign_pass0=None, dev_index=None):
    """oracle/ on the first services of every block (same inputs) + parity of the engine on them."""
    from traceweaver_b200.batch import build_batch_from_blocks
    per = max(1, n_services_sample // len(blocks))
    sample = sample_blocks(blocks, per)
    shb = build_batch_from_blocks(sample)
    n_spans = int(sum(s.in_start.size * (1 + len(s.out_start)) for s in sample))
    res, dt, cores = run_oracle_pinned(shb, seed)
    # iteration 0 alone (everything before the refit), untimed: the refit's BIC arg-min is ill-conditioned
    # on samples with a handful of distinct delays (millisecond clocks; tests/gmm_conditioning.py), so the
    # final comparison can differ there for reasons of summation order while iteration 0 must not
    pass0 = None
    if gpu_assign_pass0 is not None:
        from oracle import tw_oracle
        ob = tw_oracle.OracleBatch(shb)
        g0 = ob.params_pass0()
        pass0 = ob.stitch(ob.score(gauss=g0)["cut"], gauss=g0, want_topk=False)["assign"]
    same, same0, pos, cum = True, True, 0, 0
    for b, s in zip(blocks, sample):
        S, n = b.in_start.shape
        E = len(b.out_start)
        k = s.in_start.shape[0]
        same = same and bool(np.array_equal(gpu_assign[cum:cum + k * n * E], res["assign"][pos:pos + k * n * E]))
        if pass0 is not None:
            same0 = same0 and bool(np.array_equal(gpu_assign_pass0[cum:cum + k * n * E], pass0[pos:pos + k * n * E]))
        cum += S * n * E
        pos += k * n * E
    # When the final assignments differ although iteration 0 agrees, the refit chose another component
    # count somewhere (ill-conditioned BIC arg-min).  Show that nothing else differs: the engine's second
    # pass run with the ORACLE's refitted mixtures must reproduce the oracle's final assignments.
    same_given_refit = None
    if not same and dev_index is not None:
        try:
            import torch
            from traceweaver_b200.engine import Engine
            eng = Engine(dev_index)
            eng.bind(shb)
            eng.prepare()
            p0 = eng.params_pass0()
            sc = eng.score(p0, want_used=True)
            eng.stitch(p0, sc["cut"], undeleted=sc)
            p1 = eng.params_from_host(mix=res["mix"])
            top = eng.score(p1, out=dict(used_lo=sc["used_lo"], used_bits=sc["used_bits"], used_wide=sc["used_wide"],
                                         cut=sc["cut"]), keep_windows=True)
            r1 = eng.stitch(p1, sc["cut"], undeleted=top)
            eng.status()
            same_given_refit = bool(np.array_equal(r1["assign"].cpu().numpy(), res["assign"]))
            eng.close()
        except Exception as ex:
            same_given_refit = repr(ex)[:120]
    return {"value": n_spans / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"first {per} services of each of the {len(blocks)} blocks ({shb.n_problems} services, "
                      f"{n_spans} spans), {dt:.1f} s wall, one pinned thread per physical core",
            "engine_equals_oracle_on_sample": same,
            "engine_equals_oracle_iteration0_on_sample": same0 if pass0 is not None else None,
            "engine_equals_oracle_given_the_oracle_refit": same_given_refit}


def measure(args, blocks, hb, dev_index, steps, warmup, gather=None, rank=0, world=1, want_cpu=True,
            clock=False, cpu_sample=None, want_outputs=False):
    """All legs for one service list on this rank.  Returns a dict of raw measurements (and, with
    want_outputs, the host copy of what the last timed step returned)."""
    import torch
    import torch.distributed as dist
    from traceweaver_b200 import synth
    from traceweaver_b200.engine import Engine
    from traceweaver_b200.predictor import solve_bound
    from traceweaver_b200.api import BatchSolver

    dev = torch.device("cuda", dev_index)
    n_spans = synth.span_count(blocks)
    truth = torch.from_numpy(synth.truth_assign(blocks)).to(dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def step(eng):
        res = solve_bound(eng, seed_select=args.seed)
        if gather is not None:
            res["gathered"] = gather(res["assign"], rank)       # the data path's one collective
        return res

    # ---- leg 1: inputs resident in HBM
    eng = Engine(dev_index)
    eng.bind(hb)
    for _ in range(warmup):
        res = step(eng)
    barrier()
    l0 = eng.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(dev_index).start() if clock else None
    ev0.record()
    for _ in range(steps):
        res = step(eng)
    ev1.record()
    barrier()
    if sampler:
        sampler.finish()
    resident_ms = max_over_ranks(ev0.elapsed_time(ev1))
    launches = eng.launch_count() - l0
    outputs = host_outputs(res) if want_outputs else None
    acc = accuracy(eng, res["assign"], truth, hb)
    unassigned = int(res["counters"][:, 1].sum().item())
    gather_ok = None
    if gather is not None:
        mine = gather.shards(res["gathered"])[rank]
        gather_ok = bool(torch.equal(mine, res["assign"]))
    assign_pass0 = res["assign_pass0"].cpu().numpy() if (want_cpu and rank == 0 and world == 1) else None

    # ---- roofline of the scoring kernel (GMM pass: the final top-K lists), CUDA events on our stream
    p1 = res["params_pass1"]
    reps = 5
    top = eng.score(p1, out=dict(cut=res["cut"]), keep_windows=True)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        eng.score(p1, out=top, keep_windows=True)
    b.record()
    torch.cuda.synchronize()
    score_ms = a.elapsed_time(b) / reps
    E_of = np.diff(hb.prob_ep_off).astype(np.int64)
    n_of = np.diff(hb.prob_in_off).astype(np.int64)
    alg_bytes = int(np.sum(n_of * (16 * (1 + E_of) + 5 * (8 + 4 * E_of))))     # SURVEY.md §8(d)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = alg_bytes / (score_ms * 1e-3) / 1e9
    traffic = None
    try:
        per = json.load(open(os.path.join(ROOT, "profiles", "score_traffic.json"))).get("dram_bytes_per_in_span")
        traffic = int(per * int(n_of.sum())) if per else None   # ncu capture scaled to this launch's in-spans
    except Exception:
        pass
    roofline = {"kernel": "k_score3<E> (one launch per E present; + sequential redo of flagged tiles): GMM pass, "
                          "final top-K", "bound": "hbm",
                "achieved": round(achieved, 2), "peak": peak,
                "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback 6650 GB/s",
                "unit": "GB/s", "frac": round(achieved / peak, 5), "traffic": traffic,
                "algorithmic_bytes_per_launch": alg_bytes, "launch_ms": round(score_ms, 4),
                "tiles_redone_sequentially": eng.redo_tile_count(), "tiles": eng.tile_count()}
    # ---- FP64 roofline of the refit (27 ms of the step is here): the EM sweeps of k_gmm_bic<K> / k_gmm_final<K>
    # count their sample-component evaluations (tw_gmm_work); one evaluation is 27 FP64 instructions in
    # scikit-learn's unfused operation order, 10 of them FMAs (DESIGN.md §4) = 37 flops; the peak is this
    # device's measured DFMA rate (tw_measure_fp64_peak, builder-measured, not in MEASURED_PEAKS.json)
    roofline_refit = None
    try:
        dly, cnt = eng.delays(res["assign_pass0"])
        eng.gmm_refit(dly, cnt, seed_select=args.seed)
        eng.gmm_work(reset=True)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        eng.gmm_refit(dly, cnt, seed_select=args.seed)
        b.record()
        torch.cuda.synchronize()
        refit_ms = a.elapsed_time(b)
        evals = eng.gmm_work(reset=True)
        peak_tf = eng.fp64_peak_tflops()
        ach_tf = evals * 37.0 / (refit_ms * 1e-3) / 1e12
        roofline_refit = {"kernel": "refit: EM sweeps of k_gmm_bic<1..5> + k_gmm_final<K> (whole tw_gmm_refit time as the "
                                    "denominator, k-means seeding / Lloyd kernels included)",
                          "bound": "fp64", "achieved": round(ach_tf, 3), "peak": round(peak_tf, 2),
                          "peak_source": "tw_measure_fp64_peak (builder-measured DFMA rate of this device)",
                          "unit": "TFLOP/s", "frac": round(ach_tf / peak_tf, 4),
                          "fp64_issue_frac": round(evals * 27.0 / (refit_ms * 1e-3) / (peak_tf * 1e12 / 2.0), 4),
                          "em_sample_component_evaluations": int(evals), "flops_per_evaluation": 37,
                          "fp64_instructions_per_evaluation": 27, "refit_ms": round(refit_ms, 3)}
    except Exception as ex:       # a measurement aid must not take the line down
        roofline_refit = {"error": repr(ex)[:200]}
    eng.close()

    # ---- leg 2: end to end through the public batch API, host buffers in and out.  The caller's
    # arrays are rewritten in place before every step (time shift: same problem, new bytes).
    solver = BatchSolver(device=dev_index, seed_select=args.seed)
    for _ in range(max(warmup, 1)):
        out = solver.solve(hb)
    barrier()
    e2e_ms_sum = 0.0
    span_arrays = ("in_start", "in_end", "out_start", "out_end")
    for k in range(steps):
        for name in span_arrays:
            hb.arrays[name] += 1                      # untimed: the caller refills its buffers
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        out = solver.solve(hb)
        if gather is not None:
            gather(torch.from_numpy(out["assign"]).to(dev, non_blocking=True), rank)
        e1.record()
        barrier()
        e2e_ms_sum += max_over_ranks(e0.elapsed_time(e1))
    e2e = {"ms": e2e_ms_sum, "h2d": solver.h2d_bytes, "d2h": solver.d2h_bytes, "chunks": solver.last_chunks}
    gpu_assign = np.array(out["assign"])
    for name in span_arrays:
        hb.arrays[name] -= steps
    solver.close()

    cpu = None
    if want_cpu and rank == 0 and world == 1:
        cpu = cpu_baseline(blocks, gpu_assign, cpu_sample or args.cpu_sample, args.seed, assign_pass0, dev_index)
    return dict(n_spans=n_spans, resident_ms=resident_ms, launches=launches, accuracy=acc, unassigned=unassigned,
                roofline=roofline, roofline_refit=roofline_refit, e2e=e2e, cpu=cpu, gather_ok=gather_ok,
                clocks=sampler.summary() if sampler else None, outputs=outputs)


def shipped_directories(dev_index):
    """BASELINE configs[1]/[2] as shipped: the service problems of the reference's Jaeger directories
    (tests/golden holds the arrays the reference's loader produced), each directory solved as one
    batch through the public API, compared with the reference's own assignments."""
    import glob
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from golden_util import Golden, GOLDEN_DIR
    from traceweaver_b200 import refit
    from traceweaver_b200.api import BatchSolver
    from traceweaver_b200.batch import build_batch
    files = sorted(glob.glob(os.path.join(GOLDEN_DIR, "*__*.npz")))
    if not files:
        return None
    by_dir = {}
    for f in files:
        by_dir.setdefault(os.path.basename(f).split("__")[0], []).append(Golden(f))
    solver = BatchSolver(device=dev_index, seed_select=10)
    rows, tot_spans, tot_ms, equal_all, ref_s, differing = [], 0, 0.0, True, 0.0, []
    for name, gs in sorted(by_dir.items()):
        probs = [g.problem() for g in gs]
        hb = build_batch(probs)
        spans = int(sum(p.n_in + sum(len(o) for o in p.out_start) for p in probs))
        # the reference's refit draws from NumPy's global stream: per service the fits on the TRUE
        # assignments come first and the terms are visited in the caller's ep order
        # (traceweaver_v3.py:796-818); both only move the k-means++ starting points, and both are
        # inputs of the reference's call (true_assignments, the order of out_span_partitions)
        truth = np.concatenate([np.ascontiguousarray(g.z["truth"], np.int32).reshape(-1) for g in gs])
        order, t0_ = [], 0
        for g, p in zip(gs, probs):
            given_pos = [g.topo.index(ep) for ep in g.meta["out_eps_given"]]
            lo = refit.reference_term_order(p, given_pos)
            order.extend(t0_ + t for t in lo)
            t0_ += len(lo)
        order = np.asarray(order, np.int32)
        solver.solve(hb, truth_assign=truth, term_order=order)
        torch.cuda.synchronize()
        reps = 3
        t0 = time.perf_counter()
        for _ in range(reps):
            out = solver.solve(hb, truth_assign=truth, term_order=order)
        ms = (time.perf_counter() - t0) * 1e3 / reps
        equal = True
        for p, g in enumerate(gs):
            t0_, t1_ = int(hb.prob_tuple_off[p]), int(hb.prob_tuple_off[p + 1])
            ok = bool(np.array_equal(out["assign"][t0_:t1_].reshape(g.E, -1), g.z["assign"]))
            if not ok:
                differing.append(g.name)
            equal = equal and ok
        equal_all = equal_all and equal
        ref_s += sum(float(g.meta.get("reference_seconds", 0.0)) for g in gs)
        rows.append({"directory": name, "services": len(gs), "spans": spans, "ms": round(ms, 3),
                     "assignments_equal_reference": equal})
        tot_spans += spans
        tot_ms += ms
    solver.close()
    return {"workload": "shipped Jaeger directories (hotel / media / nodejs problems as the reference's loader built "
                        "them), one directory per call through BatchSolver, wall clock incl. staging, H2D and D2H",
            "directories": len(rows), "spans": tot_spans, "ms_total": round(tot_ms, 2),
            "e2e_value": tot_spans / (tot_ms * 1e-3), "unit": UNIT,
            "assignments_equal_reference": equal_all, "services_differing": differing,
            "note": "nodejs services whose delay samples hold 7-15 distinct values have ill-conditioned BIC "
                    "arg-mins in scikit-learn itself (tests/gmm_conditioning.py); a service listed in "
                    "services_differing differs there, not in the engine's search",
            "reference_python_seconds_when_minted": round(ref_s, 1), "per_directory": rows}


def cache_mode_fixtures(dev_index):
    """SURVEY §8 row f-4: the services of the reference's cache-mode runs (exps/exp2: hotel `frontend` with
    --cache_rate 5..50 %, tests/golden_cache) through the skip regime of the engine (tw_skip_solve), each
    compared with the assignments the reference returned."""
    import glob
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from golden_util import Golden
    from traceweaver_b200 import skipmode
    from traceweaver_b200.engine import Engine
    files = sorted(glob.glob(os.path.join(ROOT, "tests", "golden_cache", "*__*.npz")))
    rows, equal_all, ref_s, tot_ms, tot_spans = [], True, 0.0, 0.0, 0
    eng = Engine(dev_index)
    for f in files:
        g = Golden(f)
        if not any(v != 0 for v in g.meta["skip_budget"].values()):
            continue
        prob = g.problem()
        labels = [g.meta["in_ep"]] + g.topo
        wins = [tuple(w) for w in g.meta["time_windows_before"]]

        def once():
            st = skipmode.SkipState()
            st.time_windows = list(wins)
            return skipmode.solve(eng, prob.in_start, prob.in_end, prob.out_start, prob.out_end, prob.preds,
                                  labels=labels, state=st, want_topk=False)
        once()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = once()
        ms = (time.perf_counter() - t0) * 1e3
        ok = bool(np.array_equal(res["assign"], g.z["assign"]))
        equal_all = equal_all and ok
        spans = int(prob.n_in + sum(len(o) for o in prob.out_start))
        rows.append({"fixture": os.path.basename(f)[:-4], "spans": spans, "ms": round(ms, 2),
                     "skip_assignments": int((res["assign"] == -2).sum()), "assignments_equal_reference": ok,
                     "reference_python_seconds": round(float(g.meta.get("reference_seconds", 0.0)), 1)})
        ref_s += float(g.meta.get("reference_seconds", 0.0))
        tot_ms += ms
        tot_spans += spans
    eng.close()
    if not rows:
        return None
    return {"workload": "cache-mode services (skip budgets, exps/exp2 shape): hotel `frontend` fixtures minted from the "
                        "reference with --cache_rate, one service per call through skipmode.solve (host arrays in and out)",
            "services": len(rows), "spans": tot_spans, "ms_total": round(tot_ms, 2),
            "e2e_value": tot_spans / (tot_ms * 1e-3), "unit": UNIT, "assignments_equal_reference": equal_all,
            "reference_python_seconds_when_minted": round(ref_s, 1), "per_service": rows}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from traceweaver_b200 import shard
    from traceweaver_b200.batch import build_batch_from_blocks

    rank, local_rank, world = dist_env()
    torch.cuda.set_device(local_rank)
    # torchrun exports OMP_NUM_THREADS=1; the end-to-end leg copies ~0.5 GB of caller arrays into pinned
    # staging on the host every step, which torch does with its intra-op threads: give every rank its share
    try:
        torch.set_num_threads(max(1, len(physical_cores()) // max(world, 1)))
    except RuntimeError:
        pass
    if world > 1:
        # stdout carries the one JSON line only: NCCL prints its version banner with printf when the
        # first communicator is created, so stdout points at stderr until that has happened
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            warm = torch.zeros(1, device=torch.device("cuda", local_rank))
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    dev = torch.device("cuda", local_rank)

    # ---- ONE global service list, partitioned by span count; this rank generates only its slice
    if args.scaling == "weak":
        n_services = args.services * world
    else:
        probe = shard.stream_spec(args.workload, 1200, args.n_in, args.seed)
        n_services = int(round(args.spans / shard.spec_span_counts(probe).mean()))
    specs = shard.stream_spec(args.workload, n_services, args.n_in, args.seed)
    span_counts = shard.spec_span_counts(specs)
    bounds = shard.partition_by_spans(span_counts, world)
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    blocks = shard.generate_slice(specs, lo, hi)
    hb = build_batch_from_blocks(blocks)
    total_spans = int(span_counts.sum())
    gather = shard.AssignGather(shard.spec_tuple_counts(specs), bounds, dev) if world > 1 else None

    m = measure(args, blocks, hb, local_rank, args.steps, args.warmup, gather=gather, rank=rank, world=world,
                clock=True, want_outputs=rank == 0 and args.dump_outputs is not None)
    if m["outputs"] is not None:
        dump_outputs(args.dump_outputs, m["outputs"], hb)

    extra = []
    if rank == 0 and world == 1 and not args.no_extra:
        # the other BASELINE shapes: smaller lists and fewer steps so the default run stays within minutes
        for wl, ns, n_in in (("media", 2046, 1000), ("alibaba", 2016, 1250)):
            if wl == args.workload:
                continue
            try:
                sp = shard.stream_spec(wl, ns, n_in, args.seed)
                bl = shard.generate_slice(sp, 0, ns)
                h2 = build_batch_from_blocks(bl)
                r = measure(args, bl, h2, local_rank, 3, 3, want_cpu=True, cpu_sample=108)
                extra.append({"workload": WORKLOAD_TEXT[wl], "services": h2.n_problems, "spans": r["n_spans"],
                              "value": r["n_spans"] * 3 / (r["resident_ms"] * 1e-3), "unit": UNIT,
                              "ms_per_step": r["resident_ms"] / 3,
                              "e2e_value": r["n_spans"] * 3 / (r["e2e"]["ms"] * 1e-3),
                              "accuracy": r["accuracy"], "unassigned": r["unassigned"], "roofline": r["roofline"],
                              "cpu_baseline": r["cpu"],
                              "engine_equals_oracle_on_sample": r["cpu"]["engine_equals_oracle_on_sample"],
                              "engine_equals_oracle_iteration0_on_sample":
                                  r["cpu"]["engine_equals_oracle_iteration0_on_sample"],
                              "engine_equals_oracle_given_the_oracle_refit":
                                  r["cpu"]["engine_equals_oracle_given_the_oracle_refit"]})
            except Exception as ex:       # an extra leg must not take the headline line down with it
                extra.append({"workload": WORKLOAD_TEXT[wl], "error": repr(ex)[:300]})
        try:
            sd = shipped_directories(local_rank)
            if sd:
                extra.append(sd)
        except Exception as ex:
            extra.append({"workload": "shipped Jaeger directories", "error": repr(ex)[:300]})
        try:
            cm = cache_mode_fixtures(local_rank)
            if cm:
                extra.append(cm)
        except Exception as ex:
            extra.append({"workload": "cache-mode services", "error": repr(ex)[:300]})

    if rank == 0:
        K = args.steps
        sharding = (f"one list of {n_services} services partitioned by span count over {world} rank(s); "
                    + ("one NCCL all_gather_into_tensor of the assignment arrays per step, inside the timed region"
                       if world > 1 else "single rank: no collective"))
        cfg = {"workload": WORKLOAD_TEXT[args.workload], "services_total": int(n_services),
               "services_this_rank": int(hb.n_problems), "in_spans_per_service": args.n_in,
               "spans_total": total_spans, "sharding": sharding,
               "l2": "inputs+outputs per step (>1 GB) exceed the 126 MB L2; no explicit flush",
               "passes": 2, "refit": "device GMM (BIC over 1..5 components) between passes"}
        line = {
            "metric": METRIC, "value": total_spans * K / (m["resident_ms"] * 1e-3), "unit": UNIT,
            "n_gpus": world, "steps": K, "warmup": args.warmup,
            "ms_per_step": m["resident_ms"] / K, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "int64 timestamps, f64 log-likelihoods", "data": "synthetic",
            "config": cfg,
            "accuracy": {"assignment_accuracy": m["accuracy"], "unassigned": m["unassigned"],
                         "note": "fraction of incoming spans with all children correct vs generator ground truth "
                                 "(rank 0's services)"},
            "e2e": {"value": total_spans * K / (m["e2e"]["ms"] * 1e-3), "unit": UNIT,
                    "ms_per_step": m["e2e"]["ms"] / K,
                    "h2d_bytes_per_step": m["e2e"]["h2d"], "d2h_bytes_per_step": m["e2e"]["d2h"],
                    "api": "traceweaver_b200.api.BatchSolver.solve(host batch) -> host arrays",
                    "host_staging": "caller arrays rewritten in place before every step; solve() memcpys them into "
                                    "pinned staging every call (inside the timed region)",
                    "overlap": f"{m['e2e']['chunks']} service groups round-robin on 2 streams (copies overlap kernels)"},
            "gpu_launches": int(m["launches"]),
            "collective": None if gather is None else {
                "op": "all_gather_into_tensor(int32 assign)",
                "bytes_received_per_rank_per_step": gather.bytes_received_per_rank,
                "own_shard_round_trips": m["gather_ok"]},
            "clocks": m["clocks"], "roofline": m["roofline"], "roofline_refit": m["roofline_refit"],
            "cpu_baseline": m["cpu"], "impl": "ours",
            "extra_workloads": extra,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_reference(args):
    """CPU arm: the reference's algorithm (oracle/ C port; the Python reference cannot travel to the
    GPU box and needs Gurobi), one pinned thread per physical core, each step = a bounded sample of
    the workload sized for seconds of CPU work.  The sample holds max(--cpu-sample, 24 x physical cores)
    services so that every core has work: its inputs, and so its --dump-outputs files, repeat exactly on
    the same host but differ between hosts with different core counts."""
    rank, _, world = dist_env()
    if rank != 0:
        return
    from oracle import tw_oracle
    from traceweaver_b200 import shard, synth
    from traceweaver_b200.batch import build_batch_from_blocks
    tw_oracle.build()
    cores = len(physical_cores())
    n_services = max(args.cpu_sample, 24 * cores)
    specs = shard.stream_spec(args.workload, n_services, args.n_in, args.seed, block_services=max(1, n_services // 12))
    blocks = shard.generate_slice(specs, 0, n_services)
    hb = build_batch_from_blocks(blocks)
    n_spans = synth.span_count(blocks)
    for _ in range(min(args.warmup, 1)):
        run_oracle_pinned(hb, args.seed)
    dt = 0.0
    for _ in range(args.steps):
        res, t, _ = run_oracle_pinned(hb, args.seed)
        dt += t
    if args.dump_outputs is not None:
        dump_outputs(args.dump_outputs, res, hb)
    v = n_spans * args.steps / dt
    sample = f"{hb.n_problems} services ({n_spans} spans) per step on {cores} pinned threads (one per physical core)"
    cfg = {"workload": WORKLOAD_TEXT[args.workload], "services_total": None, "in_spans_per_service": args.n_in,
           "sample": sample, "passes": 2, "refit": "C restatement of the sklearn GMM refit between passes"}
    print(json.dumps({
        "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "int64 timestamps, f64 log-likelihoods", "data": "synthetic", "config": cfg, "impl": "reference",
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
