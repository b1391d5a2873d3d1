#!/usr/bin/env python3
"""bench.py -- tree log-likelihood evaluations/sec on B200 (BASELINE.json metric).

A "step" is one full tree log-likelihood evaluation (all nodes dirty): the BEAGLE call sequence
BeagleDataLikelihoodDelegate.calculateLikelihood issues (BDLD:812-937) --
setEigenDecomposition, setCategoryRates/Weights, setStateFrequencies, updateTransitionMatrices
(2N-2 branches), updatePartials (N-1 operations), calculateRootLogLikelihoods -- through the C ABI
of libhmsbeagle.so, with BEAST's double-buffer index flipping between steps.

  value : exactly K = --steps timed steps enqueued back to back on the instance stream (tip data / partials resident in
          HBM, result left on the device), bracketed by barrier + synchronize, CUDA-event timed on the engine's stream, max
          over ranks.  Events split the K steps into `repeats` (up to 25) consecutive windows without a synchronize between
          them, and the MEDIAN window's per-step time is reported (`block_ms_p10/p50/p90` = K x the per-step quantiles):
          a host hiccup idles the GPU inside one window only instead of becoming the result.
  --dump-outputs DIR : after the timed steps, what their last step computed, as a caller receives it: the (joint)
          log-likelihood (DIR/logL.npy) and the per-pattern site log-likelihoods (DIR/site_logL.npy; one file per rank,
          site_logL_rank<r>.npy, when N > 1), float64.  The inputs are seeded, so two builds can be compared output for output.
  e2e   : the same sequence through the synchronous reference-facing calls with HOST buffers:
          every step uploads the eigen system, rates, frequencies, branch lengths and op list and
          lands the 8-byte (joint) log-likelihood on the host; median per step, max over ranks.
  N > 1 : one process per GPU.  Weak scaling on the headline workload -- every rank owns one 10,000-pattern shard of an
          (N x 10,000)-pattern alignment (BEAST's -beagle_instances pattern split, Patterns.java:142-169); the
          per-shard log-likelihoods are summed INSIDE the root kernel over NVLink (reduce group, csrc/multi.cu: CUDA IPC
          mappings set up once; no NCCL call and no Python in the step), every rank ends with the joint value.
          value = shard evaluations/sec over all ranks = N x joint evaluations/sec (`joint_evals_per_s`).
          torch.distributed (NCCL) is plumbing only: handle exchange at set-up, barriers, max over ranks.
  strong_scaling (extra keys, every N): BASELINE configs[3] -- the 1610-taxon Makona-like alignment split N ways
          (joint evaluations/sec of ONE alignment) -- and configs[4] -- 8 gene-like partitions, 2000 taxa, dealt round-robin
          to the N GPUs, each rank one *ByPartition instance over its partitions.
  --impl reference : the CPU restatement of the reference path (oracle/beagle_cpu.c; the real
          BEAGLE-CPU is un-vendored and cannot be built here) on all host cores, rank 0 only.
"""
from __future__ import annotations

import argparse
import ctypes as Cc
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import beast_mcmc_b200  # noqa: E402,F401
from harness import evomodel as em  # noqa: E402
from harness import treedatalikelihood as tdl  # noqa: E402

WORKLOADS = {
    # BASELINE.json configs[1]: the configuration the metric is quoted on at N=1
    "gtr_g4_1000x10k": dict(taxa=1000, patterns=10000, states=4, categories=4, rootHeight=0.1, treeSeed=20240924),
    # the same with a scale buffer written by every op (SURVEY.md 8d: "also run with scaleWrite on every op")
    "gtr_g4_1000x10k_rescaled": dict(taxa=1000, patterns=10000, states=4, categories=4, rootHeight=0.1, treeSeed=20240924,
                                     scaling=True, data="gtr_g4_1000x10k"),
    # configs[2]: codon model on the dense-contraction path
    "codon_mg94_500x5k": dict(taxa=500, patterns=5000, states=61, categories=1, rootHeight=0.1, treeSeed=2),
    # amino-acid shape (20 states, G4): the tensor path's NT=3 instance, on the memory side of the roofline
    "aa20_g4_500x5k": dict(taxa=500, patterns=5000, states=20, categories=4, rootHeight=0.3, treeSeed=4),
    "codon_mg94_500x5k_g4": dict(taxa=500, patterns=5000, states=61, categories=4, rootHeight=0.1, treeSeed=2),
    # configs[0]-like latency case (benchmark1.xml shape: 1441 taxa, 593 patterns, HKY, no gamma)
    "hky_1441x593": dict(taxa=1441, patterns=593, states=4, categories=1, rootHeight=0.1, treeSeed=1441),
    # configs[0] as shipped: the reference's own benchmark alignments (tests/golden/benchmark{1,2}_patterns.npz, extracted
    # from examples/Benchmarks/benchmark{1,2}.xml), seeded coalescent start tree as the XMLs draw a random one
    "benchmark1_xml": dict(taxa=1441, patterns=593, states=4, categories=1, rootHeight=0.05, treeSeed=666, fixture="benchmark1",
                           scaling=True),      # underflows unscaled: evaluated the way BEAST does after its first underflow
    "benchmark2_xml": dict(taxa=62, patterns=5565, states=4, categories=4, rootHeight=0.3, treeSeed=666, fixture="benchmark2"),
    # configs[3]-like: Makona-shaped synthetic (data absent from the reference tree)
    "makona_like_1610x6k": dict(taxa=1610, patterns=6000, states=4, categories=4, rootHeight=0.0025, treeSeed=3),
}
FLU8_SITES = [2341, 2341, 2233, 1778, 1565, 1413, 1027, 890]      # SURVEY.md 8d cfg 5: segment-length-like site counts

BENCH_CACHE = os.environ.get("B200_BENCH_CACHE", os.path.join(tempfile.gettempdir(), "b200_bench_cache"))

ZERO = np.zeros(1, dtype=np.int32)
MINUS1 = np.full(1, -1, dtype=np.int32)


# ------------------------------------------------------------------------------------------------
# workload
# ------------------------------------------------------------------------------------------------
def build_workload(name, shard_index, overrides):
    w = dict(WORKLOADS[name])
    w.update({k: v for k, v in overrides.items() if k in ("taxa", "patterns", "categories", "states") and v is not None})
    tree = em.Tree.coalescent(w["taxa"], w["rootHeight"], w["treeSeed"])
    if name.startswith("makona"):
        rng = np.random.default_rng(3)
        tree.branchRate = np.exp(rng.normal(0.0, 0.3, tree.nodeCount))     # relaxed clock folded into lengths
    if w["states"] == 4:
        if name.startswith("hky") or name == "benchmark1_xml":
            model = em.HKY(2.0, np.full(4, 0.25))                  # benchmark1.xml: <HKYModel> kappa 2, uniform frequencies
        elif name == "benchmark2_xml":
            model = em.GTR(1.0, 1.0, 1.0, 1.0, 1.0, 1.0, np.full(4, 0.25))   # benchmark2.xml:702-725 start values
        else:
            model = em.GTR(1.0, 4.0, 0.7, 1.2, 5.0, 1.0, np.array([0.30, 0.22, 0.24, 0.24]))
    elif w["states"] == 61:
        model = em.MG94HKYCodonModel(1.0, 0.3, 2.0)
    else:
        rng = np.random.default_rng(7)
        S = w["states"]
        model = em.SubstitutionModel(rng.uniform(0.2, 3.0, S * (S - 1) // 2), rng.dirichlet(np.full(S, 5.0)))
    site = em.GammaSiteRateModel(shape=0.5, gammaCategoryCount=w["categories"]) if w["categories"] > 1 \
        else em.GammaSiteRateModel()
    # the simulated alignment is cached outside the tree, in the temporary directory (sweeps re-use it); it is regenerated
    # when absent
    cache = os.path.join(BENCH_CACHE,
                         f"{w.get('data', name)}_{w['taxa']}_{w['patterns']}_{w['states']}_{w['categories']}_{shard_index}.npz")
    if w.get("fixture"):
        z = np.load(os.path.join(ROOT, "tests", "golden", w["fixture"] + "_patterns.npz"))
        pats = em.Patterns(z["states"].astype(np.int32), z["weights"], 4)
        assert pats.taxonCount == w["taxa"] and pats.patternCount == w["patterns"]
    elif os.path.exists(cache):
        z = np.load(cache)
        pats = em.Patterns(z["states"], z["weights"], w["states"])
    else:
        pats = em.synthetic_patterns(tree, model, site, w["patterns"], seed=1 + 1000003 * shard_index)
        try:
            os.makedirs(os.path.dirname(cache), exist_ok=True)
            np.savez(cache + f".{os.getpid()}.tmp.npz", states=pats.states, weights=pats.weights)
            os.replace(cache + f".{os.getpid()}.tmp.npz", cache)
        except OSError:
            pass
    return w, tree, pats, model, site


def _traversal(tree, traversal):
    like = tdl.TreeDataLikelihood.__new__(tdl.TreeDataLikelihood)
    like.tree, like.traversalType, like.updateNode = tree, traversal, np.ones(tree.nodeCount, dtype=bool)
    like._dispatch()
    return like.branchOperations, like.nodeOperations


class Evaluation:
    """Pre-built call arguments of one full evaluation (what the Java side hands to JNI), in the two
    buffer-index parities BEAST's BufferIndexHelper alternates between."""

    def __init__(self, tree, pats, model, site, traversal, scaling=False):
        self.tree, self.pats, self.model, self.site = tree, pats, model, site
        self.scaling = scaling
        N, n = tree.tipCount, tree.nodeCount
        self.N, self.n = N, n
        branchOps, self.nodeOps = _traversal(tree, traversal)
        self.branchNodes = np.array([b for b, _ in branchOps], dtype=np.int32)
        self.lengths = np.array([t for _, t in branchOps], dtype=np.float64)
        internal = n - N
        self.ops, self.probIdx, self.rootIdx, self.scaleIdx, self.cumIdx = [], [], [], [], []
        for parity in (0, 1):
            pidx = lambda k: k if k < N else k + parity * internal       # BufferIndexHelper.getOffsetIndex
            midx = lambda k: k + parity * n
            sidx = lambda k: (k - N) + parity * (internal + 1)           # scale buffers: BDLD:203,626-628,868-881
            ops = np.empty(len(self.nodeOps) * 7, dtype=np.int32)
            for q, (node, c1, c2) in enumerate(self.nodeOps):
                ops[7 * q: 7 * q + 7] = (pidx(node), sidx(node) if scaling else -1, -1, pidx(c1), midx(c1), pidx(c2), midx(c2))
            self.scaleIdx.append(np.array([sidx(node) for node, _, _ in self.nodeOps], dtype=np.int32))
            self.cumIdx.append(internal + parity * (internal + 1))
            self.ops.append(ops)
            self.probIdx.append((self.branchNodes + parity * n).astype(np.int32))
            self.rootIdx.append(pidx(tree.root))
        self.eig = model.getEigenDecomposition()
        # op mix for the algorithmic byte/flop count (BASELINE.md section 3)
        self.mix = {"pp": 0, "sp": 0, "ss": 0}
        for _, c1, c2 in self.nodeOps:
            k = (c1 < N) + (c2 < N)
            self.mix["pp" if k == 0 else ("sp" if k == 1 else "ss")] += 1

    def algorithmic(self, S, C, P):
        """bytes and flops of ONE updatePartials call (whole op list), SURVEY.md 8(d) figures."""
        pp, sp, ss = self.mix["pp"], self.mix["sp"], self.mix["ss"]
        byt = pp * (3 * C * P * S * 8 + 2 * C * S * S * 8) + sp * (2 * C * P * S * 8 + 4 * P + 2 * C * S * S * 8) + \
            ss * (C * P * S * 8 + 8 * P + 2 * C * S * S * 8)
        flo = pp * C * P * S * (4 * S + 1) + sp * C * P * S * (2 * S + 1) + ss * C * P * S
        return byt, flo

    def h2d_bytes(self, S, C):
        return int(self.ops[0].nbytes + self.probIdx[0].nbytes + self.lengths.nbytes +
                   (2 * S * S + S) * 8 + 2 * C * 8 + S * 8)


def create_instance(factory, ev, S, C, P, resource):
    N, n = ev.N, ev.n
    inst = factory(N, 2 * (n - N) + N, N, S, P, 2, 2 * n, C, 2 * (n - N + 1), resource, 0, 0)
    for t in range(N):
        inst.setTipStates(t, np.ascontiguousarray(ev.pats.states[t], dtype=np.int32))
    inst.setPatternWeights(np.ascontiguousarray(ev.pats.weights))
    return inst


def issue_sync(inst, ev, parity, out):
    """One evaluation through the synchronous reference-facing calls, host buffers in / host double out."""
    inst.setEigenDecomposition(parity, ev.eig.Evec, ev.eig.Ievc, ev.eig.Eval)
    inst.setCategoryRates(ev.site.getCategoryRates())
    inst.setCategoryWeights(0, ev.site.getCategoryProportions())
    inst.setStateFrequencies(0, ev.model.getFrequencies())
    inst.updateTransitionMatrices(parity, ev.probIdx[parity], None, None, ev.lengths, len(ev.lengths))
    inst.updatePartials(ev.ops[parity], len(ev.nodeOps), -1)
    cum = MINUS1
    if ev.scaling:             # BDLD:915-926
        inst.resetScaleFactors(ev.cumIdx[parity])
        inst.accumulateScaleFactors(ev.scaleIdx[parity], len(ev.nodeOps), ev.cumIdx[parity])
        cum = np.array([ev.cumIdx[parity]], dtype=np.int32)
    inst.calculateRootLogLikelihoods(np.array([ev.rootIdx[parity]], dtype=np.int32), ZERO, ZERO, cum, 1, out)
    return out[0]


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi in loop mode (-lms) for the duration of the timed regions (B200_PROFILING.md clocks line)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown," \
        "clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.gpu_index, self.proc = gpu_index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu_index), "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.15)            # let the first sample land before the timed region starts
        except OSError:
            self.proc = None

    def stop(self):
        rows = []
        if self.proc is not None:
            self.proc.terminate()
            try:
                out, _ = self.proc.communicate(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
                out, _ = self.proc.communicate()
            rows = [[c.strip() for c in line.split(",")] for line in out.splitlines() if line.count(",") >= 8]
        sm = [float(r[1]) for r in rows if r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in rows if r[2].replace(".", "").isdigit()]
        pw = [float(r[3]) for r in rows if r[3].replace(".", "").isdigit()]
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(rows)}


# ------------------------------------------------------------------------------------------------
# CPU arm (oracle port): cpu_baseline and --impl reference
# ------------------------------------------------------------------------------------------------
def cpu_pick_threads(ev, S, C, P, cores):
    """The port's thread pool does not scale to every host (shared boxes, NUMA): try a few thread counts, five
    evaluations each, and keep the one with the best MEDIAN -- the baseline gets its best configuration."""
    from oracle import cpu
    best, best_t = None, cores
    tried = []
    for th in sorted({cores, max(1, cores // 2), max(1, cores // 4), min(cores, 32), min(cores, 16), min(cores, 8)}, reverse=True):
        inst = create_instance(cpu.factory(threads=th), ev, S, C, P, None)
        out = np.zeros(1)
        issue_sync(inst, ev, 0, out)
        ts = []
        for k in range(5):
            t0 = time.perf_counter()
            issue_sync(inst, ev, (k + 1) & 1, out)
            ts.append(time.perf_counter() - t0)
        inst.finalize()
        dt = statistics.median(ts)
        tried.append((th, dt))
        if best is None or dt < best:
            best, best_t = dt, th
    return best_t, tried


def cpu_time_evaluations(ev, S, C, P, threads, min_evals, budget_s):
    from oracle import cpu                      # checker / baseline only, never the product path
    inst = create_instance(cpu.factory(threads=threads), ev, S, C, P, None)
    out = np.zeros(1)
    issue_sync(inst, ev, 0, out)                # warm-up (allocations)
    times, val = [], 0.0
    t_all = time.perf_counter()
    k = 0
    while k < min_evals or (time.perf_counter() - t_all < budget_s and k < 1000):
        t0 = time.perf_counter()
        val = issue_sync(inst, ev, (k + 1) & 1, out)
        times.append(time.perf_counter() - t0)
        k += 1
    inst.finalize()
    return times, val


def run_reference_arm(args, meta_base):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from beast_mcmc_b200 import build
    build.build_oracle()
    w, tree, pats, model, site = build_workload(args.workload, 0, vars(args))
    S, C, P = w["states"], site.getCategoryCount(), pats.patternCount
    ev = Evaluation(tree, pats, model, site, "POST_ORDER", scaling=bool(w.get("scaling")))
    cores = os.cpu_count() or 1
    from oracle import cpu
    threads, tried = cpu_pick_threads(ev, S, C, P, cores)
    inst = create_instance(cpu.factory(threads=threads), ev, S, C, P, None)
    out = np.zeros(1)
    for k in range(args.warmup):
        issue_sync(inst, ev, k & 1, out)
    per = []
    t0 = time.perf_counter()
    for k in range(args.steps):
        tc = time.perf_counter()
        issue_sync(inst, ev, k & 1, out)
        per.append(time.perf_counter() - tc)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        site_logL = np.zeros(P)
        inst.getSiteLogLikelihoods(site_logL)
        dump_outputs(args.dump_outputs, float(out[0]), site_logL, 0, 1)
    inst.finalize()
    value = 1.0 / statistics.median(per)        # median step: the same statistic as the cpu_baseline leg of the GPU arm
    line = dict(meta_base)
    line.update({
        "impl": "reference", "value": value, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * statistics.median(per), "mean_ms_per_step": 1e3 * dt / args.steps, "vs_baseline": None,
        "logL": float(out[0]),
        "cpu_baseline": {"value": value, "unit": "evals/s", "cores": threads, "kind": "port", "host_cores": cores,
                         "sample": f"{args.steps} full evaluations of the same workload, median step (oracle/beagle_cpu.c, "
                                   f"{threads} threads over pattern blocks = best median of {[t for t, _ in tried]})"},
        "e2e": {"value": value, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class Dist:
    """torch.distributed as plumbing: barriers, max over ranks, one all-gather of CUDA IPC handles at set-up."""

    def __init__(self):
        import torch
        self.torch = torch
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local_rank)
        self.device = torch.device("cuda", self.local_rank)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.device)
            self.dist = dist

    def bracket(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, values):
        values = [float(v) for v in values]
        if self.dist is None:
            return values
        t = self.torch.tensor(values, dtype=self.torch.float64, device=self.device)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t.cpu()]

    def join_reduce_group(self, lib, inst):
        """Reduce group over the ranks: every member's root kernel stores its sum into all members' slot arrays (CUDA IPC
        mappings over NVLink) and adds the others'.  The 64-byte handles are exchanged once, here."""
        if self.dist is None:
            return
        handle = (Cc.c_char * 64)()
        rc = lib.b200ExchangeCreate(inst.instance, self.rank, self.world, Cc.cast(handle, Cc.c_void_p))
        assert rc == 0, rc
        gathered = [None] * self.world
        self.dist.all_gather_object(gathered, bytes(handle.raw))
        blob = b"".join(gathered)
        buf = (Cc.c_char * len(blob)).from_buffer_copy(blob)
        rc = lib.b200ExchangeConnect(inst.instance, Cc.cast(buf, Cc.c_void_p))
        assert rc == 0, f"b200ExchangeConnect failed ({rc}): no peer path between the GPUs?"
        self.dist.barrier()

    def close(self):
        if self.dist is not None:
            self.dist.destroy_process_group()


def _quantiles(xs):
    xs = sorted(xs)
    pick = lambda f: xs[min(len(xs) - 1, int(f * len(xs)))]
    return pick(0.10), pick(0.50), pick(0.90)


def timed_blocks(D, stream, step_async, steps, warmup, windows=25):
    """Exactly `steps` timed steps after the warm-up, enqueued back to back and bracketed by barrier + synchronize.  CUDA
    events on the engine's stream split them into up to `windows` consecutive windows of (nearly) equal length; nothing
    synchronizes between windows, so the GPU never idles at a window boundary.  Per-window max over ranks, then the
    quantiles of the per-step time over the windows, scaled to the `steps`-step block."""
    torch = D.torch
    for k in range(max(3, warmup)):
        step_async(k)
    D.bracket()
    repeats = max(1, min(windows, steps))
    bounds = [steps * i // repeats for i in range(repeats + 1)]
    events = [torch.cuda.Event(enable_timing=True) for _ in range(repeats + 1)]
    t0 = time.perf_counter()
    events[0].record(stream)
    for i in range(repeats):
        for k in range(bounds[i], bounds[i + 1]):
            step_async(k)
        events[i + 1].record(stream)
    D.bracket()
    wall = time.perf_counter() - t0
    ms = D.max_over_ranks([events[i].elapsed_time(events[i + 1]) for i in range(repeats)])
    p10, p50, p90 = _quantiles([m / (bounds[i + 1] - bounds[i]) for i, m in enumerate(ms)])
    return {"repeats": repeats, "block_ms_p10": steps * p10, "block_ms_p50": steps * p50, "block_ms_p90": steps * p90,
            "timed_ms": sum(ms), "wall_ms_per_step": 1e3 * wall / steps}


def timed_e2e(D, step_e2e, steps):
    for k in range(3):
        step_e2e(k)
    D.bracket()
    per, last = [], 0.0
    for k in range(steps):
        tc = time.perf_counter()
        last = step_e2e(k)
        per.append(time.perf_counter() - tc)
    D.bracket()
    p10, p50, p90 = _quantiles(per)
    p50 = D.max_over_ranks([p50])[0]
    return {"median_s": p50, "p10_ms": 1e3 * p10, "median_ms": 1e3 * p50, "p90_ms": 1e3 * p90, "logL": float(last), "steps": steps}


def external_stream(D, strm):
    return D.torch.cuda.ExternalStream(strm.value, device=D.device)


def device_double(D, ptr, index=0):
    class _Dev:      # zero-copy torch view of the engine's device-resident result
        __cuda_array_interface__ = {"shape": (index + 1,), "typestr": "<f8", "data": (ptr, False), "version": 3}
    return D.torch.as_tensor(_Dev(), device=D.device)


def measure_single_partition(D, lib, beagle, w, tree, pats, model, site, steps, warmup, kernel_timing=True, e2e_steps=None):
    """One instance per rank over `pats` (this rank's shard), reduce group over the ranks; returns the measurements."""
    S, C, P = w["states"], site.getCategoryCount(), pats.patternCount
    scaling = bool(w.get("scaling"))
    ev = Evaluation(tree, pats, model, site, "REVERSE_LEVEL_ORDER", scaling=scaling)     # what BEAST sends a non-CPU instance
    inst = create_instance(beagle.BeagleFactory.loadBeagleInstance, ev, S, C, P, [D.local_rank + 1, 0])
    D.join_reduce_group(lib, inst)
    devp, strm = Cc.c_void_p(), Cc.c_void_p()
    out = np.zeros(1)
    first = issue_sync(inst, ev, 0, out)
    rc = lib.b200RootLogLikelihoodDevice(inst.instance, ev.rootIdx[0], 0, 0, ev.cumIdx[0] if scaling else -1,
                                         Cc.byref(devp), Cc.byref(strm))
    assert rc == 0
    stream = external_stream(D, strm)
    dres = device_double(D, devp.value)

    def step_async(k):
        p = k & 1
        # eigen system, rates and frequencies are resident (slot 0); buffers flip like BEAST's do
        inst.updateTransitionMatrices(0, ev.probIdx[p], None, None, ev.lengths, len(ev.lengths))
        inst.updatePartials(ev.ops[p], len(ev.nodeOps), -1)
        cum = -1
        if scaling:
            inst.resetScaleFactors(ev.cumIdx[p])
            inst.accumulateScaleFactors(ev.scaleIdx[p], len(ev.nodeOps), ev.cumIdx[p])
            cum = ev.cumIdx[p]
        lib.b200RootLogLikelihoodDevice(inst.instance, ev.rootIdx[p], 0, 0, cum, None, None)     # joint value stays on the device

    def step_e2e(k):
        return issue_sync(inst, ev, k & 1, out)       # host buffers up, the (joint) log-likelihood down

    res = {"ev": ev, "inst": inst, "S": S, "C": C, "P": P, "first_logL": float(first), "out": out}
    # resident eigen system for the asynchronous loop: slot 0 holds it (issue_sync above used parity 0)
    res["blocks"] = timed_blocks(D, stream, step_async, steps, warmup)
    res["joint"] = float(dres.cpu()[0])
    res["site_logL"] = np.zeros(P)
    inst.getSiteLogLikelihoods(res["site_logL"])           # the last timed step's root launch wrote them
    if kernel_timing:
        # kernel classes timed live on the engine's stream, in a block of their own (event pairs around every launch)
        D.bracket()
        inst.setKernelTiming(True)
        for k in range(steps):
            step_async(k)
        D.bracket()
        res["kernels"] = [inst.getKernelTiming(c) for c in range(3)]
        inst.setKernelTiming(False)
    res["e2e"] = timed_e2e(D, step_e2e, e2e_steps or max(steps, 100))
    res["e2e"]["c_abi_replay"] = full_evaluations_from_c(inst, ev, min(e2e_steps or max(steps, 100), 400)) if D.world == 1 else None
    return res


def replay_from_c(inst, paths, out):
    """The same 64 evaluations issued from C (harness/cdriver.c) -- the three C-ABI calls per evaluation back to back, as a
    JVM's JNI thread issues them, without the Python interpreter and ctypes marshalling between the calls."""
    import ctypes as C
    lib_file = os.path.join(os.path.dirname(os.path.abspath(__file__)), "harness", "libcdriver.so")
    if not os.path.exists(lib_file):
        return None
    drv = C.CDLL(lib_file)
    ops = np.ascontiguousarray(np.concatenate([p[0] for p in paths]), dtype=np.int32)
    opOff = np.concatenate([[0], np.cumsum([p[1] for p in paths])]).astype(np.int32)
    matOff = np.arange(len(paths) + 1, dtype=np.int32)
    probIdx = np.ascontiguousarray(np.concatenate([p[2] for p in paths]), dtype=np.int32)
    lengths = np.ascontiguousarray(np.concatenate([p[3] for p in paths]), dtype=np.float64)
    rootIdx = np.ascontiguousarray(np.concatenate([p[4] for p in paths]), dtype=np.int32)
    rounds = 12
    secs = np.zeros(rounds * len(paths))
    last = C.c_double(0.0)
    ptr = lambda a, t: a.ctypes.data_as(C.POINTER(t))
    drv.cdriver_replay.restype = C.c_int
    rc = drv.cdriver_replay(C.c_int(inst.instance), C.c_int(len(paths)), C.c_int(rounds), ptr(opOff, C.c_int), ptr(ops, C.c_int),
                            ptr(matOff, C.c_int), ptr(probIdx, C.c_int), ptr(lengths, C.c_double), ptr(rootIdx, C.c_int),
                            C.c_int(0), C.c_int(-1), ptr(secs, C.c_double), C.byref(last))
    if rc != 0:
        return {"error": rc}
    per = sorted(secs[2 * len(paths):])                        # two warm-up rounds
    expect = np.zeros(1)
    o, cnt, pidx, blen, ridx = paths[-1]
    inst.updateTransitionMatrices(0, pidx, None, None, blen, 1)
    inst.updatePartials(o, cnt, -1)
    inst.calculateRootLogLikelihoods(ridx, ZERO, ZERO, MINUS1, 1, expect)
    return {"us_per_eval": 1e6 * per[len(per) // 2], "us_p10": 1e6 * per[len(per) // 10], "us_p90": 1e6 * per[(9 * len(per)) // 10],
            "evals_per_s": 1.0 / per[len(per) // 2], "same_value_as_python_calls": bool(expect[0] == last.value),
            "what": "the same evaluations, the three C-ABI calls issued from C (harness/cdriver.c): no interpreter between calls"}


def full_evaluations_from_c(inst, ev, steps):
    """issue_sync's call sequence issued from C (harness/cdriver.c): the same host buffers go up, the same double comes down,
    but no interpreter / ctypes marshalling between the nine calls -- what a JVM's JNI thread would see."""
    import ctypes as C
    lib_file = os.path.join(os.path.dirname(os.path.abspath(__file__)), "harness", "libcdriver.so")
    if not os.path.exists(lib_file):
        return None
    drv = C.CDLL(lib_file)
    i32 = lambda a: np.ascontiguousarray(a, dtype=np.int32)
    f64 = lambda a: np.ascontiguousarray(a, dtype=np.float64)
    ops2, prob2, scale2 = i32(np.concatenate(ev.ops)), i32(np.concatenate(ev.probIdx)), i32(np.concatenate(ev.scaleIdx))
    root2, cum2 = i32(ev.rootIdx), i32(ev.cumIdx)
    evec, ievc, evl = f64(ev.eig.Evec), f64(ev.eig.Ievc), f64(ev.eig.Eval)
    rates, wts, frq = f64(ev.site.getCategoryRates()), f64(ev.site.getCategoryProportions()), f64(ev.model.getFrequencies())
    lengths = f64(ev.lengths)
    secs = np.zeros(steps + 10)
    last = C.c_double(0.0)
    pi = lambda a: a.ctypes.data_as(C.POINTER(C.c_int))
    pd = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    drv.cdriver_full_evaluations.restype = C.c_int
    rc = drv.cdriver_full_evaluations(C.c_int(inst.instance), C.c_int(steps + 10), C.c_int(len(frq)), C.c_int(len(ev.nodeOps)), pi(ops2),
                                      C.c_int(len(lengths)), pi(prob2), pd(lengths), pi(root2), pd(evec), pd(ievc), pd(evl), pd(rates),
                                      pd(wts), pd(frq), C.c_int(1 if ev.scaling else 0), pi(scale2), pi(cum2), pd(secs), C.byref(last))
    if rc != 0:
        return {"error": rc}
    per = sorted(secs[10:])
    return {"value": 1.0 / per[len(per) // 2], "unit": "evals/s", "ms_per_step": 1e3 * per[len(per) // 2],
            "p10_ms": 1e3 * per[len(per) // 10], "p90_ms": 1e3 * per[(9 * len(per)) // 10], "logL": last.value, "steps": steps,
            "what": "the same synchronous call sequence with the same host buffers, issued from C (harness/cdriver.c)"}


def incremental_section(inst, ev, tree, out, steps):
    """The evaluation MCMC mostly issues: one branch length changed -> 1 matrix, the tip-to-root path of ops, root."""
    issue_sync(inst, ev, 0, out)                       # parity-0 buffers hold the current state
    rng = np.random.default_rng(5)
    N, n, internal = ev.N, ev.n, ev.n - ev.N
    paths = []
    for _ in range(64):
        node, path = int(rng.integers(0, N)), []
        while tree.parent[node] >= 0:
            par = int(tree.parent[node])
            sib = int(tree.child[par][0]) if int(tree.child[par][1]) == node else int(tree.child[par][1])
            path.append((par, node, sib))
            node = par
        ops = np.empty(7 * len(path), dtype=np.int32)
        for q, (par, child, sib) in enumerate(path):
            cidx = child if (child < N or q == 0) else child + internal        # freshly written -> parity 1
            ops[7 * q: 7 * q + 7] = (par + internal, -1, -1, cidx, child + (n if q == 0 else 0), sib, sib)
        first = path[0][1]
        paths.append((ops, len(path), np.array([first + n], dtype=np.int32),
                      np.array([tree.branchLength(first) * 1.01]), np.array([tree.root + internal], dtype=np.int32)))

    def run_incremental(target, rounds):
        for ops, cnt, pidx, blen, rootIdx in paths[:8]:
            target.updateTransitionMatrices(0, pidx, None, None, blen, 1)
            target.updatePartials(ops, cnt, -1)
            target.calculateRootLogLikelihoods(rootIdx, ZERO, ZERO, MINUS1, 1, out)
        per = []
        for _ in range(rounds):
            for ops, cnt, pidx, blen, rootIdx in paths:
                t0 = time.perf_counter()
                target.updateTransitionMatrices(0, pidx, None, None, blen, 1)
                target.updatePartials(ops, cnt, -1)
                target.calculateRootLogLikelihoods(rootIdx, ZERO, ZERO, MINUS1, 1, out)
                per.append(time.perf_counter() - t0)
        return per

    per = run_incremental(inst, max(2, min(steps, 2000) // 64 + 1))
    inc = {"evals_per_s": 1.0 / statistics.median(per), "us_per_eval": 1e6 * statistics.median(per),
           "us_p10": 1e6 * _quantiles(per)[0], "us_p90": 1e6 * _quantiles(per)[2],
           "mean_ops_per_eval": float(np.mean([c for _, c, _, _, _ in paths])),
           "c_abi_replay": replay_from_c(inst, paths, out),
           "what": "one branch length changed: 1 matrix, tip-to-root path of partials ops, root; host buffers, synchronous; "
                   "64 different paths in rotation (no plan-cache hits beyond the cache size); median"}
    return inc, run_incremental


def cold_plan_section(inst, ev, out, steps):
    """Full evaluations whose operation list changes EVERY step (what topology moves do to the plan cache): one run of
    mutually independent ops of the reverse-level-order list is rotated differently each time -> never a cache hit,
    never a graph replay; the result is unchanged (asserted)."""
    rng = np.random.default_rng(11)
    base = ev.ops[0].reshape(-1, 7)
    issue_sync(inst, ev, 0, out)
    want = out[0]
    per = []
    for k in range(min(steps, 200)):
        order = np.arange(len(base))
        i = int(rng.integers(0, len(base) - 2))
        run, dests = [i], {int(base[i][0])}
        j = i + 1
        while j < len(base) and int(base[j][3]) not in dests and int(base[j][5]) not in dests:
            run.append(j)
            dests.add(int(base[j][0]))
            j += 1
        if len(run) > 1:
            order[run] = np.roll(order[run], 1 + k % (len(run) - 1))
        ops = np.ascontiguousarray(base[order]).reshape(-1)
        t0 = time.perf_counter()
        inst.updateTransitionMatrices(0, ev.probIdx[0], None, None, ev.lengths, len(ev.lengths))
        inst.updatePartials(ops, len(ev.nodeOps), -1)
        inst.calculateRootLogLikelihoods(np.array([ev.rootIdx[0]], dtype=np.int32), ZERO, ZERO, MINUS1, 1, out)
        per.append(time.perf_counter() - t0)
        assert abs(out[0] - want) <= 1e-12 * abs(want)
    return {"evals_per_s": 1.0 / statistics.median(per), "ms_per_eval": 1e3 * statistics.median(per),
            "what": "full evaluation with a DIFFERENT operation order every step (plan-cache miss each time: validation, "
                    "planning, H2D of the records; no graph replay); host buffers, synchronous; median"}


def strong_makona(D, lib, beagle, steps, warmup):
    """BASELINE configs[3]: ONE 1610-taxon alignment, its 6000 patterns split over the N GPUs by BEAST's block rule."""
    w, tree, pats, model, site = build_workload("makona_like_1610x6k", 0, {})
    w = dict(w, scaling=True)                      # deep tree: evaluated rescaled, the way BEAST does after its first underflow
    shard = pats.subSet(D.rank, D.world) if D.world > 1 else pats
    r = measure_single_partition(D, lib, beagle, w, tree, shard, model, site, steps, warmup, kernel_timing=True,
                                 e2e_steps=max(steps, 100))
    b = r["blocks"]
    ms = b["block_ms_p50"] / steps
    k_ms = r["kernels"][0][0] / steps
    r["inst"].finalize()
    return {"workload": "makona_like_1610x6k split into %d contiguous pattern blocks (Patterns.java:142-169), rescaled" % D.world,
            "patterns_per_gpu": shard.patternCount, "joint_evals_per_s": 1e3 / ms, "ms_per_step": ms,
            "e2e_joint_evals_per_s": 1.0 / r["e2e"]["median_s"], "e2e_ms_per_step": r["e2e"]["median_ms"],
            "partials_ms_per_step_rank0": k_ms, "repeats": b["repeats"], "block_ms_p10": b["block_ms_p10"],
            "block_ms_p90": b["block_ms_p90"], "logL": r["joint"], "steps": steps}


def flu8_partitions():
    tree = em.Tree.coalescent(2000, 0.05, 5)
    parts, models, sites = [], [], []
    cache = os.path.join(BENCH_CACHE, "flu8_2000.npz")
    z = np.load(cache, allow_pickle=False) if os.path.exists(cache) else None
    for k, ns in enumerate(FLU8_SITES):
        rng = np.random.default_rng(10 + k)
        model = em.GTR(*rng.uniform(0.5, 4.0, 6), rng.dirichlet(np.full(4, 20.0)))
        site = em.GammaSiteRateModel(shape=float(rng.uniform(0.3, 1.0)), gammaCategoryCount=4)
        if z is not None:
            parts.append(em.Patterns(z[f"s{k}"], z[f"w{k}"], 4))
        else:
            parts.append(em.Patterns.fromAlignment(em.simulate_alignment(tree, model, site, ns, 100 + k)))
        models.append(model)
        sites.append(site)
    if z is None:
        try:
            os.makedirs(os.path.dirname(cache), exist_ok=True)
            tmp = cache + f".{os.getpid()}.tmp.npz"
            np.savez(tmp, **{f"s{k}": p.states for k, p in enumerate(parts)}, **{f"w{k}": p.weights for k, p in enumerate(parts)})
            os.replace(tmp, cache)
        except OSError:
            pass
    return tree, parts, models, sites


def strong_flu8(D, lib, beagle, steps, warmup):
    """BASELINE configs[4]: 8 gene-like partitions on a shared 2000-taxon tree, GTR+G4 each, dealt round-robin to the N
    GPUs; every rank holds ONE instance and drives its partitions through the *ByPartition calls (the route BEAST's
    MultiPartitionDataLikelihoodDelegate takes), the ranks' totals meet in the reduce group."""
    tree, parts, models, sites = flu8_partitions()
    mine = [k for k in range(len(parts)) if k % D.world == D.rank]
    K = len(mine)
    N, n = tree.tipCount, tree.nodeCount
    counts = [parts[k].patternCount for k in mine]
    P = int(sum(counts))
    branches, nodeOps = _traversal(tree, "REVERSE_LEVEL_ORDER")
    b = beagle.BeagleFactory.loadBeagleInstance(N, n, N, 4, P, K, K * n, 4, 1, [D.local_rank + 1, 0], 0, 0)
    states = np.concatenate([parts[k].states for k in mine], axis=1)
    for t in range(N):
        b.setTipStates(t, np.ascontiguousarray(states[t], dtype=np.int32))
    b.setPatternWeights(np.concatenate([parts[k].weights for k in mine]))
    b.setPatternPartitions(K, np.repeat(np.arange(K, dtype=np.int32), counts))
    D.join_reduce_group(lib, b)
    eig, rate, prob, lens = [], [], [], []
    for q, k in enumerate(mine):
        e = models[k].getEigenDecomposition()
        b.setEigenDecomposition(q, e.Evec, e.Ievc, e.Eval)
        b.setCategoryRatesWithIndex(q, sites[k].getCategoryRates())
        b.setCategoryWeights(q, sites[k].getCategoryProportions())
        b.setStateFrequencies(q, models[k].getFrequencies())
        for node, t in branches:
            eig.append(q); rate.append(q); prob.append(node + q * n); lens.append(t)
    eig, rate, prob = (np.array(x, dtype=np.int32) for x in (eig, rate, prob))
    lens = np.array(lens)
    ops = np.array([v for node, c1, c2 in nodeOps for q in range(K)
                    for v in (node, -1, -1, c1, c1 + q * n, c2, c2 + q * n, q, -1)], dtype=np.int32)
    root = np.full(K, tree.root, dtype=np.int32)
    idx = np.arange(K, dtype=np.int32)
    none = np.full(K, -1, dtype=np.int32)
    byPart, total = np.zeros(K), np.zeros(1)
    ip = lambda a: a.ctypes.data_as(Cc.POINTER(Cc.c_int))
    devp, strm = Cc.c_void_p(), Cc.c_void_p()

    def step_async(k):
        b.updateTransitionMatricesWithMultipleModels(eig, rate, prob, None, None, lens, len(lens))
        b.updatePartialsByPartition(ops, len(ops) // 9)
        rc = lib.b200RootLogLikelihoodsByPartitionDevice(b.instance, ip(root), ip(idx), ip(idx), ip(none), ip(idx), K,
                                                         Cc.byref(devp), Cc.byref(strm))
        assert rc == 0, rc

    def step_e2e(k):
        b.updateTransitionMatricesWithMultipleModels(eig, rate, prob, None, None, lens, len(lens))
        b.updatePartialsByPartition(ops, len(ops) // 9)
        b.calculateRootLogLikelihoodsByPartition(root, idx, idx, none, idx, K, 1, byPart, total)
        return total[0]

    step_async(0)
    stream = external_stream(D, strm)
    blocks = timed_blocks(D, stream, step_async, steps, warmup)
    e2e = timed_e2e(D, step_e2e, max(steps, 50))
    ms = blocks["block_ms_p50"] / steps
    b.finalize()
    return {"workload": "flu8_like: 8 partitions (%s sites), 2000 taxa, GTR+G4 each, partition k on GPU k mod %d, one "
                        "*ByPartition instance per GPU" % ("/".join(map(str, FLU8_SITES)), D.world),
            "patterns_rank0": counts, "partitions_per_gpu": K, "joint_evals_per_s": 1e3 / ms, "ms_per_step": ms,
            "e2e_joint_evals_per_s": 1.0 / e2e["median_s"], "e2e_ms_per_step": e2e["median_ms"],
            "repeats": blocks["repeats"], "block_ms_p10": blocks["block_ms_p10"], "block_ms_p90": blocks["block_ms_p90"],
            "logL": e2e["logL"], "steps": steps}


MAX_DUMP_BYTES = 64 << 20


def dump_outputs(path, logL, site_logL, rank, world):
    """Writes the last timed step's results: DIR/logL.npy (rank 0: the joint log-likelihood) and this rank's site
    log-likelihoods.  Past its share of MAX_DUMP_BYTES a rank writes a fixed seeded sample of its patterns (sorted)."""
    os.makedirs(path, exist_ok=True)
    if rank == 0:
        np.save(os.path.join(path, "logL.npy"), np.array([logL], dtype=np.float64))
    keep = (MAX_DUMP_BYTES // world - 4096) // 8
    if site_logL.size > keep:
        site_logL = site_logL[np.sort(np.random.default_rng(12345).choice(site_logL.size, keep, replace=False))]
    name = "site_logL.npy" if world == 1 else f"site_logL_rank{rank}.npy"
    np.save(os.path.join(path, name), np.ascontiguousarray(site_logL, dtype=np.float64))


def load_json(path):
    try:
        return json.load(open(path))
    except (OSError, ValueError):
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="gtr_g4_1000x10k", choices=list(WORKLOADS))
    ap.add_argument("--taxa", type=int)
    ap.add_argument("--patterns", type=int)
    ap.add_argument("--categories", type=int)
    ap.add_argument("--states", type=int)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the strong-scaling / incremental / cold-plan sections")
    ap.add_argument("--cpu-budget", type=float, default=12.0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's log-likelihood and site "
                                                          "log-likelihoods to DIR/*.npy")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3

    world = int(os.environ.get("WORLD_SIZE", "1"))
    w0 = dict(WORKLOADS[args.workload])
    w0.update({k: v for k, v in vars(args).items() if k in w0 and v is not None})
    meta_base = {
        "metric": "tree log-likelihood evals/sec", "unit": "evals/s", "higher_is_better": True,
        "scaling": "weak", "dtype": "f64", "data": "synthetic",
        "config": {"workload": args.workload, "taxa": w0["taxa"], "patterns_per_gpu": w0["patterns"],
                   "states": w0["states"], "categories": w0["categories"],
                   "step": "full evaluation, all nodes dirty: eigen+rates+freqs upload, 2N-2 matrices, N-1 partials ops, root",
                   "sharding": f"{world} x {w0['patterns']}-pattern shards, one per GPU; per-shard sums added inside the root "
                               "kernel over NVLink (reduce group), no NCCL call in the step",
                   "l2": "inputs larger than L2: each step writes N-1 partials buffers (1.28 GB at the default "
                         "workload) into the alternate buffer parity"},
    }
    if args.impl == "reference":
        run_reference_arm(args, meta_base)
        return

    from beast_mcmc_b200 import beagle
    D = Dist()
    lib = beagle.load_library()
    rank = D.rank
    custom = any(getattr(args, k) is not None for k in ("taxa", "patterns", "categories", "states"))

    w, tree, pats, model, site = build_workload(args.workload, rank, vars(args))
    sampler = ClockSampler(D.local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    r = measure_single_partition(D, lib, beagle, w, tree, pats, model, site, args.steps, args.warmup)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, r["joint"], r["site_logL"], rank, world)
    ev, inst, S, C, P, out = r["ev"], r["inst"], r["S"], r["C"], r["P"], r["out"]
    scaling = bool(w.get("scaling"))

    inc = cold = run_incremental = None
    if world == 1 and not scaling and not args.no_extras:
        inc, run_incremental = incremental_section(inst, ev, tree, out, args.steps)
        cold = cold_plan_section(inst, ev, out, args.steps)
    inst.finalize()

    strong = None
    if not args.no_extras and not custom and args.workload == "gtr_g4_1000x10k":
        ssteps = max(20, min(args.steps, 200))
        strong = {"what": "ONE alignment / ONE partitioned data set over the N GPUs of this run (joint evaluations per "
                          "second; compare across the driver's N = 1, 2, 4, 8 lines)",
                  "n_gpus": world,
                  "makona_like_1610x6k": strong_makona(D, lib, beagle, ssteps, args.warmup),
                  "flu8_2000": strong_flu8(D, lib, beagle, max(20, ssteps // 2), args.warmup)}

    if rank != 0:
        D.close()
        return

    blocks = r["blocks"]
    dev_ms = blocks["block_ms_p50"]
    value = world * args.steps / (dev_ms * 1e-3)
    byt, flo = ev.algorithmic(S, C, P)
    (k_ms, k_n), (m_ms, m_n), (r_ms, r_n) = r["kernels"]
    k_avg_ms = k_ms / args.steps
    peaks = load_json(os.path.join(ROOT, "MEASURED_PEAKS.json"))
    fp64 = load_json(os.path.join(ROOT, "profiles", "r02_fp64_peaks.json"))
    traffic_tab = load_json(os.path.join(ROOT, "profiles", "r02_traffic.json")) or {}
    tj = None if custom else traffic_tab.get(args.workload)
    traffic = (tj["dram_bytes_read_per_step"] + tj["dram_bytes_write_per_step"]) if tj else None
    if S > 20:
        # dense contraction: the FP64 tensor pipe (mma.sync m8n8k4, SASS DMMA) is the roofline (10.2 flop/B at S = 61)
        peak = fp64["dmma_m8n8k4_tflops"] if fp64 else 37.0
        peak_src = "profiles/r02_fp64_peaks.json dmma_m8n8k4_tflops (tools/fp64_peaks.cu, measured on this pool's B200)" \
            if fp64 else "fallback 37 TFLOP/s"
        achieved = flo / (k_avg_ms * 1e-3) / 1e12
        roof = {"bound": "fp64", "kernel": "k_walk_mma (updatePartials on the fp64 tensor pipe, DMMA m8n8k4)",
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak}
    else:
        peak = peaks["hbm_gbs"] if peaks else 6650.0
        peak_src = "MEASURED_PEAKS.json hbm_gbs (copy, burst)" if peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
        achieved = byt / (k_avg_ms * 1e-3) / 1e9
        roof = {"bound": "hbm", "kernel": ("k_walk4e (updatePartials in eigen form, whole op list in a few launches)"
                                           if S <= 4 else "k_walk_mma (updatePartials on the fp64 tensor pipe)"),
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak}
    hbm_peak = peaks["hbm_gbs"] if peaks else 6650.0
    roof.update({
        "traffic": traffic, "traffic_source": tj["source"] if tj else None, "peak_source": peak_src,
        # DRAM-side view of the same launches: measured bytes (ncu) over the live time.  The algorithmic bytes count every
        # child read, of which those forwarded in registers or served by L2 never reach HBM; dram_frac cannot exceed 1.
        "dram_achieved": (traffic / (k_avg_ms * 1e-3) / 1e9) if traffic else None,
        "dram_frac": (traffic / (k_avg_ms * 1e-3) / 1e9 / hbm_peak) if traffic else None,
        "algorithmic_bytes_per_step": byt, "algorithmic_flops_per_step": flo,
        "gflops": flo / (k_avg_ms * 1e-3) / 1e9, "hbm_gbs_algorithmic": byt / (k_avg_ms * 1e-3) / 1e9,
        "partials_ms_per_step": k_avg_ms, "launches_per_step": k_n / args.steps,
        "op_mix": ev.mix, "share_of_step": k_ms / (k_ms + m_ms + r_ms),
        "other_kernels_ms_per_step": {"transition_matrices": m_ms / args.steps, "root": r_ms / args.steps},
        "timing": "CUDA events around every launch of the class on the engine's stream, in a K-step block of its own"})
    e2e = r["e2e"]
    line = dict(meta_base)
    line.update({
        "value": value, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dev_ms / args.steps, "wall_ms_per_step": blocks["wall_ms_per_step"],
        "repeats": blocks["repeats"], "block_ms_p10": blocks["block_ms_p10"], "block_ms_p50": blocks["block_ms_p50"],
        "block_ms_p90": blocks["block_ms_p90"],
        "timed_ms": blocks["timed_ms"],
        "statistic": "`steps` timed steps in `repeats` consecutive windows, each window = max over ranks of its CUDA-event "
                     "time; median per-step time over the windows",
        "vs_baseline": None, "logL": r["joint"], "joint_evals_per_s": args.steps / (dev_ms * 1e-3),
        "roofline": roof,
        "e2e": {"value": world / e2e["median_s"], "unit": "evals/s", "ms_per_step": e2e["median_ms"],
                "h2d_bytes_per_step": ev.h2d_bytes(S, C), "d2h_bytes_per_step": 8, "logL": e2e["logL"],
                "steps": e2e["steps"], "statistic": "median step, max over ranks", "c_abi_replay": e2e.get("c_abi_replay"),
                "per_call_rank0": {k: e2e[k] for k in ("p10_ms", "median_ms", "p90_ms")}},
        "gpu_launches": int(k_n + m_n + r_n),
        "clocks": clocks,
        "incremental": inc,
        "cold_plan": cold,
        "strong_scaling": strong,
    })
    if not args.no_cpu_baseline:
        from beast_mcmc_b200 import build
        build.build_oracle()
        cores = os.cpu_count() or 1
        evc = Evaluation(tree, pats, model, site, "POST_ORDER", scaling=scaling)
        threads, tried = cpu_pick_threads(evc, S, C, P, cores)
        times, cval = cpu_time_evaluations(evc, S, C, P, threads, 5, args.cpu_budget)
        line["cpu_baseline"] = {"value": 1.0 / statistics.median(times), "unit": "evals/s", "cores": threads,
                                "host_cores": cores, "kind": "port",
                                "sample": f"{len(times)} full evaluations of this rank-0 shard (median), "
                                          f"oracle/beagle_cpu.c with {threads} threads (best median of "
                                          f"{[t for t, _ in tried]})",
                                "logL": cval, "rel_diff_vs_gpu": abs(cval - r["first_logL"]) / abs(cval)
                                if world == 1 else None}
        t1, _ = cpu_time_evaluations(evc, S, C, P, 1, 1, 0.0)
        line["cpu_baseline"]["single_thread"] = 1.0 / statistics.median(t1)
        if inc is not None:
            from oracle import cpu
            cinst = create_instance(cpu.factory(threads=threads), evc, S, C, P, None)
            issue_sync(cinst, evc, 0, out)
            cper = run_incremental(cinst, 2)
            cinst.finalize()
            inc["cpu_port_evals_per_s"] = 1.0 / statistics.median(cper)
    print(json.dumps(line), flush=True)
    D.close()


if __name__ == "__main__":
    main()
