#!/usr/bin/env python
"""bench.py -- co-occurrence updates/sec of the GloVe TRAIN step on B200 (metric of BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload wiki6b|text8|cc|topk]
                    [--adam-mode replay|replay_exact|lazy|dense] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...        # the reference path's CPU restatement on the box's host cores

A "step" is one full TRAIN step (gather + loss + gradient + optimizer) over one batch of B_local*N synthetic
co-occurrence triples.  Default workload = BASELINE.json configs[2] ("wiki6b": Zipf co-occurrence, V=400k, d=300,
Adam, B=65,536 per GPU, data-parallel at 1/2/4/8 GPUs) -- the configuration the metric's "at 1/2/4/8 B200" is quoted
on; it fits one GPU.  ``--workload text8`` is configs[1] (V=10,001, d=64, B=65,536), ``cc`` is configs[3]'s table
shape (V=2.2M; row-sharded tables at N>1); ``topk`` is configs[4] alone (cosine top-k over a 2.2M x 300 table, k=10,
65,536 queries per call, tensor-core roofline) -- the default run also appends it as the ``topk`` record at N=1.

N = 1: whole plan chunks (16 steps) go out as one CUDA-graph launch each (``--no-graph``: step by step); the timed region
starts after 2,048 real TRAIN steps.  N > 1: row-sharded tables with a frequency-balanced owner map, exchange fused into
the stage kernel over NVLink peer memory and device-side synchronisation (``--shard-exchange peer-push``; no NCCL on the
step path), plans built by one rank per chunk and shared over peer memory (``--no-plan-sharing``: every rank builds every
plan); the e2e leg feeds every rank 1/N of each batch from pinned host memory.

One JSON line is printed by rank 0 (see DESIGN.md "Measurement" for every key).
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

WORKLOADS = {
    #            V        d    B_local  nnz (per job)
    "wiki6b": (400_000, 300, 65_536, 1 << 28),
    "text8": (10_001, 64, 65_536, 873_186),
    "cc": (2_200_000, 300, 65_536, 1 << 28),
}
ADAM_K = 6  # read + write of (x, m, v)
T0 = 2048   # TRAIN steps run from the cold start before the timed region (or the step the emulated state resumes at)
TOPK = (2_200_000, 300, 65_536, 10)   # BASELINE configs[4]: V, d, queries per call, k


def algorithmic_bytes(B, U_r, U_c, d, k_opt=ADAM_K):
    """SURVEY §8(d): B*16 + (U_r + U_c) * (4d + 4) * k_opt."""
    return B * 16 + (U_r + U_c) * (4 * d + 4) * k_opt


# ------------------------------------------------------------------------------------------------------------------
# synthetic data (SURVEY §8d cfg3 generator): Zipf(s=1) ids by inverse CDF, reject i == j, Pareto counts
# ------------------------------------------------------------------------------------------------------------------
def zipf_cdf(V):
    p = 1.0 / np.arange(1, V + 1, dtype=np.float64)
    p /= p.sum()
    return p, np.cumsum(p)


def gen_coo_numpy(V, n, seed):
    rng = np.random.default_rng(seed)
    p, cdf = zipf_cdf(V)
    row = np.minimum(np.searchsorted(cdf, rng.random(n)), V - 1).astype(np.int32)
    col = np.minimum(np.searchsorted(cdf, rng.random(n)), V - 1).astype(np.int32)
    col = np.where(col == row, (col + 1) % V, col).astype(np.int32)
    count = 10 + np.floor(np.minimum(rng.pareto(1.0, n), 1e6))
    value = count * rng.uniform(0.3, 0.6, n)
    return {"row": row, "col": col, "target": np.log(value).astype(np.float32),
            "weight": np.minimum(1.0, (count / 100.0) ** 0.75).astype(np.float32)}


def gen_coo_device(V, n, seed, device):
    import torch
    gen = torch.Generator(device=device).manual_seed(seed)
    _, cdf = zipf_cdf(V)
    cdf_t = torch.from_numpy(cdf.astype(np.float32)).to(device)
    row = torch.empty(n, dtype=torch.int32, device=device)
    col = torch.empty(n, dtype=torch.int32, device=device)
    tgt = torch.empty(n, dtype=torch.float32, device=device)
    wgt = torch.empty(n, dtype=torch.float32, device=device)
    chunk = 1 << 24
    for s in range(0, n, chunk):
        m = min(chunk, n - s)
        r = torch.searchsorted(cdf_t, torch.rand(m, device=device, generator=gen)).clamp_(max=V - 1)
        c = torch.searchsorted(cdf_t, torch.rand(m, device=device, generator=gen)).clamp_(max=V - 1)
        c = torch.where(c == r, (c + 1) % V, c)
        u = torch.rand(m, device=device, generator=gen).clamp_(min=1e-6)
        count = 10 + torch.floor(torch.clamp(1.0 / u - 1.0, max=1e6))      # Pareto(alpha=1) by inverse CDF
        value = count * (0.3 + 0.3 * torch.rand(m, device=device, generator=gen))
        row[s:s + m] = r.to(torch.int32)
        col[s:s + m] = c.to(torch.int32)
        tgt[s:s + m] = torch.log(value)
        wgt[s:s + m] = torch.clamp((count / 100.0) ** 0.75, max=1.0)
    return row, col, tgt, wgt


def steady_state(eng, V, B_global, seed):
    """Emulate resuming a long run at step T0: per-row last_step drawn from the stationary gap distribution of a row
    with Zipf touch probability, non-zero Adam slots on rows that have been touched.  Without this a short benchmark
    would see only first-touch rows and skip the replay work that the reference-exact Adam schedule costs."""
    import torch
    dev = eng.device
    gen = torch.Generator(device=dev).manual_seed(seed)
    p, _ = zipf_cdf(V)
    q = -np.expm1(B_global * np.log1p(-p))                      # P(row touched in a step)
    q_t = torch.from_numpy(q.astype(np.float32)).to(dev).clamp_(1e-12, 1 - 1e-7)
    def local(t):   # row-sharded tables: keep the rows this rank owns (id % world == rank), zero-padded
        if not eng.sharded:
            return t
        own = t[eng.dp_rank::eng.dp_world]
        out = torch.zeros((eng.V,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        out[: own.shape[0]] = own
        return out
    for side in ("row", "col"):
        u = torch.rand(V, device=dev, generator=gen).clamp_(min=1e-12)
        gap = torch.floor(torch.log(u) / torch.log1p(-q_t))     # Geometric(q): idle steps since last touch
        ls = torch.where(gap < T0, T0 - gap, torch.zeros_like(gap)).to(torch.int32)
        touched = (ls > 0).to(torch.float32)
        m = torch.randn(V, eng.d, device=dev, generator=gen) * 1e-6 * touched[:, None]
        v = torch.rand(V, eng.d, device=dev, generator=gen) * 1e-12 * touched[:, None]
        eng.set_plane(side, 1, local(m), local(torch.randn(V, device=dev, generator=gen) * 1e-6 * touched))
        eng.set_plane(side, 2, local(v), local(torch.rand(V, device=dev, generator=gen) * 1e-12 * touched))
        eng.set_last_step(side, local(ls))
        del m, v
    eng.set_step(T0)


# ------------------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """One persistent `nvidia-smi -lms 100` process; samples are time-stamped so that those inside the timed region can
    be picked out (the region is short: when no sample falls inside it, the nearest ones under load are used)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def run(self):
        if self.proc is None:
            return
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.strip().split(",")]))

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            self.proc = None

    def summary(self, t_start, t_end):
        if self.proc is not None:
            time.sleep(0.15)
        rows = [(t, r) for t, r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        inside = [r for t, r in rows if t_start - 0.05 <= t <= t_end + 0.15]
        used = inside if inside else [r for _, r in sorted(rows, key=lambda tr: abs(tr[0] - t_end))[:3]]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[3 + k].lower().startswith("active") for r in used)]
        return {"sm_mhz": float(np.median([float(r[0]) for r in used])), "sm_max_mhz": float(used[0][1]),
                "reasons": reasons, "samples": len(used), "samples_in_timed_region": len(inside),
                "power_w_max": max(float(r[2]) for r in used)}


# ------------------------------------------------------------------------------------------------------------------
def cpu_reference(V, d, B, steps, warmup, seed=0):
    """Times the C port of the oracle (legacy-Keras dense Adam, OpenMP over host cores) on `steps` TRAIN steps of the
    same workload shape.  Returns (updates/s, seconds, cores)."""
    from oracle import c_oracle, glove_oracle as o
    n = max(B * 4, 1 << 20)
    coo = gen_coo_numpy(V, n, seed)
    rng = np.random.default_rng(seed + 1)
    st = o.init_state(V, d, seed + 2)
    co = c_oracle.COracle(st.R, st.C, st.rb, st.cb, optimizer="Adam")
    alpha = o.alpha_table(0.001, warmup + steps + 1)
    if warmup:
        co.train(coo, rng.integers(0, n, (warmup, B)), alpha=alpha)
    idx = rng.integers(0, n, (steps, B))
    t0 = time.perf_counter()
    co.train(coo, idx, alpha=alpha)
    dt = time.perf_counter() - t0
    return steps * B / dt, dt, c_oracle.num_threads()


DUMP_HEAD, DUMP_SAMPLE = 4096, 12288   # rows dumped per table: the most frequent ids + a seeded sample of the rest
DUMP_LIMIT = 64 << 20                  # bytes


def train_outputs(eng, losses):
    """What a caller of the TRAIN step holds after the last timed step: the losses of the timed steps and the variables in
    reference layout (lazy Adam state replayed up to the current step, as GloveEngine.get_state gives them), on a fixed
    set of rows: ids 0 .. DUMP_HEAD-1 (Zipf head: touched by nearly every step) and a seeded sample of the others."""
    import torch
    V = eng.V
    rows = np.arange(V)
    if V > DUMP_HEAD + DUMP_SAMPLE:
        tail = np.random.default_rng(0).choice(np.arange(DUMP_HEAD, V), DUMP_SAMPLE, replace=False)
        rows = np.concatenate([rows[:DUMP_HEAD], np.sort(tail)])
    eng.flush()
    idx = torch.from_numpy(rows).to(eng.device)
    out = {"losses": losses, "rows": rows}
    for name, bname, table in (("R", "rb", eng.row_table), ("C", "cb", eng.col_table)):
        e, b = eng._unpack(table, 0)
        out[name], out[bname] = e[idx].cpu().numpy(), b[idx].cpu().numpy()
        del e, b
    out["g"] = np.array([eng.read_scalars()["g"]], np.float32)
    return out


def dump_outputs(out_dir, arrays):
    """<out_dir>/<name>.npy for every array: float32 stays float32, anything else (ids included, exactly) is float64."""
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    arrays = {k: v if v.dtype == np.float32 else v.astype(np.float64) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_LIMIT:
        raise ValueError("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT))
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def load_traffic(key):
    """(bytes per step, source) from profiles/step_traffic.json: {key: {"dram_bytes": n, "source": "profiles/..."}}."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "step_traffic.json")))[key]
        return float(t["dram_bytes"]), t.get("source")
    except Exception:
        return None, None


def topk_record(dev, sampler, full_line=False, n_gpus=1, steps=5, warmup=3, outputs=None):
    """BASELINE configs[4]: cosine top-k of Q = 65,536 query rows over a 2.2M x 300 table, k = 10 (tcgen05 candidate pass +
    exact fp32 re-score), per GPU (N > 1: replicas, queries sharded -- every rank runs the same call).  Algorithmic flops
    = 2*Q*V*d (padding d to 320 is overhead, not credit).  `value` is device-timed (CUDA events around the whole topk
    call incl. normalised-query gather, candidate pass, re-score, guarantee check; query ids resident); `e2e` is the wall
    time of GloveEngine.topk from HOST query ids to HOST results.  `outputs` (a dict) receives the last timed call's
    results as topk_sim / topk_idx [Q, k]."""
    import torch
    from glove_tensorflow_b200.engine import GloveEngine
    V, d, Q, k = TOPK
    iters = max(1, steps)
    eng = GloveEngine(V, d, optimizer="SGD", batch_size=64, plan_steps=1, max_steps=4, device=dev)
    eng.init_uniform(0)
    q = torch.randint(0, V, (Q,), generator=torch.Generator().manual_seed(1)).numpy().astype(np.int32)
    for _ in range(max(1, min(warmup, 3))):
        eng.topk(q, k)                                                  # warm-up (normalises the table once)
    torch.cuda.synchronize()
    t_start = time.time()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    qd = torch.from_numpy(q).to(dev)
    inv, nb = eng._normalised_table()
    ev[0].record()
    for _ in range(iters):
        sim, idx = eng._topk_call(inv, nb, eng.row_table, eng.P, nb, qd, Q, k, False)
    ev[1].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1]) / iters
    fallbacks = eng.last_topk_fallbacks
    if outputs is not None:
        outputs["topk_sim"], outputs["topk_idx"] = sim.cpu().numpy().reshape(Q, k), idx.cpu().numpy().reshape(Q, k)
    t0 = time.perf_counter()
    for _ in range(iters):
        eng.topk(q, k)
    wall = (time.perf_counter() - t0) / iters
    t_end = time.time()
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("bf16_tflops", 1590.0))
    flop = 2.0 * Q * V * d
    tf = flop / (ms * 1e-3) / 1e12
    rec = {"metric": "cosine top-k algorithmic TFLOP/s (2*Q*V*d)", "value": tf * n_gpus, "unit": "TFLOP/s", "ms_per_call": ms,
           "queries_per_s": Q / (ms * 1e-3) * n_gpus, "fallbacks": fallbacks,
           "config": {"workload": "topk: cosine top-k, V=%d, d=%d, k=%d, Q=%d queries per call per GPU, table U(-0.05,0.05)"
                                  % (V, d, k, Q), "l2_flush": "bf16 table 1.4 GB + fp32 table 2.7 GB, larger than L2"},
           "roofline": {"bound": "tensor", "achieved": tf, "peak": peak, "unit": "TFLOP/s", "frac": tf / peak,
                        "traffic": None, "peak_source": "measured bf16 burst (MEASURED_PEAKS.json)" if peaks else "fallback 1590",
                        "kernel": "topk_tc_kernel (tcgen05 candidate pass) + exact fp32 re-score; flops are algorithmic"},
           "e2e": {"value": flop / wall / 1e12 * n_gpus, "unit": "TFLOP/s", "h2d_bytes_per_step": 4 * Q, "d2h_bytes_per_step": 8 * Q * k,
                   "path": "GloveEngine.topk: host query ids -> device -> candidates -> re-score -> host (sim, idx)"},
           "clocks": sampler.summary(t_start, t_end) if sampler is not None else None}
    if full_line:
        rec.update({"n_gpus": n_gpus, "steps": iters, "warmup": max(1, min(warmup, 3)), "ms_per_step": ms, "higher_is_better": True,
                    "scaling": "weak", "vs_baseline": None, "dtype": "bf16 candidates, f32 re-score", "data": "synthetic",
                    "gpu_launches": iters * 6, "cpu_baseline": None})
    del eng
    torch.cuda.empty_cache()
    return rec


def topk_reference_line(args):
    """--impl reference --workload topk: the reference's own PREDICT arithmetic (l2-normalise the whole table, matmul,
    top_k; src/models/utils.py:12-19, model_utils.py:97-99) restated in NumPy fp32 on the host cores, on a bounded sample
    of the queries of the same table shape."""
    from oracle import glove_oracle as o
    V, d, Q, k = TOPK
    rng = np.random.default_rng(0)
    T = rng.uniform(-0.05, 0.05, (V, d)).astype(np.float32)
    nq = 64
    q = rng.integers(0, V, nq)
    o.cosine_topk(T[:1000], q[:4] % 1000, k)
    t0 = time.perf_counter()
    o.cosine_topk(T, q, k)
    dt = time.perf_counter() - t0
    tf = 2.0 * nq * V * d / dt / 1e12
    cores = os.cpu_count() or 1
    return {"metric": "cosine top-k algorithmic TFLOP/s (2*Q*V*d)", "value": tf, "unit": "TFLOP/s", "n_gpus": args.gpus, "steps": 1,
            "warmup": 1, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": "topk: cosine top-k, V=%d, d=%d, k=%d, Q=%d queries per call per GPU, table U(-0.05,0.05)"
                                   % (V, d, k, Q), "l2_flush": "bf16 table 1.4 GB + fp32 table 2.7 GB, larger than L2"},
            "cpu_baseline": {"value": tf, "unit": "TFLOP/s", "cores": cores, "kind": "port",
                             "sample": "%d queries (of %d) against the full table, NumPy fp32 restatement of cosine_similarity + "
                                       "top_k incl. the per-call normalisation of the table, BLAS threads" % (nq, Q)},
            "e2e": {"value": tf, "unit": "TFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="wiki6b", choices=sorted(WORKLOADS) + ["topk"])
    ap.add_argument("--adam-mode", default="replay", choices=["replay", "replay_exact", "lazy", "dense"],
                    help="replay = closed-form replay of idle Adam steps (default; reference semantics), replay_exact = "
                         "step-by-step replay with the dense sweep's fp32 operations, dense = replay_exact + flush after "
                         "every step, lazy = LazyAdam (not the reference's arithmetic)")
    ap.add_argument("--batch", type=int, default=None, help="per-GPU batch (default: workload's)")
    ap.add_argument("--nnz", type=int, default=None)
    ap.add_argument("--plan-steps", type=int, default=16)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cold-state", action="store_true", help="time from step 0 with empty Adam state")
    ap.add_argument("--emulate-state", action="store_true",
                    help="instead of really training %d steps first, start from a synthetic steady state (round-1 method)" % T0)
    ap.add_argument("--pretrain-steps", type=int, default=T0,
                    help="TRAIN steps run from the cold start before the timed region (default %d; profiling runs use fewer)" % T0)
    ap.add_argument("--no-balance", action="store_true",
                    help="N>1, row-sharded tables: keep owner = id %% N instead of the frequency-balanced owner map")
    ap.add_argument("--no-plan-sharing", action="store_true",
                    help="N>1, row-sharded tables: every rank builds the plan of every chunk itself (round-2 behaviour) instead "
                         "of taking turns and pulling slices over peer memory")
    ap.add_argument("--step-priority", action="store_true", help="run the steps on a high-priority CUDA stream (experiment)")
    ap.add_argument("--no-graph", action="store_true",
                    help="launch every step's kernels one by one instead of one CUDA graph per plan chunk (N=1)")
    ap.add_argument("--no-topk", action="store_true", help="skip the cfg5 top-k record of the default N=1 run")
    ap.add_argument("--shard-exchange", default="peer-push", choices=["alltoall", "allgather", "peer", "peer-direct", "peer-sync", "peer-push"],
                    help="N>1, row-sharded tables: how the snapshot rows reach the shards that need them (peer = one pull "
                         "kernel over NVLink peer memory; falls back to alltoall when symmetric memory is unavailable)")
    ap.add_argument("--dp-mode", default="sharded", choices=["sharded", "replicated"],
                    help="N>1: row-sharded tables (owner-computes) or replicated tables with gradient all-reduce")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (a fixed sample of the "
                         "tables; with --workload topk or the default run's topk record, the top-k results too)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs needs --impl b200 on one GPU")

    V, d, B_local, nnz = WORKLOADS["wiki6b" if args.workload == "topk" else args.workload]
    B_local = args.batch or B_local
    nnz = args.nnz or nnz
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    N = max(world, 1)
    B = B_local * N                                            # global batch (weak scaling)
    S_pad = (d + 2 + 7) // 8 * 8

    def make_config():
        """The workload description BOTH arms print (every value is derivable without a GPU)."""
        return {"workload": "%s: synthetic Zipf(s=1) co-occurrence, V=%d, d=%d, Adam lr 1e-3, l2 0.01, B=%d per GPU"
                            % (args.workload, V, d, B_local), "nnz": nnz, "batch_per_gpu": B_local, "global_batch": B,
                "adam_mode": args.adam_mode,
                "parallelism": ("dp%d" % N) if N == 1 else ("dp%d-%s-tables%s" % (
                    N, args.dp_mode, "-" + args.shard_exchange if args.dp_mode == "sharded" else "")),
                "l2_flush": "inputs larger than L2 (tables+slots %.1f GB, COO %.1f GB)"
                            % (2 * V * 3 * S_pad * 4 / 1e9, nnz * 16 / 1e9),
                "state": ("cold" if args.cold_state else "steady-state emulation at step %d" % T0 if args.emulate_state
                          else "trained %d steps from a cold start before the timed region" % args.pretrain_steps)}

    # ---- reference arm: CPU restatement of the reference TRAIN step on host cores -------------------------------
    if args.impl == "reference":
        if rank != 0:
            return
        if world > 1 and os.environ.get("OMP_NUM_THREADS") == "1":
            os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)   # torchrun pins 1 thread per rank; rank 0 runs alone here
        if args.workload == "topk":
            print(json.dumps(topk_reference_line(args)))
            return
        steps = max(1, min(args.steps, 96 if V >= 100_000 else 1024))   # bounded sample of the same shape
        warm = min(max(args.warmup, 3), 32)
        ups, dt, cores = cpu_reference(V, d, B, steps, warm)
        line = {"metric": "co-occurrence updates/sec", "value": ups, "unit": "updates/s", "n_gpus": args.gpus, "steps": steps,
                "warmup": warm, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
                "config": make_config(),
                "cpu_baseline": {"value": ups, "unit": "updates/s", "cores": cores, "kind": "port",
                                 "sample": "%d TRAIN steps of B=%d (requested %d) after %d warm-up steps, C port of the oracle, "
                                           "OpenMP on %d threads, legacy-Keras dense Adam (what adam_mode=replay reproduces; "
                                           "the dense sweep costs the same at any step, so the state is cold); "
                                           "restatement of the reference path, not TensorFlow"
                                           % (steps, B, args.steps, warm, cores)},
                "e2e": {"value": ups, "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    from glove_tensorflow_b200.engine import GloveEngine
    from glove_tensorflow_b200 import _lib

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if args.step_priority:
        # the step kernels run on a high-priority stream: when a plan-construction kernel (side streams, default priority)
        # and a step kernel both have blocks pending, the SMs take the step's first
        torch.cuda.set_stream(torch.cuda.Stream(device=dev, priority=-1))
    sampler = ClockSampler(local_rank)          # started early: nvidia-smi takes a while to deliver its first sample
    if rank == 0:
        sampler.start()
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    outputs = {} if args.dump_outputs else None
    if args.workload == "topk":
        line = topk_record(dev, sampler if rank == 0 else None, full_line=True, n_gpus=N, steps=args.steps, warmup=args.warmup,
                           outputs=outputs)
        if rank == 0:
            sampler.stop()
            if outputs is not None:
                dump_outputs(args.dump_outputs, outputs)
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return
    K = args.plan_steps
    steps = (args.steps + K - 1) // K * K if not args.no_e2e else args.steps
    total_steps = args.warmup + args.steps + 3 * K + 64 + 2 * 16 * K     # + warm and timed e2e calls of up to 16 chunks
    eng = GloveEngine(V, d, optimizer="Adam", learning_rate=0.001, l2_reg=0.01, reg_scale=2.0, head="glove",
                      adam_mode=args.adam_mode, batch_size=B, plan_steps=K, max_steps=2 * T0 + 2 * total_steps + steps,
                      device=dev, dp_rank=rank, dp_world=N, dp_mode=args.dp_mode)
    eng.shard_exchange = args.shard_exchange
    if args.shard_exchange.startswith("peer") and world > 1 and args.dp_mode == "sharded":
        try:
            eng.enable_peer_gather(direct=args.shard_exchange == "peer-direct", sync=args.shard_exchange == "peer-sync",
                                   push=args.shard_exchange == "peer-push")
            args.shard_exchange = eng.shard_exchange
        except Exception as exc:   # no peer-mapped memory on this box: same exchange through NCCL
            print("bench: peer memory unavailable (%s); using the all-to-all exchange" % exc, file=sys.stderr)
            args.shard_exchange = eng.shard_exchange = "alltoall"
    elif world <= 1 or args.dp_mode != "sharded":
        args.shard_exchange = eng.shard_exchange = "alltoall"
    plan_sharing = False
    if world > 1 and args.dp_mode == "sharded" and eng.shard_exchange.startswith("peer") and not args.no_plan_sharing:
        ok = torch.ones(1, device=dev)
        try:
            eng.enable_plan_sharing()       # rank c % N builds the plan of chunk c, everyone pulls its slice over NVLink
        except Exception as exc:
            print("bench: shared plan construction unavailable (%s); every rank builds every plan" % exc, file=sys.stderr)
            ok.zero_()
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        plan_sharing = bool(ok.item())
        if not plan_sharing:
            eng._ring = None
    row, col, tgt, wgt = gen_coo_device(V, nnz, 1234, dev)     # replicated COO (weak scaling: B grows with N)
    row0, col0 = row, col
    owner_load = None
    if world > 1 and args.dp_mode == "sharded" and not args.no_balance:
        owner_load = eng.balance_owners(row, col)              # frequency-balanced owner map (before any state is loaded)
    eng.init_uniform(seed=1)                                   # same seed on every rank: replicas start identical
    eng.set_coo(row, col, tgt, wgt, shuffle_key=0xC0FFEE)
    if args.emulate_state and not args.cold_state:
        steady_state(eng, V, B, seed=99)
    elif not args.cold_state:
        # REAL state: T0 TRAIN steps from the cold start (every row the timed region touches then carries the last_step,
        # m, v a long run gives it; the idle gaps the stage has to replay are the workload's own)
        for _ in range(args.pretrain_steps):
            eng.step()
    torch.cuda.synchronize()

    # N > 1: the peer-sync step is graph-capturable too, but measured slower as a graph than launched step by step at N = 2
    # (0.282 vs 0.254 ms/step: profiles/r02_scaling.md), so the multi-GPU arm launches its steps one C call at a time
    eng.use_graph = (not args.no_graph) and N == 1

    def run_steps(n):
        """exactly n TRAIN steps: whole plan chunks as one CUDA graph launch each (N = 1), single launches otherwise"""
        while n:
            k = eng.step_chunk_graph() if (eng.use_graph and n >= eng.K) else 0
            if not k:
                eng.step()
                k = 1
            n -= k

    # ---- warm-up ---------------------------------------------------------------------------------------------------
    run_steps(max(args.warmup, 3))
    torch.cuda.synchronize()
    # distinct ids per step for the roofline figure (outside the timed region)
    first_timed = eng.host_step
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_start = time.time()
    e0.record()
    run_steps(args.steps)
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    t_end = time.time()
    clocks = sampler.summary(t_start, t_end) if rank == 0 else None
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    sc = eng.read_scalars()
    assert sc["error"] == 0 and sc["step"] == eng.host_step, sc
    losses = eng.loss_out[(torch.arange(first_timed, eng.host_step, device=dev) % eng.loss_cap)].cpu().numpy()
    assert np.all(np.isfinite(losses)), "non-finite loss in the timed region"
    value = B * args.steps / (ms * 1e-3)
    final_loss = losses[-1]
    if outputs is not None:
        outputs.update(train_outputs(eng, losses))

    # ---- roofline: per-kernel durations (CUDA events on the launching stream) + algorithmic bytes -------------------
    U = np.array([eng.batch_counts(s)[:2] for s in range(first_timed, first_timed + min(args.steps, 32))], np.float64)
    U_r, U_c = U.mean(0)
    bytes_alg = algorithmic_bytes(B, U_r, U_c, d)
    roofline, kernels_ms = None, None
    if N == 1:
        prof = np.array([eng.step_profiled() for _ in range(32)])
        kernels_ms = {"stage": float(prof[:, 0].mean()), "update": float(prof[:, 1].mean())}
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        step_ms = ms / args.steps
        achieved = bytes_alg / (step_ms * 1e-3) / 1e9
        # dram__bytes_read.sum + dram__bytes_write.sum of the step's kernels, per launch, parsed at run time from the committed
        # ncu export of this workload (profiles/step_traffic.json, written by tools/ncu_summary.py); null when absent
        traffic, traffic_src = load_traffic("%s/%s/B%d" % (args.workload, args.adam_mode, B_local))
        upd_alg = bytes_alg - (U_r + U_c) * (4 * d + 4)        # everything but the first read of x (done by the stage)
        roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": "measured (MEASURED_PEAKS.json)" if peaks else "fallback 6650",
                    "kernel": "whole step = stage kernel + update_kernel (algorithmic bytes are per step)",
                    "algorithmic_bytes_per_step": bytes_alg, "U_row": U_r, "U_col": U_c,
                    "rho": (U_r + U_c) / (2.0 * B), "frac_of_nominal_8000": achieved / 8000.0,
                    "kernels_ms": kernels_ms,
                    "update_kernel": {"algorithmic_bytes": upd_alg, "ms": kernels_ms["update"],
                                      "achieved": upd_alg / (kernels_ms["update"] * 1e-3) / 1e9,
                                      "frac": upd_alg / (kernels_ms["update"] * 1e-3) / 1e9 / peak},
                    "update_kernel_share": kernels_ms["update"] / max(sum(kernels_ms.values()), 1e-9)}

    # ---- e2e: HOST buffers through the C ABI (glove_train_steps_host): H2D of every batch + D2H of every loss --------
    e2e = None
    if not args.no_e2e:
        # one call = CALL plan chunks (N == 1: pipelined inside glove_train_steps_host); host buffers of `pool` calls rotate
        CALL = 8 if N == 1 else (2 * N if plan_sharing else 4)   # shared plans: whole rounds of N chunks, two per call
        KC = K * CALL
        n_chunks = max(1, args.steps // KC)
        pool = 2
        # N > 1: every rank holds (and copies) only ITS share of each batch, [KC][B_local]; the ranks all-gather on the device
        HB = B if N == 1 else B_local
        hr = [torch.empty(KC * HB, dtype=torch.int32).pin_memory() for _ in range(pool)]
        hc = [torch.empty(KC * HB, dtype=torch.int32).pin_memory() for _ in range(pool)]
        ha = [torch.empty(KC * HB, dtype=torch.float32).pin_memory() for _ in range(pool)]
        hb = [torch.empty(KC * HB, dtype=torch.float32).pin_memory() for _ in range(pool)]
        hl = torch.empty(KC, dtype=torch.float32).pin_memory()
        for i in range(pool):
            sel = torch.arange(KC * B, device=dev, dtype=torch.int64) + i * KC * B
            if N > 1:
                sel = sel.view(KC, N, B_local)[:, rank, :].reshape(-1)
            sel = sel % nnz
            hr[i].copy_(row0[sel]); hc[i].copy_(col0[sel]); ha[i].copy_(tgt[sel]); hb[i].copy_(wgt[sel])
        torch.cuda.synchronize()

        def chunk(i):
            if N == 1:
                eng.train_steps_host(hr[i], hc[i], ha[i], hb[i], hl)      # one C-ABI call, HOST buffers in / losses out
            else:
                KB = K * HB
                eng.train_chunks_from_host([tuple(t[i][j * KB:(j + 1) * KB] for t in (hr, hc, ha, hb)) for j in range(CALL)],
                                           sliced=True)
        chunk(0)                                                          # warm
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for c in range(n_chunks):
            chunk(c % pool)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        # the e2e steps are real steps: the device step counter must have followed the host's and no kernel may have refused
        # its plan (error flag), on any rank -- reported as e2e.steps_verified
        sc2 = eng.read_scalars()
        e2e_ok = torch.tensor([1.0 if (sc2["error"] == 0 and sc2["step"] == eng.host_step) else 0.0], device=dev)
        if world > 1:
            dist.all_reduce(e2e_ok, op=dist.ReduceOp.MIN)
        if not bool(e2e_ok.item()):
            print("bench: e2e leg INVALID on rank %d or a peer (device step %d, host %d, error flag %d)"
                  % (rank, sc2["step"], eng.host_step, sc2["error"]), file=sys.stderr)
        e2e = {"value": n_chunks * KC * B / dt, "unit": "updates/s", "h2d_bytes_per_step": B * 16,
               "steps_verified": bool(e2e_ok.item()),    # device step counter == host's and no error flag, on every rank
               "d2h_bytes_per_step": 4 + 4.0 / KC, "steps": n_chunks * KC,
               "path": ("glove_train_steps_host, %d steps per call: pinned host COO -> H2D -> plans -> steps -> D2H losses; inside a "
                        "call the copy + plan of chunk c+1 overlap the steps of chunk c" % KC if N == 1 else
                        "GloveEngine.train_chunks_from_host(sliced) on every rank, %d steps per call: pinned host COO (this rank's "
                        "1/N of every batch) -> H2D -> NCCL all-gather of the chunk -> plans -> sharded steps -> D2H losses; copy + "
                        "gather + plan of chunk c+1 overlap the steps of chunk c; h2d bytes are the sum over ranks" % KC
                        if not plan_sharing else
                        "GloveEngine.train_chunks_from_host(sliced) on every rank, %d steps per call: pinned host COO (this rank's "
                        "1/N of every batch) -> H2D -> one NCCL all-to-all per round of N chunks (rank q receives chunk q) -> rank q "
                        "plans chunk q -> every rank pulls its slice of each plan over NVLink -> sharded steps -> D2H losses; copies, "
                        "exchange and planning of round R+1 overlap the steps of round R; h2d bytes are the sum over ranks" % KC)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    topk = None
    if N == 1 and not args.no_topk and args.workload == "wiki6b":
        eng = row = col = tgt = wgt = None                 # free the training state before the 2.2M-row table
        torch.cuda.empty_cache()
        topk = topk_record(dev, sampler, outputs=outputs)
    sampler.stop()
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)

    cpu = None
    if not args.no_cpu_baseline and N == 1:
        csteps = 96 if V >= 100_000 else 1024                      # about 10 s of CPU work on the box's host cores
        ups, dt, cores = cpu_reference(V, d, B_local, csteps, 3)
        cpu = {"value": ups, "unit": "updates/s", "cores": cores, "kind": "port",
               "sample": "%d TRAIN steps of B=%d (%.1f s), C port of the oracle with OpenMP, legacy-Keras dense Adam"
                         % (csteps, B_local, dt)}

    n_prep = (args.steps + K - 1) // K
    # own kernels per timed step: stage + update (N=1; the finish is fused into the update), or stage + exchange kernels +
    # update + finish on row-sharded tables; + the two Adam catch-up kernels in replay mode.  Plan construction: ~20 own
    # kernels per plan of K steps (CUB sorts / scans inside it not counted).
    if N == 1:
        per_step_launches = 2
    elif args.dp_mode == "sharded":
        per_step_launches = 3 + {"peer": 1, "peer-direct": 0, "alltoall": 2, "allgather": 0, "peer-sync": 2, "peer-push": 2}[args.shard_exchange]
    else:
        per_step_launches = 4
    per_step_launches += 2 if args.adam_mode in ("replay_exact", "dense") else 0
    line = {"metric": "co-occurrence updates/sec", "value": value, "unit": "updates/s", "n_gpus": N,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": make_config(),
            "plans": ("shared: rank c %% %d builds the plan of chunk c, every rank pulls its slice over NVLink" % N) if plan_sharing
                     else "every rank builds every plan",
            "clocks": clocks, "e2e": e2e, "gpu_launches": args.steps * per_step_launches + n_prep * 20,
            "roofline": roofline, "cpu_baseline": cpu, "final_loss": float(final_loss)}
    if topk is not None:
        line["topk"] = topk
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
