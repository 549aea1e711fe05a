"""Word-analogy throughput (GloveEngine.analogy) at the size of a real evaluation: 19,544 synthetic questions (the size of
questions-words.txt) against the cfg3 table shape, V = 400,000 rows of d = 300 (486 MB, larger than the 126 MB L2), both
methods, over the full vocabulary and the first 30,000 rows (--restrict-vocab 30000, which fits in L2).

Prints one JSON line: the card name and power limit (read in the same run), and per arm the median time of an
engine.analogy call (device events around the call: H2D of the question ids, kernels, D2H of the answers), questions/s
and algorithmic FLOP/s:
  * add: 2 n V Kp on the tensor cores (Kp = d padded to 64) -- the exact fp32 re-score of ~32 candidates per slice and
    query is < 0.01 % of that and not counted;
  * mul: 6 n V d in fp32 (three dot products of d per question and candidate).
A host NumPy float32 arm does the same work for a subset of the questions (--host-questions), for scale."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [s.strip() for s in out.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def host_arm(W, abc, method, restrict):
    """NumPy float32: normalise, score every candidate, exclude a, b, c, argmax (top-1)."""
    t0 = time.perf_counter()
    Wn = W / np.sqrt(np.maximum((W * W).sum(1, keepdims=True), np.float32(1e-12)))
    cand = Wn[:restrict]
    a, b, c = Wn[abc[:, 0]], Wn[abc[:, 1]], Wn[abc[:, 2]]
    if method == "add":
        q = b - a + c
        s = q @ cand.T
    else:
        s = ((1 + b @ cand.T) / 2) * ((1 + c @ cand.T) / 2) / ((1 + a @ cand.T) / 2 + np.float32(1e-3))
    rows = np.arange(len(abc))[:, None]
    s[rows, abc] = -np.inf
    s.argmax(1)
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--V", type=int, default=400_000)
    ap.add_argument("--d", type=int, default=300)
    ap.add_argument("--n", type=int, default=19_544)
    ap.add_argument("--restrict", type=int, default=30_000)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--host-questions", type=int, default=256)
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    a = ap.parse_args()
    import torch
    from glove_tensorflow_b200._lib import lib
    from glove_tensorflow_b200.engine import GloveEngine
    info = card()
    eng = GloveEngine(a.V, a.d, optimizer="SGD", batch_size=64, plan_steps=1, max_steps=4)
    eng.init_uniform(0)
    W = eng.row_embeddings().cpu().numpy()
    rng = np.random.default_rng(1)
    Kp = lib.glove_topk_kpad(a.d)
    arms = []
    for restrict in (None, a.restrict):
        R = a.V if restrict is None else restrict
        abc = rng.integers(0, R, (a.n, 3))
        for method in ("add", "mul"):
            eng.analogy(abc[:512], 1, method, restrict=restrict)     # warm-up: module load, normalised table, maps
            eng.analogy(abc, 1, method, restrict=restrict)
            ts = []
            for _ in range(a.iters):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                eng.analogy(abc, 1, method, restrict=restrict)
                e1.record()
                e1.synchronize()
                ts.append(e0.elapsed_time(e1) / 1e3)
            t = float(np.median(ts))
            flops = 2.0 * a.n * R * Kp if method == "add" else 6.0 * a.n * R * a.d
            nh = min(a.host_questions, a.n)
            th = host_arm(W, abc[:nh], method, R)
            arms.append({"method": method, "candidates": R, "seconds": t, "seconds_all": ts, "questions_per_s": a.n / t,
                         "algorithmic_tflops": flops / t / 1e12,
                         "flop_count": "2*n*V*Kp (tensor cores)" if method == "add" else "6*n*V*d (fp32)",
                         "host_numpy_f32": {"questions": nh, "seconds": th, "questions_per_s": nh / th,
                                            "algorithmic_tflops": flops * nh / a.n / th / 1e12}})
    line = json.dumps({"workload": "word analogies", "V": a.V, "d": a.d, "Kp": Kp, "n_questions": a.n, "k": 1,
                       "card": info, "arms": arms,
                       "note": "median of %d engine.analogy calls after warm-up, device events around the call; the "
                               "full table (486 MB) is read from HBM, the 30,000-row restriction fits in L2" % a.iters})
    print(line)
    if a.out:
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
