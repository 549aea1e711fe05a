"""Stanford GloVe's trainer (stanford_glove.StanfordGlove) on a seeded table: the Stanford scheme of the preprocessor
(window 15, symmetric) over a seeded Zipf corpus with sentence-length lines, as tools/bench_stanford_cooc.py builds it.
At d = 50 and d = 300: epoch time from device events in steady state (after one warm-up epoch), records/s, the longest
dependency chain computed from the links, and epoch time / chain, an upper bound on the latency of one dependent record.
The C oracle's single-thread epoch (glove.c's arithmetic order) is timed on a prefix of the table; it is the oracle,
not glove.c, which cannot be run here, so there is no glove.c baseline.  The card's name and power limit are read in the
same run.  The corpus and the table go to a temporary directory that is deleted at the end.

    python tools/bench_stanford_glove.py --gb 4 --out profiles/r08_stanford_glove_bench.json"""
import argparse
import os
import shutil
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_corpus import card, save  # noqa: E402
from bench_stanford_cooc import write_line_corpus  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gb", type=float, default=4.0, help="corpus size in GB")
    ap.add_argument("--dims", default="50,300")
    ap.add_argument("--epochs", type=int, default=3, help="timed epochs after one warm-up")
    ap.add_argument("--oracle-records", type=int, default=2_000_000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from glove_tensorflow_b200 import corpus
    from glove_tensorflow_b200.data_utils import read_stanford_vocab
    from glove_tensorflow_b200.stanford_glove import StanfordGlove
    from oracle import stanford_glove_oracle as sgo

    res = {"card": card(), "corpus_gb": args.gb, "window": 15, "symmetric": True}
    tmp = tempfile.mkdtemp(prefix="bench_sg_")
    try:
        text = os.path.join(tmp, "corpus.txt")
        write_line_corpus(text, int(args.gb * 1e9))
        t = time.perf_counter()
        corpus.preprocess(text, os.path.join(tmp, "data"), scheme="stanford", window_size=15)
        res["preprocess_s"] = time.perf_counter() - t
        os.remove(text)
        table = os.path.join(tmp, "data", "cooccurrence.shuf.bin")
        V = len(read_stanford_vocab(os.path.join(tmp, "data", "vocab.txt"))[0])
        res["vocab"], res["records"] = V, os.path.getsize(table) // 16
        res["runs"] = []
        chain = None
        for d in [int(x) for x in args.dims.split(",")]:
            t = time.perf_counter()
            sg = StanfordGlove(table, V, d, seed=1)
            torch.cuda.synchronize()
            load_s = time.perf_counter() - t
            if chain is None:
                t = time.perf_counter()
                chain = sgo.chain(sg.prev.cpu().numpy())
                res["longest_chain"], res["chain_host_s"] = chain, time.perf_counter() - t
            costs = [sg.epoch()]                 # warm-up
            times = []
            for _ in range(args.epochs):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                costs.append(sg.epoch())
                b.record()
                b.synchronize()
                times.append(a.elapsed_time(b) / 1e3)
            ep = float(np.median(times))
            run = {"d": d, "load_parse_links_init_s": load_s, "epoch_s": times, "epoch_median_s": ep,
                   "records_per_s": sg.n / ep, "epoch_s_per_chain_step_us": ep / chain * 1e6, "costs": costs}
            print(run, flush=True)
            res["runs"].append(run)
            if d == 50:
                m = min(args.oracle_records, sg.n)
                words, lf = sg.words[:m].cpu().numpy(), sg.lf[:m].cpu().numpy()
                W, G = sg.W.cpu().numpy(), np.ones((2 * V, d + 1))
                t = time.perf_counter()
                sgo.epoch(W, G, words, lf, order=0)
                o = time.perf_counter() - t
                res["oracle_single_thread"] = {"what": "oracle/stanford_glove_oracle.c, glove.c order, one CPU thread "
                                                       "(not glove.c; glove.c was not run)", "d": d, "records": m,
                                               "seconds": o, "records_per_s": m / o}
                print(res["oracle_single_thread"], flush=True)
            del sg
            torch.cuda.empty_cache()
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    print(res)
    if args.out:
        save(args.out, res)


if __name__ == "__main__":
    main()
