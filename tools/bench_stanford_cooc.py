"""The Stanford GloVe scheme of the streamed preprocessor (corpus.preprocess(scheme="stanford")) on a seeded Zipf corpus
with sentence-length lines: pass-1, pass-2 and write times, tokens, vocabulary, directed pairs and records at window 15,
symmetric.  In the same run, alternating, the reference scheme (context 5) on the same corpus with this tree's package and,
with --parent, with another checkout's (built) package, each in a fresh process after a warm-up on a 16 MB prefix; the
reference outputs of the two are compared byte for byte.  The corpus and the outputs go to a temporary directory that is
deleted at the end.  The card's name and power limit are read in the same run.

    python tools/bench_stanford_cooc.py --gb 4 --parent /path/to/parent --out profiles/r07_stanford_cooc_bench.json

Lines of a corpus written by tools/bench_corpus.py hold 8 M words each, which would hide the line logic; here a line
ends after each word with probability 1/20 (mean line length 20 words)."""
import argparse
import filecmp
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_corpus import card, prefix_file, save  # noqa: E402

CHILD = r"""
import json, sys, time
sys.path.insert(0, sys.argv[1])
from glove_tensorflow_b200 import corpus
kw = json.loads(sys.argv[5])
corpus.preprocess(sys.argv[2], sys.argv[4] + ".warm", **kw)
st = {}
t = time.perf_counter()
corpus.preprocess(sys.argv[3], sys.argv[4], stats=st, **kw)
st["end_to_end_s"] = time.perf_counter() - t
print("RESULT " + json.dumps(st))
"""


def write_line_corpus(path, nbytes, vocab=100_000, seed=7, mean_line=20, distinct_bytes=1 << 28):
    """Zipf(1.1) ranks over `vocab` synthetic words; after each word a '\\n' with probability 1 / mean_line, else a space.
    distinct_bytes of seeded text, then that text again until nbytes."""
    rng = np.random.default_rng(seed)
    words = np.array([("t%x" % (i * 2654435761 % (1 << 32))).encode() for i in range(vocab)], dtype=object)
    blocks, done = [], 0
    while done < min(nbytes, distinct_bytes):
        r = rng.zipf(1.1, 4_000_000)
        r = r[r <= vocab] - 1
        out = np.empty(2 * len(r), dtype=object)
        out[0::2] = words[r]
        out[1::2] = np.where(rng.random(len(r)) < 1.0 / mean_line, b"\n", b" ")
        blocks.append(b"".join(out))
        done += len(blocks[-1])
    done = 0
    with open(path, "wb") as f:
        while done < nbytes:
            for b in blocks:
                f.write(b)
                done += len(b)
    return done


def run_child(root, warm, corpus_path, dest, kw):
    out = subprocess.run([sys.executable, "-c", CHILD, root, warm, corpus_path, dest, json.dumps(kw)], capture_output=True,
                         text=True)
    if out.returncode != 0:
        raise RuntimeError("preprocess in %s failed:\n%s" % (root, out.stderr[-4000:]))
    line = [x for x in out.stdout.splitlines() if x.startswith("RESULT ")][-1]
    return json.loads(line[len("RESULT "):])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gb", type=float, default=4.0)
    ap.add_argument("--window-size", type=int, default=15)
    ap.add_argument("--rounds", type=int, default=3, help="alternating rounds of the reference-scheme timing")
    ap.add_argument("--parent", default=None, help="root of another checkout (library built) to time the reference scheme of")
    ap.add_argument("--out", default="profiles/r07_stanford_cooc_bench.json")
    args = ap.parse_args()
    import torch
    from glove_tensorflow_b200 import corpus
    if not torch.cuda.is_available():
        raise SystemExit("bench_stanford_cooc.py needs a GPU")
    res = {"card": card(), "window_size": args.window_size, "symmetric": True, "distance_weighting": True}
    tmp = tempfile.mkdtemp(prefix="glove_stanford_bench_")
    try:
        big = os.path.join(tmp, "corpus.txt")
        t = time.perf_counter()
        nbytes = write_line_corpus(big, int(args.gb * 1e9))
        res["corpus_bytes"], res["generate_s"] = nbytes, time.perf_counter() - t
        res["corpus"] = ("Zipf(1.1) over 100,000 words, seed 7, a line end after each word with probability 1/20: 256 MiB "
                         "of seeded text repeated to the size")
        warm = os.path.join(tmp, "warm.txt")
        prefix_file(big, warm, 1 << 24)
        kw = dict(scheme="stanford", window_size=args.window_size)
        corpus.preprocess(warm, os.path.join(tmp, "warm"), **kw)             # warm-up: module load, allocator
        torch.cuda.synchronize()
        st = {}
        t = time.perf_counter()
        corpus.preprocess(big, os.path.join(tmp, "stanford"), stats=st, **kw)
        total = time.perf_counter() - t
        res["stanford"] = {"end_to_end_s": total, "pass1_s": st["pass1_s"], "pass2_s": st["pass2_s"], "write_s": st["write_s"],
                           "tokens": st["tokens"], "distinct_tokens": st["distinct_tokens"], "partitions": st["partitions"],
                           "directed_pairs": st["directed_pairs"], "records": st["records"], "bin_bytes": st["bin_bytes"],
                           "text_GBps": nbytes / total / 1e9}
        shutil.rmtree(os.path.join(tmp, "stanford"))
        save(args.out, res)

        # the reference scheme, this tree against --parent, alternating, each in a fresh process
        ref_kw = dict(vocab_size=100_000, coverage=1.0, context_size=5)
        roots = {"this": ROOT}
        if args.parent:
            roots["parent"] = os.path.abspath(args.parent)
        times = {k: [] for k in roots}
        for r in range(args.rounds):
            for name, root in roots.items():
                dest = os.path.join(tmp, "ref_%s_%d" % (name, r))
                st = run_child(root, warm, big, dest, ref_kw)
                times[name].append({k: st[k] for k in ("end_to_end_s", "pass1_s", "pass2_s", "write_s")})
                if r == 0:
                    continue
                shutil.rmtree(dest, ignore_errors=True)
                shutil.rmtree(dest + ".warm", ignore_errors=True)
        ref = {"kw": ref_kw, "runs": times,
               "median_end_to_end_s": {k: float(np.median([x["end_to_end_s"] for x in v])) for k, v in times.items()}}
        if args.parent:
            ref["identical_outputs"] = all(filecmp.cmp(os.path.join(tmp, "ref_this_0", n), os.path.join(tmp, "ref_parent_0", n),
                                                       shallow=False) for n in ("vocab.csv", "vocab.txt", "interaction.csv"))
        res["reference_scheme"] = ref
        res["note"] = ("Stanford GloVe's own CPU tools (vocab_count, cooccur) were not available to run, so there is no "
                       "baseline against them.")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    save(args.out, res)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
