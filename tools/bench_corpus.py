"""Streamed corpus preprocessing on a seeded Zipf corpus (glove_tensorflow_b200/corpus.py): per pass the end-to-end and
the kernel time, text GB/s, distinct tokens, directed pairs, records and csv bytes/s; on a prefix that the in-memory path
accepts, text8.process_data + save_data timed next to the streamed path with identical outputs.  The corpus is written to
a temporary directory outside --out and deleted at the end.  The card's name and power limit are read in the same run.

    python tools/bench_corpus.py --gb 8 --prefix-gb 1.5 --out profiles/r05_corpus_bench.json
"""
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

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                       check=True).stdout.strip().split("\n")[0]
    name, power = [x.strip() for x in q.split(",")]
    return {"gpu": name, "power_limit": power}


def write_zipf_corpus(path, nbytes, vocab=500_000, seed=5, distinct_bytes=1 << 30):
    """Zipf(1.1) word ranks over `vocab` synthetic words, a newline after every 8M words: distinct_bytes of seeded text,
    then that text again until nbytes (generating text in Python is slower than preprocessing it)."""
    rng = np.random.default_rng(seed)
    words = np.array([("t%x" % (i * 2654435761 % (1 << 32))).encode() for i in range(vocab)], dtype=object)
    blocks, done = [], 0
    while done < min(nbytes, distinct_bytes):
        r = rng.zipf(1.1, 8_000_000)
        blocks.append(b" ".join(words[r[r <= vocab] - 1]) + b"\n")
        done += len(blocks[-1])
    done = 0
    with open(path, "wb") as f:
        while done < nbytes:
            for b in blocks:
                f.write(b)
                done += len(b)
    return done


def prefix_file(src, dst, nbytes):
    with open(src, "rb") as f:
        data = f.read(nbytes)
    data = data[:max(data.rfind(b" "), data.rfind(b"\n")) + 1]
    with open(dst, "wb") as f:
        f.write(data)
    return len(data)


def kernel_seconds(fn):
    """Device time of the kernels launched inside the corpus.* ranges of one call of fn, per range."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
    ranges = [(e.name, e.time_range.start, e.time_range.end) for e in prof.events() if e.name.startswith("corpus.")
              and e.device_type == torch.autograd.DeviceType.CPU]
    out = {name: 0.0 for name, _, _ in ranges}
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA or "Memcpy" in e.name or "Memset" in e.name:
            continue
        for name, t0, t1 in ranges:
            if t0 <= e.time_range.start <= t1:
                out[name] += e.time_range.elapsed_us() / 1e6
                break
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gb", type=float, default=8.0)
    ap.add_argument("--prefix-gb", type=float, default=1.5)
    ap.add_argument("--vocab-size", type=int, default=100_000)
    ap.add_argument("--context-size", type=int, default=5)
    ap.add_argument("--out", default="profiles/r05_corpus_bench.json")
    args = ap.parse_args()
    import torch
    from glove_tensorflow_b200 import corpus, text8
    if not torch.cuda.is_available():
        raise SystemExit("bench_corpus.py needs a GPU")
    res = {"card": card(), "context_size": args.context_size, "vocab_size": args.vocab_size}
    tmp = tempfile.mkdtemp(prefix="glove_corpus_bench_")
    try:
        big = os.path.join(tmp, "corpus.txt")
        t = time.perf_counter()
        nbytes = write_zipf_corpus(big, int(args.gb * 1e9))
        res["corpus_bytes"], res["generate_s"] = nbytes, time.perf_counter() - t
        res["corpus"] = "Zipf(1.1) over 500,000 words, seed 5: 1 GiB of seeded text repeated to the size"
        kw = dict(vocab_size=args.vocab_size, coverage=1.0, context_size=args.context_size)

        # prefix: the in-memory path and the streamed one, same outputs
        small = os.path.join(tmp, "prefix.txt")
        pbytes = prefix_file(big, small, int(args.prefix_gb * 1e9))
        warm = os.path.join(tmp, "warm.txt")
        prefix_file(big, warm, 1 << 24)
        corpus.preprocess(warm, os.path.join(tmp, "warm"), **kw)             # warm-up: module load, allocator
        torch.cuda.synchronize()
        t = time.perf_counter()
        with open(small) as f:
            text = f.read()
        text8.save_data(text8.process_data(text, **kw), os.path.join(tmp, "ref"))
        del text
        t_ref = time.perf_counter() - t
        st = {}
        t = time.perf_counter()
        corpus.preprocess(small, os.path.join(tmp, "new"), stats=st, **kw)
        t_new = time.perf_counter() - t
        same = all(filecmp.cmp(os.path.join(tmp, "ref", n), os.path.join(tmp, "new", n), shallow=False)
                   for n in ("vocab.csv", "vocab.txt", "interaction.csv"))
        res["prefix"] = {"bytes": pbytes, "in_memory_s": t_ref, "streamed_s": t_new, "speedup": t_ref / t_new,
                         "identical_outputs": same, "records": st["records"]}
        shutil.rmtree(os.path.join(tmp, "ref"))
        save(args.out, res)

        # the whole corpus, end to end
        st = {}
        t = time.perf_counter()
        _, n = corpus.preprocess(big, os.path.join(tmp, "full"), stats=st, **kw)
        total = time.perf_counter() - t
        res["full"] = {"end_to_end_s": total, "stats": st}
        save(args.out, res)
        ks = kernel_seconds(lambda: corpus.preprocess(big, os.path.join(tmp, "prof"), **kw))
        res["full"] = {
            "end_to_end_s": total,
            "pass1": {"end_to_end_s": st["pass1_s"], "kernel_s": ks.get("corpus.pass1"), "text_GBps": nbytes / st["pass1_s"] / 1e9,
                      "tokens": st["tokens"], "distinct_tokens": st["distinct_tokens"]},
            "pass2": {"end_to_end_s": st["pass2_s"], "kernel_s": ks.get("corpus.pass2"), "text_GBps": nbytes / st["pass2_s"] / 1e9,
                      "partitions": st["partitions"], "directed_pairs": st["directed_pairs"]},
            "write": {"end_to_end_s": st["write_s"], "kernel_s": ks.get("corpus.write"), "records": n,
                      "csv_bytes": st["csv_bytes"], "csv_GBps": st["csv_bytes"] / st["write_s"] / 1e9},
            "note": "kernel_s: device time of the kernels inside each pass, from a second, profiled run",
        }
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    save(args.out, res)
    print(json.dumps(res))


def save(path, res):
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
