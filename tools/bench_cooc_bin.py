"""Stanford GloVe co-occurrence import and writing (csrc/glove_crec.cu, data_utils.load_cooc_bin,
corpus.preprocess(format=...)):

- a seeded table of --records records (16 bytes each) written to a temporary directory;
- glove_cooc_bin_parse alone, timed with CUDA events on a device-resident chunk, as GB/s of its HBM traffic (16 bytes
  read + 16 bytes written per record) against the 7.7 TB/s data-sheet figure;
- load_cooc_bin end to end from a warm page cache;
- ingest_csv of the first --csv-records records of the same table written as interaction.csv (by the preprocessor's
  device csv writer);
- the preprocessor's write stage, csv against stanford, on the seeded Zipf corpus of tools/bench_corpus.py.

The card's name and power limit are read in the same run.  Temporary files are deleted at the end.

    python tools/bench_cooc_bin.py --out profiles/r06_cooc_bin_bench.json
"""
import argparse
import json
import os
import shutil
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

HBM_TBPS = 7.7


def write_table(path, n, V, seed=6, piece=1 << 24):
    from oracle.cooc_bin_oracle import write
    rng = np.random.default_rng(seed)
    with open(path, "wb") as f:
        for s in range(0, n, piece):
            m = min(piece, n - s)
            f.write(write(rng.integers(0, V, m), rng.integers(0, V, m), np.exp(rng.uniform(0, np.log(1e4), m))))


def warm(path):
    with open(path, "rb") as f:
        while f.read(1 << 26):
            pass


def kernel_rate(path, V, n_chunk=1 << 26, reps=20):
    import torch
    from glove_tensorflow_b200 import _lib
    raw = torch.from_numpy(np.fromfile(path, np.uint8, count=16 * n_chunk)).cuda()
    n = raw.numel() // 16
    outs = [torch.empty(n, dtype=dt, device="cuda") for dt in (torch.int32, torch.int32, torch.float32, torch.float32)]
    err = torch.full((1,), -1, dtype=torch.int64, device="cuda")
    st = torch.cuda.current_stream().cuda_stream

    def call():
        _lib.check(_lib.lib.glove_cooc_bin_parse(raw.data_ptr(), n, 0, V, 100.0, 0.75, *[t.data_ptr() for t in outs],
                                                 err.data_ptr(), st), "glove_cooc_bin_parse")
    for _ in range(3):
        call()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for _ in range(reps):
        e0.record()
        call()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1) / 1e3)
    assert int(err.item()) == -1
    t = float(np.median(times))
    return {"records": n, "median_s": t, "min_s": float(min(times)), "max_s": float(max(times)),
            "GBps": 32 * n / t / 1e9, "share_of_hbm_datasheet": 32 * n / t / (HBM_TBPS * 1e12),
            "bytes_per_record": 32, "note": "working set %.1f GB, past the 126 MB L2" % (32 * n / 1e9)}


def write_csv(path, bin_path, n, V):
    """The first n records of the .bin as interaction.csv, formatted on the device (corpus._CsvWriter)."""
    import torch
    from glove_tensorflow_b200 import corpus
    d = corpus._Device("cuda:0", None)
    rec = np.fromfile(bin_path, np.dtype([("w1", "<i4"), ("w2", "<i4"), ("val", "<f8")]), count=n)
    with open(path, "wb") as f:
        w = corpus._CsvWriter(d, f, ["t%d" % i for i in range(V)])
        try:
            for s in range(0, n, 1 << 24):
                r = rec[s:s + (1 << 24)]
                val = torch.from_numpy(r["val"].copy()).cuda()
                cols = [torch.from_numpy(r["w1"] - 1).cuda(), torch.from_numpy(r["w2"] - 1).cuda(),
                        torch.full((len(r),), 10, dtype=torch.int64, device="cuda"), val, val,
                        torch.ones(len(r), dtype=torch.float64, device="cuda"), torch.log(val)]
                w.write(cols, 1 << 22)
        finally:
            w.close()
    return os.path.getsize(path)


def timed(fn, reps):
    import torch
    out = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        out.append(time.perf_counter() - t)
        del r
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=250_000_000)
    ap.add_argument("--csv-records", type=int, default=50_000_000)
    ap.add_argument("--vocab", type=int, default=400_000)
    ap.add_argument("--corpus-gb", type=float, default=8.0)
    ap.add_argument("--out", default="profiles/r06_cooc_bin_bench.json")
    args = ap.parse_args()
    import torch
    from bench_corpus import card, save, write_zipf_corpus
    from glove_tensorflow_b200 import corpus, data_utils
    if not torch.cuda.is_available():
        raise SystemExit("bench_cooc_bin.py needs a GPU")
    res = {"card": card(), "records": args.records, "vocab": args.vocab,
           "table": "seeded: ids uniform in 1..V, val log-uniform in 1..1e4 (seed 6)"}
    tmp = tempfile.mkdtemp(prefix="glove_cooc_bin_bench_")
    try:
        binp = os.path.join(tmp, "cooccurrence.bin")
        t = time.perf_counter()
        write_table(binp, args.records, args.vocab)
        res["bin_bytes"], res["generate_s"] = os.path.getsize(binp), time.perf_counter() - t
        res["kernel"] = kernel_rate(binp, args.vocab)
        save(args.out, res)
        torch.cuda.empty_cache()

        warm(binp)
        ts = timed(lambda: data_utils.load_cooc_bin(binp, args.vocab), 3)
        res["import_end_to_end"] = {"runs_s": ts, "best_s": min(ts), "file_GBps": res["bin_bytes"] / min(ts) / 1e9,
                                    "Mrecords_per_s": args.records / min(ts) / 1e6, "page_cache": "warm"}
        save(args.out, res)
        torch.cuda.empty_cache()

        csvp, vocp = os.path.join(tmp, "interaction.csv"), os.path.join(tmp, "vocab.txt")
        with open(vocp, "w") as f:
            f.write("\n".join("t%d" % i for i in range(args.vocab)))
        n_csv = min(args.csv_records, args.records)
        csv_bytes = write_csv(csvp, binp, n_csv, args.vocab)
        warm(csvp)
        ts = timed(lambda: data_utils.ingest_csv(csvp, vocp), 2)
        res["ingest_csv"] = {"records": n_csv, "csv_bytes": csv_bytes, "runs_s": ts, "best_s": min(ts),
                             "file_GBps": csv_bytes / min(ts) / 1e9, "Mrecords_per_s": n_csv / min(ts) / 1e6,
                             "page_cache": "warm", "note": "the first csv-records records of the same table"}
        os.remove(csvp)
        os.remove(binp)
        save(args.out, res)
        torch.cuda.empty_cache()

        text = os.path.join(tmp, "corpus.txt")
        nbytes = write_zipf_corpus(text, int(args.corpus_gb * 1e9))
        kw = dict(vocab_size=100_000, coverage=1.0, context_size=5)
        res["preprocess"] = {"corpus_bytes": nbytes, "corpus": "tools/bench_corpus.py's seeded Zipf text"}
        for fmt in ("csv", "stanford", "csv", "stanford"):
            st = {}
            t = time.perf_counter()
            corpus.preprocess(text, os.path.join(tmp, fmt), stats=st, format=fmt, **kw)
            run = {"end_to_end_s": time.perf_counter() - t, "write_s": st["write_s"], "records": st["records"],
                   "bytes": st.get("csv_bytes", st.get("bin_bytes"))}
            res["preprocess"].setdefault(fmt, []).append(run)
            shutil.rmtree(os.path.join(tmp, fmt))
            save(args.out, res)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    save(args.out, res)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
