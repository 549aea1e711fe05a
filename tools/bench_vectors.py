"""Word vectors in the GloVe text format (vectors.py, csrc/glove_vectors.cu) at the size of glove.6B.300d: a seeded
synthetic table of V = 400,000 rows of d = 300 N(0, 0.4) values with words of 1-20 bytes, about 1 GB of text.

Arms, in one run, with the card name and power limit read in the same run:
  * export end to end: vectors.write_vectors from the device table to a file (format kernels, device -> pinned copies,
    writer thread, the file write into the page cache); this run also writes the file the other arms read;
  * export kernels only: glove_vectors_format_size + glove_vectors_format of all rows in one call, text on the device;
  * import end to end: vectors.read_vectors of the file, read after one full warm-up read (page cache warm);
  * import kernels only: glove_vectors_index + glove_vectors_parse of the whole file as one device-resident chunk;
  * host: a typical Python loader, ``line.split()`` + ``np.asarray(fields[1:], np.float32)`` per line, on the first
    --host-lines lines of the same file (its rate, not extrapolated to the whole file).
Rates: GB/s of text and M values/s.  Times are medians of --iters runs after one warm-up; every timed region ends in a
device synchronise.  One JSON line is printed (and appended to --out)."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [s.strip() for s in out.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def words_of(V, seed):
    rng = np.random.default_rng(seed)
    lens = rng.integers(1, 21, V)
    letters = rng.integers(ord("a"), ord("z") + 1, int(lens.sum()), dtype=np.uint8).tobytes().decode()
    off = np.concatenate([[0], np.cumsum(lens)])
    return [letters[off[i]:off[i + 1]] for i in range(V)]


def timed(fn, iters):
    import torch
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), ts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--V", type=int, default=400_000)
    ap.add_argument("--d", type=int, default=300)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--host-lines", type=int, default=40_000)
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    a = ap.parse_args()
    import torch
    from glove_tensorflow_b200 import _lib, vectors
    lib, check = _lib.lib, _lib.check
    info = card()
    gen = torch.Generator(device="cuda").manual_seed(0)
    rows = torch.randn(a.V, a.d, generator=gen, device="cuda") * 0.4
    words = words_of(a.V, 0)
    n_vals = a.V * a.d
    st = torch.cuda.current_stream().cuda_stream
    out = {"workload": "word vectors, GloVe text format", "V": a.V, "d": a.d, "card": info}
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "vectors.txt")
        t, ts = timed(lambda: vectors.write_vectors(path, words, rows), a.iters)
        size = os.path.getsize(path)
        out["text_bytes"] = size
        out["export_e2e"] = {"seconds": t, "seconds_all": ts, "GB_per_s": size / t / 1e9, "Mvalues_per_s": n_vals / t / 1e6}

        # kernels only, the whole table in one call
        enc = [w.encode() for w in words]
        woff = torch.from_numpy(np.concatenate([[0], np.cumsum([len(w) for w in enc])]).astype(np.int64)).cuda()
        blob = torch.frombuffer(bytearray(b"".join(enc)), dtype=torch.uint8).cuda()
        ws = torch.empty(lib.glove_vectors_workspace_bytes(0, a.V), dtype=torch.uint8, device="cuda")
        text = torch.empty(size + 16, dtype=torch.uint8, device="cuda")

        def fmt():
            nb = ctypes.c_int64()
            check(lib.glove_vectors_format_size(rows.data_ptr(), a.d, a.d, a.V, woff.data_ptr(), ws.data_ptr(), ws.numel(),
                                                ctypes.byref(nb), st), "format_size")
            check(lib.glove_vectors_format(rows.data_ptr(), a.d, a.d, a.V, blob.data_ptr(), woff.data_ptr(), ws.data_ptr(),
                                           ws.numel(), text.data_ptr(), text.numel(), st), "format")
        t, ts = timed(fmt, a.iters)
        out["export_kernels"] = {"seconds": t, "seconds_all": ts, "GB_per_s": size / t / 1e9, "Mvalues_per_s": n_vals / t / 1e6}
        with open(path, "rb") as f:
            same = f.read() == text[:size].cpu().numpy().tobytes()
        out["export_kernels"]["text_equals_the_file"] = same

        with open(path, "rb") as f:                         # warm the page cache
            while f.read(64 << 20):
                pass
        got = {}

        def imp():
            got["w"], got["r"] = vectors.read_vectors(path)
        t, ts = timed(imp, a.iters)
        exact = len(got["w"]) == a.V and got["w"][:1000] == words[:1000] and torch.equal(got["r"].view(torch.int32), rows.view(torch.int32))
        out["import_e2e"] = {"seconds": t, "seconds_all": ts, "GB_per_s": size / t / 1e9, "Mvalues_per_s": n_vals / t / 1e6,
                             "page_cache": "warm (one full read before the timed runs)", "bit_exact_round_trip": exact}

        n_nl = ctypes.c_int64()
        pws = torch.empty(lib.glove_vectors_workspace_bytes(size, a.V + 1), dtype=torch.uint8, device="cuda")
        dst = torch.empty(a.V, a.d, dtype=torch.float32, device="cuda")
        wst = torch.empty(a.V + 1, dtype=torch.int64, device="cuda")
        wln = torch.empty(a.V + 1, dtype=torch.int32, device="cuda")

        def parse():
            n, c = ctypes.c_int64(), ctypes.c_int64()
            check(lib.glove_vectors_index(text.data_ptr(), size, pws.data_ptr(), pws.numel(), ctypes.byref(n_nl), st), "index")
            check(lib.glove_vectors_parse(text.data_ptr(), size, 1, a.d, n_nl.value, pws.data_ptr(), pws.numel(), dst.data_ptr(),
                                          a.d, a.V, wst.data_ptr(), wln.data_ptr(), 1, ctypes.byref(n), ctypes.byref(c), st),
                  "parse")
        t, ts = timed(parse, a.iters)
        out["import_kernels"] = {"seconds": t, "seconds_all": ts, "GB_per_s": size / t / 1e9, "Mvalues_per_s": n_vals / t / 1e6,
                                 "bit_exact": torch.equal(dst.view(torch.int32), rows.view(torch.int32))}

        t0 = time.perf_counter()
        nv, nb = 0, 0
        with open(path, "rb") as f:
            for i, line in enumerate(f):
                if i == a.host_lines:
                    break
                parts = line.split()
                np.asarray(parts[1:], np.float32)
                nv += len(parts) - 1
                nb += len(line)
        th = time.perf_counter() - t0
        out["host_python_split_asarray"] = {"lines": a.host_lines, "seconds": th, "GB_per_s": nb / th / 1e9,
                                            "Mvalues_per_s": nv / th / 1e6}
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
