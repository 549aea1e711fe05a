"""Stanford GloVe's trainer (glove.c, one thread) restated for the tests and the benchmark: the records, the links, the
seeded initialisation, one epoch (C, oracle/stanford_glove_oracle.c, in glove.c's or the GPU kernel's arithmetic order),
the epoch cost's fixed-shape sum, and the rows of the vectors file.  TEST / BENCHMARK INFRASTRUCTURE ONLY.

State in glove.c's layout: W and gradsq are float64 [2V, d + 1] (rows V.. are the context vectors, column d the bias).
Records: words int32 [n, 2] = (word1 - 1, word2 - 1), lf float64 [n, 2] = (log(val), f)."""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "stanford_glove_oracle.c")
# -ffp-contract=off: no fused multiply-add unless the source calls fma() (glibc's is correctly rounded)
_CFLAGS = ["-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-Wall", "-shared"]
SUM_THREADS, SUM_PER_THREAD = 256, 32        # csrc/glove_sgd.cu: kSumThreads, kSumChunk / kSumThreads
_lib = None


def build():
    """Compiles the oracle into the temporary directory (the source tree may be read-only), once per source text."""
    tag = hashlib.sha256(open(_SRC, "rb").read() + " ".join(_CFLAGS).encode()).hexdigest()[:16]
    so = os.path.join(tempfile.gettempdir(), "stanford_glove_oracle_%d_%s.so" % (os.getuid(), tag))
    if not os.path.exists(so):
        tmp = "%s.%d.tmp" % (so, os.getpid())
        subprocess.check_call(["/usr/bin/gcc"] + _CFLAGS + ["-o", tmp, _SRC, "-lm"])
        os.replace(tmp, so)
    return so


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
        _lib.sg_oracle_epoch.restype = ctypes.c_int
        _lib.sg_oracle_chain.restype = ctypes.c_int64
    return _lib


def records(raw, x_max=100.0, alpha=0.75):
    """(words, lf) of cooccurrence.bin bytes: ids - 1, log(val), val > x_max ? 1 : (val / x_max) ** alpha (NumPy's
    log / pow; the GPU's differ by at most 1 ulp)."""
    rec = np.frombuffer(raw, np.dtype([("w1", "<i4"), ("w2", "<i4"), ("val", "<f8")]))
    words = np.stack([rec["w1"] - 1, rec["w2"] - 1], 1).astype(np.int32)
    val = rec["val"].astype(np.float64)
    f = np.where(val > x_max, 1.0, np.power(val / x_max, alpha))
    return words, np.stack([np.log(val), f], 1)


def links(words):
    """prev int32 [n, 2]: the last earlier record with the same word1 / word2, -1 if none."""
    n = len(words)
    prev = np.full((n, 2), -1, np.int32)
    for s in range(2):
        order = np.argsort(words[:, s], kind="stable")
        k = words[order, s]
        same = np.zeros(n, bool)
        same[1:] = k[1:] == k[:-1]
        prev[order[1:][same[1:]], s] = order[:-1][same[1:]]
    return prev


def chain(prev):
    """Longest dependency chain over the links, in records."""
    prev = np.ascontiguousarray(prev, np.int32)
    r = lib().sg_oracle_chain(prev.ctypes.data_as(ctypes.c_void_p), ctypes.c_int64(len(prev)))
    if r < 0:
        raise ValueError("a link does not point to an earlier record")
    return int(r)


def splitmix64(z):
    z = np.asarray(z, np.uint64)
    with np.errstate(over="ignore"):
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def init_params(V, d, seed):
    """W float64 [2V, d + 1]: element i (row-major) is (u - 0.5) / d with u = (splitmix64(seed * 0xD1B54A32D192ED03 +
    i * 0x9E3779B97F4A7C15) >> 11) * 2^-53, all arithmetic on uint64 modulo 2^64."""
    i = np.arange(2 * V * (d + 1), dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = splitmix64(np.uint64(seed) * np.uint64(0xD1B54A32D192ED03) + i * np.uint64(0x9E3779B97F4A7C15))
    u = (z >> np.uint64(11)).astype(np.float64) * 2.0 ** -53
    return ((u - 0.5) / d).reshape(2 * V, d + 1)


def epoch(W, G, words, lf, eta=0.05, clip=100.0, order=1, hits=None):
    """One epoch in place on W, G (C-contiguous float64).  Returns the per-record costs (0 for a skipped record).
    ``hits`` (int64 [4], optional) accumulates the branch counts: skipped records, clipped products, records whose
    update sums were not finite, bias steps zeroed by check_nan."""
    assert W.dtype == G.dtype == np.float64 and W.flags.c_contiguous and G.flags.c_contiguous and W.shape == G.shape
    V, d = W.shape[0] // 2, W.shape[1] - 1
    words = np.ascontiguousarray(words, np.int32)
    lf = np.ascontiguousarray(lf, np.float64)
    cost = np.zeros(len(words), np.float64)
    if hits is not None:
        assert hits.dtype == np.int64 and hits.shape == (4,) and hits.flags.c_contiguous
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    rc = lib().sg_oracle_epoch(ctypes.c_int64(V), ctypes.c_int32(d), p(W), p(G), p(words), p(lf),
                               ctypes.c_int64(len(words)), ctypes.c_double(eta), ctypes.c_double(clip),
                               ctypes.c_int32(order), p(cost), None if hits is None else p(hits))
    assert rc == 0
    return cost


def _tree_level(x):
    """The sums of the chunks of SUM_THREADS * SUM_PER_THREAD values: thread t adds the chunk's values t, t + 256, ...
    in ascending order from 0.0, then the 256 partial sums are halved pairwise (s[t] += s[t + h], h = 128 .. 1)."""
    chunk = SUM_THREADS * SUM_PER_THREAD
    m = -(-len(x) // chunk)
    a = np.zeros(m * chunk, np.float64)
    a[:len(x)] = x
    a = a.reshape(m, SUM_PER_THREAD, SUM_THREADS)
    s = np.zeros((m, SUM_THREADS), np.float64)
    for k in range(SUM_PER_THREAD):
        s = s + a[:, k, :]
    h = SUM_THREADS // 2
    while h:
        s = s[:, :h] + s[:, h:2 * h]
        h //= 2
    return s[:, 0]


def kernel_cost(cost):
    """The epoch cost as the GPU sums it (levels of _tree_level until one value, then / n)."""
    x = np.asarray(cost, np.float64)
    while True:
        x = _tree_level(x)
        if len(x) == 1:
            return float(x[0] / np.float64(len(cost)))


def glove_cost(cost):
    """The epoch cost as glove.c sums it: ascending, then / n."""
    t = 0.0
    for c in np.asarray(cost, np.float64).tolist():
        t += c
    return t / len(cost)


def unk_halves(W):
    """glove.c's <unk>: per element the sum over the last m = min(100, V) rows of W / m, ascending from 0.0, for the word
    and the context half."""
    V = W.shape[0] // 2
    m = min(100, V)
    vec, ctx = np.zeros(W.shape[1]), np.zeros(W.shape[1])
    for a in range(V - m, V):
        vec = vec + W[a] / m
        ctx = ctx + W[V + a] / m
    return vec, ctx


def rows(W, model=2, unk=True):
    """float32 rows of the vectors file: model 0 = W and W~ rows with biases, 1 = W, 2 = W + W~ in float64."""
    V, d = W.shape[0] // 2, W.shape[1] - 1
    a, c = W[:V], W[V:]
    if unk:
        vec, ctx = unk_halves(W)
        a, c = np.vstack([a, vec]), np.vstack([c, ctx])
    out = {0: np.hstack([a, c]), 1: a[:, :d], 2: a[:, :d] + c[:, :d]}[model]
    return out.astype(np.float32)
