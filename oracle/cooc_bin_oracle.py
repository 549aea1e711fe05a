"""TEST INFRASTRUCTURE ONLY -- NumPy restatement of the Stanford GloVe co-occurrence container, the checker for the CUDA
import and writer (glove_tensorflow_b200/csrc/glove_crec.cu, data_utils.load_cooc_bin, corpus.preprocess(format=...)).
Nothing in the product path may import this file.

The container is what Stanford GloVe's cooccur.c / shuffle.c write and glove.c reads in the default build (real =
double): packed little-endian records ``struct { int32 word1; int32 word2; float64 val; }``, 16 bytes, no header; word1
and word2 are 1-based lines of vocab.txt, whose lines are ``word count`` as vocab_count writes them ("%s %lld\\n").
glove.c fits ``w . w~ + b + b~ - log(val)`` with the weight ``val > x_max ? 1 : (val / x_max)^alpha``."""
import re

import numpy as np

RECORD = np.dtype([("word1", "<i4"), ("word2", "<i4"), ("val", "<f8")])
assert RECORD.itemsize == 16


def read(data, vocab_size, x_max=100.0, alpha=0.75):
    """bytes of a co-occurrence file -> {'row', 'col' (int32, id - 1), 'glove_value' = float32(log(val)),
    'glove_weight' = float32(val >= x_max ? 1 : (val / x_max) ** alpha)}, both computed in float64 and rounded once.

    Raises ValueError naming the lowest offending record, 1-based, and its byte offset: an id outside 1..vocab_size, a
    val that is not finite and > 0, or a truncated last record (which comes after every whole record)."""
    n = len(data) // RECORD.itemsize
    rec = np.frombuffer(data, RECORD, count=n)
    w1, w2, val = rec["word1"].astype(np.int64), rec["word2"].astype(np.int64), rec["val"]
    with np.errstate(invalid="ignore"):
        bad = np.stack([(w1 < 1) | (w1 > vocab_size), (w2 < 1) | (w2 > vocab_size), ~((val > 0) & np.isfinite(val))])
    hit = np.flatnonzero(bad.any(axis=0))
    if len(hit):
        g = int(hit[0])
        kind = int(np.flatnonzero(bad[:, g])[0])
        what = ("word1 id %d outside 1..%d" % (w1[g], vocab_size), "word2 id %d outside 1..%d" % (w2[g], vocab_size),
                "val %r is not a finite value > 0" % float(val[g]))[kind]
        raise ValueError("record %d (byte %d): %s" % (g + 1, 16 * g, what))
    if len(data) % RECORD.itemsize:
        raise ValueError("record %d (byte %d): truncated" % (n + 1, 16 * n))
    with np.errstate(divide="ignore"):
        weight = np.where(val >= x_max, 1.0, np.power(val / x_max, alpha))
    return {"row": (w1 - 1).astype(np.int32), "col": (w2 - 1).astype(np.int32),
            "glove_value": np.log(val).astype(np.float32), "glove_weight": weight.astype(np.float32)}


def write(row, col, value):
    """0-based ids and float64 values -> the bytes of a co-occurrence file (ids + 1)."""
    rec = np.empty(len(row), RECORD)
    rec["word1"] = np.asarray(row, np.int64) + 1
    rec["word2"] = np.asarray(col, np.int64) + 1
    rec["val"] = value
    return rec.tobytes()


def read_vocab(text):
    """Stanford vocab.txt text -> (tokens, counts); every line is ``word count`` (a line that is not raises ValueError
    with its 1-based number)."""
    lines = text.split("\n")
    if lines and lines[-1] == "":
        lines.pop()
    tokens, counts = [], []
    for i, line in enumerate(lines, 1):
        m = re.fullmatch(r"(\S+) ([0-9]+)", line)
        if m is None:
            raise ValueError("line %d: %r" % (i, line))
        tokens.append(m.group(1))
        counts.append(int(m.group(2)))
    return tokens, np.array(counts, np.int64)
