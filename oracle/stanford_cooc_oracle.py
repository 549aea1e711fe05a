"""Stanford GloVe's vocab_count and cooccur in plain Python with exact sums: the oracle of
``corpus.preprocess(scheme="stanford")`` (DESIGN.md §3, "Stanford GloVe preprocessing").  Nothing in the package imports
it.

The contract it restates:

- Tokens are separated by space, tab and '\\n'; a '\\r' directly before '\\n' belongs to the line end.
- A file holding any other '\\r', a '\\v', a '\\f', a byte 0x1c-0x1f or a non-ASCII separator that str.split() knows is
  refused, naming the lowest such byte offset.  A token ``<unk>`` is refused, naming its first offset.
- Vocabulary: counts over all tokens; count >= min_count; by count descending, ties in byte order; the first max_vocab
  (0: all).  Token id = rank, record id = rank + 1.
- Words outside the vocabulary are removed before windowing.  For kept words w1 (left) and w2 (right) on one line at
  distance 1 <= k <= window, (w1, w2) gets 1/k (or 1 without distance weighting) and, when symmetric, (w2, w1) gets the
  same; self pairs are kept; every pair is written.
- val is the exact sum rounded once to float64 (here: a Fraction converted by float())."""
import re
from fractions import Fraction

import numpy as np

_REFUSED = re.compile(rb"[\x0b\x0c\x1c-\x1f]|\r(?!\n)")
_UNICODE_SPACE = re.compile(rb"\xc2[\x85\xa0]|\xe1\x9a\x80|\xe2\x80[\x80-\x8a\xa8\xa9\xaf]|\xe2\x81\x9f|\xe3\x80\x80")
_TOKEN = re.compile(rb"\n|[^ \t\r\n]+")


def check(data):
    """Raises ValueError("byte N: ...") for the lowest refused byte or the first ``<unk>``."""
    bad = [m.start() for m in (_REFUSED.search(data), _UNICODE_SPACE.search(data)) if m is not None]
    if bad:
        raise ValueError("byte %d: refused" % min(bad))
    for m in _TOKEN.finditer(data):
        if m.group() == b"<unk>":
            raise ValueError("byte %d: <unk>" % m.start())


def lines(data):
    """The corpus as a list of lines, each a list of tokens (bytes)."""
    check(data)
    out = [[]]
    for m in _TOKEN.finditer(data):
        if m.group() == b"\n":
            out.append([])
        else:
            out[-1].append(m.group())
    return out


def vocab(data, min_count=1, max_vocab=0):
    """[(token bytes, count)] in id order."""
    counts = {}
    for line in lines(data):
        for t in line:
            counts[t] = counts.get(t, 0) + 1
    kept = sorted(((t, c) for t, c in counts.items() if c >= min_count), key=lambda tc: (-tc[1], tc[0]))
    return kept[:max_vocab] if max_vocab else kept


def vocab_txt(voc):
    """vocab.txt as vocab_count prints it."""
    return b"".join(t + b" %d\n" % c for t, c in voc)


def cooccur(data, voc, window=15, symmetric=True, distance_weighting=True):
    """{(id1, id2): exact Fraction sum}, 0-based ids."""
    ids = {t: i for i, (t, _) in enumerate(voc)}
    table = {}
    for line in lines(data):
        kept = [ids[t] for t in line if t in ids]
        for j, w2 in enumerate(kept):
            for k in range(1, min(window, j) + 1):
                w1 = kept[j - k]
                v = Fraction(1, k) if distance_weighting else Fraction(1)
                table[(w1, w2)] = table.get((w1, w2), 0) + v
                if symmetric:
                    table[(w2, w1)] = table.get((w2, w1), 0) + v
    return table


def records(table):
    """The table as sorted arrays (row, col, val): 0-based ids, val the exactly rounded float64 sum."""
    keys = sorted(table)
    row = np.array([k[0] for k in keys], np.int32)
    col = np.array([k[1] for k in keys], np.int32)
    val = np.array([float(table[k]) for k in keys], np.float64)
    return row, col, val
