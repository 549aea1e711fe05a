"""CPU checks of the Stanford GloVe preprocessing scheme: the oracle (oracle/stanford_cooc_oracle.py) against a literal
transcription of Stanford's vocab_count.c / cooccur.c loops on seeded corpora, hand-made cases of the contract, the
host vocabulary rule, the argument checks of preprocess(scheme="stanford") and of the new C entries."""
import ctypes
from fractions import Fraction

import numpy as np
import pytest

from glove_tensorflow_b200 import corpus
from oracle import stanford_cooc_oracle as so


# ---- a literal transcription of Stanford GloVe's C loops (common.c get_word, vocab_count.c, cooccur.c) -------------
def _get_word(data, pos):
    """get_word: (word, flag, pos); flag 1 = a newline (or EOF) before any byte of a word.  pos > len(data): feof."""
    word = bytearray()
    while True:
        ch = data[pos] if pos < len(data) else -1
        pos += 1
        if ch == 13:
            continue
        if not word and ch in (10, -1):
            return b"", 1, pos
        if not word and ch in (32, 9):
            continue
        if ch in (-1, 32, 9, 10):
            if ch == 10:
                pos -= 1                          # ungetc: the newline ends the line on the next call
            break
        word.append(ch)
    return bytes(word), 0, pos


def _vocab_count_c(data, min_count, max_vocab):
    counts, pos = {}, 0
    while pos <= len(data):                       # while (!feof(fid))
        w, nl, pos = _get_word(data, pos)
        if nl:
            continue
        counts[w] = counts.get(w, 0) + 1
    voc = sorted(counts.items(), key=lambda wc: (-wc[1], wc[0]))      # CompareVocabTie: count, then strcmp
    if 0 < max_vocab < len(voc):
        voc = voc[:max_vocab]
    out = []
    for w, c in voc:
        if c < min_count:
            break
        out.append((w, c))
    return out


def _cooccur_c(data, voc, window, symmetric, distance_weighting):
    """{(w1 - 1, w2 - 1): (double sum, count)} in cooccur.c's loop order."""
    ids = {w: i + 1 for i, (w, _) in enumerate(voc)}
    history, j, pos, table = [0] * window, 0, 0, {}

    def add(a, b, v):
        s, n = table.get((a - 1, b - 1), (0.0, 0))
        table[(a - 1, b - 1)] = (s + v, n + 1)
    while True:
        w, flag, pos = _get_word(data, pos)
        if pos > len(data):                       # if (feof(fid)) break;
            break
        if flag == 1:
            j = 0
            continue
        if w not in ids:
            continue
        w2 = ids[w]
        for k in range(j - 1, (j - window if j > window else 0) - 1, -1):
            w1 = history[k % window]
            v = 1.0 / (j - k) if distance_weighting else 1.0
            add(w1, w2, v)
            if symmetric:
                add(w2, w1, v)
        history[j % window] = w2
        j += 1
    return table


def _random_corpus(rng):
    n_words = int(rng.integers(3, 40))
    words = [b"w%d" % i for i in range(n_words)]
    p = 1.0 / np.arange(1, n_words + 1) ** rng.uniform(0.5, 1.5)
    out = []
    for _ in range(int(rng.integers(1, 30))):
        n = int(rng.choice([0, 0, 1, 2, 3, 5, 8, 13, 20]))
        picks = rng.choice(n_words, size=n, p=p / p.sum())
        if n > 3 and rng.random() < 0.3:
            picks[1:3] = picks[0]                 # repeated words: self pairs
        seps = [rng.choice([b" ", b"  ", b"\t", b" \t "]) for _ in range(n)]
        out.append(b"".join(words[i] + s for i, s in zip(picks, seps)).rstrip() + rng.choice([b"\n", b"\r\n", b" \n"]))
    return b"".join(out)


def test_oracle_equals_the_c_loops_on_seeded_corpora():
    rng = np.random.default_rng(2024)
    for case in range(300):
        data = _random_corpus(rng)
        window = case % 15 + 1
        symmetric, weighting = bool(case % 2), bool(case // 2 % 2)
        min_count = int(rng.choice([1, 1, 2, 3]))
        max_vocab = int(rng.choice([0, 0, 3, 10]))
        voc_c = _vocab_count_c(data, min_count, max_vocab)
        voc = so.vocab(data, min_count, max_vocab)
        if max_vocab == 0:                        # with a cut Stanford's survivors of a tie are arbitrary: sets differ
            assert voc == voc_c, case
        else:
            assert [c for _, c in voc] == [c for _, c in voc_c], case
            voc_c = voc
        want = _cooccur_c(data, voc, window, symmetric, weighting)
        got = so.cooccur(data, voc, window, symmetric, weighting)
        assert set(got) == set(want), case
        for key, (s, n) in want.items():
            if not weighting:
                assert got[key] == n, (case, key)
            assert abs(float(got[key]) - s) <= 1e-13 * s, (case, key)


def test_oracle_hand_made_cases():
    # a self pair doubled (symmetric), once (asymmetric)
    voc = so.vocab(b"a a\n")
    assert so.cooccur(b"a a\n", voc, 5) == {(0, 0): Fraction(2)}
    assert so.cooccur(b"a a\n", voc, 5, symmetric=False) == {(0, 0): Fraction(1)}
    # OOV words take no position: x and y are cut by min_count, so a and b are at distance 1
    data = b"a x y b\na b\n"
    voc = so.vocab(data, min_count=2)
    assert [t for t, _ in voc] == [b"a", b"b"]
    assert so.cooccur(data, voc, 1, symmetric=False) == {(0, 1): Fraction(2)}
    # a window cut by a newline and by CRLF
    for data in (b"a b\nc d\n", b"a b\r\nc d\r\n"):
        voc = so.vocab(data)
        t = so.cooccur(data, voc, 15, symmetric=False, distance_weighting=False)
        names = {i: w for i, (w, _) in enumerate(voc)}
        assert {(names[a], names[b]) for a, b in t} == {(b"a", b"b"), (b"c", b"d")}
    # distance weighting: 1/k over kept words
    voc = so.vocab(b"a b c\n")
    t = so.cooccur(b"a b c\n", voc, 2, symmetric=False)
    assert t[(0, 2)] == Fraction(1, 2) and t[(0, 1)] == 1 and t[(1, 2)] == 1
    # min_count exactly at a count keeps the word
    assert [t for t, _ in so.vocab(b"a a b b b c\n", min_count=2)] == [b"b", b"a"]
    # a max_vocab cut inside a tie keeps the byte-order first
    assert so.vocab(b"z y x z y x w\n", max_vocab=2) == [(b"x", 2), (b"y", 2)]
    # refusals name the byte offset
    for data, off in ((b"ab <unk> c\n", 3), (b"ab c\rd\n", 4), (b"ab\x0bc\n", 2), (b"a\r\nb\r", 4), (b"ab\x1fc\n", 2),
                      (b"a b\x0c\n", 3)):
        with pytest.raises(ValueError, match="byte %d:" % off):
            so.check(data)


def test_host_vocabulary_equals_the_oracle():
    rng = np.random.default_rng(5)
    for case in range(50):
        data = _random_corpus(rng)
        toks = [t for line in so.lines(data) for t in line]
        distinct = list(dict.fromkeys(toks))
        counts = np.array([toks.count(t) for t in distinct], np.int64)
        min_count, max_vocab = case % 3 + 1, [0, 2, 5][case % 3]
        got = corpus.stanford_vocab([t.decode() for t in distinct], counts, min_count, max_vocab)
        want = so.vocab(data, min_count, max_vocab)
        assert got[0] == [t.decode() for t, _ in want] and got[1].tolist() == [c for _, c in want]
    # byte order, not code-point-insensitive or locale order
    assert corpus.stanford_vocab(["b", "B", "é", "a"], np.array([1, 1, 1, 1]))[0] == ["B", "a", "b", "é"]


def test_stanford_arguments_are_refused_without_a_gpu(tmp_path):
    p = tmp_path / "c.txt"
    p.write_bytes(b"a b\n")
    for w in (0, 16):
        with pytest.raises(ValueError, match="window_size must be 1..15"):
            corpus.preprocess(str(p), str(tmp_path / "o"), scheme="stanford", window_size=w)
    with pytest.raises(ValueError, match="min_count"):
        corpus.preprocess(str(p), str(tmp_path / "o"), scheme="stanford", min_count=0)
    with pytest.raises(ValueError, match="scheme"):
        corpus.preprocess(str(p), str(tmp_path / "o"), scheme="glove")
    # the reference scheme keeps its own limit, whatever the window
    with pytest.raises(ValueError, match="context_size"):
        corpus.preprocess(str(p), str(tmp_path / "o"), context_size=9, window_size=15)


def test_partition_bound_counts_the_diagonal():
    assert corpus._part_bits(60, 10 ** 6, 5, 100, diagonal=True) == 6       # 3600 / 100
    assert corpus._part_bits(64, 10 ** 6, 5, 1024, diagonal=True) == 2      # 4096 / 1024, where 64 * 63 needs 2 as well
    assert corpus._part_bits(2, 10 ** 6, 5, 2, diagonal=True) == 1 and corpus._part_bits(2, 10 ** 6, 5, 2) == 0


def test_numerator_bound():
    # window 15: lcm 360360, sum_k 360360 / k = 1195757; symmetric doubles it
    assert corpus._stanford_numerator_bound(10, 15, True, True) == 10 * 1195757 * 2
    assert corpus._stanford_numerator_bound(10, 15, False, False) == 150
    assert corpus._stanford_numerator_bound(4 * 10 ** 12, 15, True, True) > 2 ** 63 > \
        corpus._stanford_numerator_bound(4 * 10 ** 12, 15, True, False)


def test_newline_after_the_last_token():
    f = lambda b, before=False: corpus._newline_after_last_token(np.frombuffer(b, np.uint8), before)
    assert f(b"a b \n") and f(b"a\r\n") and f(b"a\n\n ")
    assert not f(b"a\nb ") and not f(b"a b")
    assert not f(b"  ") and f(b"  ", True) and f(b" \n ")
    assert f(b"x" + b" " * 10000 + b"\n" + b" " * 70000)


def test_stanford_entries_refuse_bad_arguments_without_a_gpu():
    from glove_tensorflow_b200 import _lib
    lib, E = _lib.lib, _lib.EINVAL
    n, last = ctypes.c_int64(), ctypes.c_uint32()
    fake = ctypes.c_void_p(1 << 20)
    counts = np.zeros(8, np.int64)
    assert lib.glove_text_refused(None, 16, -1, fake, ctypes.byref(n), None) == E
    assert lib.glove_text_refused(fake, 16, 256, fake, ctypes.byref(n), None) == E
    assert lib.glove_text_refused(ctypes.c_void_p((1 << 20) + 1), 16, -1, fake, ctypes.byref(n), None) == E
    vt = [fake, 1024, fake, fake]
    assert lib.glove_tokens_stream(fake, 0, fake, fake, 4, 0, 0, *vt, fake, 1 << 20, fake, 3, ctypes.byref(n),
                                   ctypes.byref(last), None) == E                        # capacity < n_tokens
    assert lib.glove_tokens_stream(fake, 0, fake, fake, 4, 0, 0, *vt, fake, 1, fake, 4, ctypes.byref(n), ctypes.byref(last),
                                   None) == _lib.EWORKSPACE
    for w in (0, 16):
        assert lib.glove_cooc_chunk_stanford(fake, 4, 4, 10, w, 1, fake, 1 << 30, fake, fake, 64, ctypes.byref(n), None) == E
        assert lib.glove_cooc_finish_stanford(fake, fake, 4, 10, w, 1, fake, 100, 0, fake, 1 << 30, *[fake] * 7, 8,
                                              ctypes.byref(n), None) == E
    assert lib.glove_cooc_chunk_stanford(fake, 4, 4, 10, 15, 1, fake, 1, fake, fake, 64, ctypes.byref(n), None) == _lib.EWORKSPACE
    assert lib.glove_cooc_route_stanford(fake, fake, 4, 10, 0, 1, 1, fake, 1 << 20, fake, fake, 7, counts.ctypes.data,
                                         None) == E                                      # symmetric: capacity 2n
    assert lib.glove_cooc_route_stanford(fake, fake, 4, 10, 0, 1, 0, fake, 1 << 20, fake, fake, 3, counts.ctypes.data,
                                         None) == E                                      # asymmetric: capacity n
    assert lib.glove_cooc_route_stanford(fake, fake, 4, 10, 0, 13, 0, fake, 1 << 20, fake, fake, 8, counts.ctypes.data,
                                         None) == E
    assert lib.glove_tokens_stream_workspace_bytes(100) > 0
