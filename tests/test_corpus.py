"""CPU checks of the streamed corpus preprocessor (glove_tensorflow_b200/corpus.py): the float64 formatter of the csv
writer (glove_format_float64, the host build of the routine the kernel runs) against repr(float), the chunk cutting and
carry logic of the file reader, csv quoting of tokens, the partition count, and argument errors of the new C entries."""
import ctypes
import struct

import numpy as np
import pytest

from glove_tensorflow_b200 import corpus
from glove_tensorflow_b200.data_utils import _HEAD


def _fmt(lib, x):
    buf, n = ctypes.create_string_buffer(32), ctypes.c_int32()
    assert lib.glove_format_float64(float(x), buf, 32, ctypes.byref(n)) == 0
    return buf.raw[:n.value].decode()


def _bits_to_f64(b):
    return struct.unpack("<d", struct.pack("<Q", int(b)))[0]


def special_bit_patterns():
    """±0, every power of two and ten in range, the neighbourhood of 2^53, both extremes and the layout switches."""
    xs = [0.0, -0.0, 5e-324, -5e-324, 2.2250738585072014e-308, 2.225073858507201e-308, 1.7976931348623157e308,
          -1.7976931348623157e308, float("inf"), float("-inf"), float("nan"), 2.0, 1e-05, 1e16, 1.2345678901234568e+17]
    xs += [2.0 ** p for p in range(-1074, 1024)] + [float("1e%d" % p) for p in range(-323, 309)]
    for c in (1e-5, 1e-4, 1e15, 1e16, 2.0 ** 53):
        xs += list(np.nextafter(np.float64(c), -np.inf, dtype=np.float64) * np.ones(1)) + [np.nextafter(c, np.inf)]
        xs += [float(np.nextafter(np.nextafter(c, 0), 0)), float(np.nextafter(np.nextafter(c, np.inf), np.inf))]
    xs += [float(2 ** 53 + k) for k in range(-4, 5)]
    return [struct.unpack("<Q", struct.pack("<d", float(x)))[0] for x in xs]


def random_bit_patterns(n, seed=2026):
    """n patterns with uniformly random exponent fields (every exponent, subnormals and NaN/inf included) and mantissas."""
    rng = np.random.default_rng(seed)
    m = rng.integers(0, 1 << 52, n, dtype=np.uint64)
    e = rng.integers(0, 2048, n, dtype=np.uint64)
    s = rng.integers(0, 2, n, dtype=np.uint64)
    return (s << np.uint64(63)) | (e << np.uint64(52)) | m


def test_format_float64_equals_repr():
    from glove_tensorflow_b200 import _lib
    lib = _lib.lib
    patterns = [int(b) for b in random_bit_patterns(1_000_000)] + special_bit_patterns()
    for b in patterns:
        x = _bits_to_f64(b)
        s = _fmt(lib, x)
        assert s == repr(x), (hex(b), s, repr(x))
        if x == x:
            assert struct.pack("<d", float(s)) == struct.pack("<d", x)


def test_format_float64_layout_and_capacity():
    from glove_tensorflow_b200 import _lib
    lib = _lib.lib
    for x, s in ((2.0, "2.0"), (1e-05, "1e-05"), (0.0001, "0.0001"), (1e16, "1e+16"), (1e15, "1000000000000000.0"),
                 (1.2345678901234568e+17, "1.2345678901234568e+17"), (-0.0, "-0.0"), (5e-324, "5e-324"), (1e100, "1e+100")):
        assert _fmt(lib, x) == s
    buf, n = ctypes.create_string_buffer(32), ctypes.c_int32()
    assert lib.glove_format_float64(1.0, buf, 23, ctypes.byref(n)) == _lib.EINVAL


def _chunks(path, chunk):
    bufs = [np.empty(_HEAD + chunk, np.uint8) for _ in range(2)]
    out = []
    for k, lo, hi, origin, final in corpus.text_chunks(str(path), chunk, bufs):
        out.append((bufs[k % 2][lo:hi].tobytes(), origin, final))
    return out


@pytest.mark.parametrize("chunk", [64, 80, 4096, 1 << 20])
def test_text_chunks_cut_at_whitespace_and_carry_the_tail(tmp_path, chunk):
    rng = np.random.default_rng(chunk)
    words = ["w%d" % i for i in range(50)] + ["café", "中文", "x" * 150, "a,b", '"q"']
    seps = [" ", "\n", "\r\n", "\t", " \x0b\x0c ", "\x1c", "\x1f "]
    text = "".join(words[rng.integers(len(words))] + seps[rng.integers(len(seps))] for _ in range(3000)) + "tail"
    raw = text.encode("utf8")
    path = tmp_path / "c.txt"
    path.write_bytes(raw)
    got = _chunks(path, chunk)
    assert got[-1][2] and not any(f for _, _, f in got[:-1])
    tokens = []
    for body, origin, final in got:
        stripped = body.lstrip(b"\n")
        start = origin + len(body) - len(stripped)
        assert raw[start:start + len(stripped)] == stripped           # origin is the file offset of the chunk's text
        if not final:
            assert corpus._SPACE[body[-1]]                            # cut after a whitespace byte
        tokens += body.decode("utf8").split()
    assert tokens == text.split()                                     # tokens that straddle a cut are counted once


def test_text_chunks_crlf_and_no_final_newline(tmp_path):
    path = tmp_path / "c.txt"
    path.write_bytes(b"alpha\r\nbeta\r\ngamma delta")
    got = _chunks(path, 64)
    assert b"".join(b.lstrip(b"\n") for b, _, _ in got).split() == [b"alpha", b"beta", b"gamma", b"delta"]
    path.write_bytes(b"one two\r\n" * 40 + b"last")
    toks = []
    for b, _, _ in _chunks(path, 64):
        toks += b.split()
    assert toks == [b"one", b"two"] * 40 + [b"last"]


def test_text_chunks_refuse_a_token_longer_than_the_carry_area(tmp_path):
    path = tmp_path / "c.txt"
    start = 1000
    path.write_bytes(b"ab " * (start // 3) + b"c" * (start - 3 * (start // 3)) + b"z" * (2 * _HEAD) + b" end" * 100000)
    first = path.read_bytes().index(b"z") - (start - 3 * (start // 3))
    with pytest.raises(ValueError, match="token at byte %d is longer than %d bytes" % (first, _HEAD - 16)):
        _chunks(path, 1 << 16)


def test_csv_quote_is_pandas_quoting():
    import io
    import pandas as pd
    toks = ["a,b", '"q"', "plain", "café", "<UNK>", "na", "x'y", 'a"b,c']
    buf = io.StringIO()
    pd.DataFrame({"t": toks}).to_csv(buf, index=False)
    assert buf.getvalue().split("\n")[1:-1] == [corpus.csv_quote(t) for t in toks]
    assert corpus.csv_quote("a,b") == '"a,b"' and corpus.csv_quote('"q"') == '"""q"""'


def test_partition_count_follows_the_table_bound():
    assert corpus._part_bits(60, 1000, 5, 1 << 27) == 0
    assert corpus._part_bits(100_000, 1_500_000_000, 5, 1 << 27) == 7    # 2 * 1.5e9 * 5 = 1.5e10 directed pairs at most
    assert corpus._part_bits(60, 10 ** 6, 5, 100) == 6                   # 60 * 59 = 3540 pairs / 100 per partition


def test_preprocess_refuses_bad_input_without_a_gpu(tmp_path):
    empty = tmp_path / "empty.txt"
    empty.write_bytes(b"")
    with pytest.raises(ValueError, match="empty corpus"):
        corpus.preprocess(str(empty), str(tmp_path / "out"))
    with pytest.raises(ValueError, match="context_size"):
        corpus.preprocess(str(empty), str(tmp_path / "out"), context_size=9)


def test_corpus_entries_refuse_bad_arguments_without_a_gpu():
    from glove_tensorflow_b200 import _lib
    lib, E = _lib.lib, _lib.EINVAL
    n = ctypes.c_int64()
    u = ctypes.c_int64()
    fake = ctypes.c_void_p(1 << 20)
    counts = np.zeros(8, np.int64)
    # route: null pointers, n = 0, part_bits out of range, capacity < 2n
    assert lib.glove_cooc_route(None, fake, 4, 10, 0, 1, fake, 1 << 20, fake, fake, 8, counts.ctypes.data, None) == E
    assert lib.glove_cooc_route(fake, fake, 0, 10, 0, 1, fake, 1 << 20, fake, fake, 8, counts.ctypes.data, None) == E
    assert lib.glove_cooc_route(fake, fake, 4, 10, 0, 13, fake, 1 << 20, fake, fake, 8, counts.ctypes.data, None) == E
    assert lib.glove_cooc_route(fake, fake, 4, 10, 0, 1, fake, 1 << 20, fake, fake, 7, counts.ctypes.data, None) == E
    assert lib.glove_cooc_route(fake, fake, 4, 10, 0, 1, fake, 1, fake, fake, 8, counts.ctypes.data, None) == _lib.EWORKSPACE
    assert b"2n" in lib.glove_last_error() or b"workspace" in lib.glove_last_error()
    # finish_sorted: n = 0, context 9
    cols = [fake] * 7
    assert lib.glove_cooc_finish_sorted(fake, fake, 0, 10, 5, 10, fake, 100, 0, fake, 1 << 30, *cols, 8, ctypes.byref(n), None) == E
    assert lib.glove_cooc_finish_sorted(fake, fake, 4, 10, 9, 10, fake, 100, 0, fake, 1 << 30, *cols, 8, ctypes.byref(n), None) == E
    # vocab merge: null pointer, n_chunk = 0, a global table without its arrays, pool_used > capacity
    g = [fake] * 5
    assert lib.glove_vocab_merge(None, 0, fake, fake, fake, 4, *g, 0, fake, 0, 16, fake, 1 << 20, *g, 8, ctypes.byref(n),
                                 ctypes.byref(u), None) == E
    assert lib.glove_vocab_merge(fake, 0, fake, fake, fake, 0, *g, 0, fake, 0, 16, fake, 1 << 20, *g, 8, ctypes.byref(n),
                                 ctypes.byref(u), None) == E
    assert lib.glove_vocab_merge(fake, 0, fake, fake, fake, 4, *([None] * 5), 3, fake, 0, 16, fake, 1 << 20, *g, 8,
                                 ctypes.byref(n), ctypes.byref(u), None) == E
    assert lib.glove_vocab_merge(fake, 0, fake, fake, fake, 4, *g, 0, fake, 17, 16, fake, 1 << 20, *g, 8, ctypes.byref(n),
                                 ctypes.byref(u), None) == E
    # csv writer: n = 0, null column, small workspace, formatter capacity
    assert lib.glove_cooc_csv_size(*cols, 0, fake, fake, 1 << 20, ctypes.byref(n), None) == E
    assert lib.glove_cooc_csv_size(None, *cols[1:], 4, fake, fake, 1 << 20, ctypes.byref(n), None) == E
    assert lib.glove_cooc_csv_size(*cols, 4, fake, fake, 1, ctypes.byref(n), None) == _lib.EWORKSPACE
    assert lib.glove_cooc_csv_format(*cols, 4, fake, fake, fake, 1, fake, 100, None) == _lib.EWORKSPACE
    assert lib.glove_format_float64_device(None, 4, fake, fake, None) == E
    assert lib.glove_cooc_route_workspace_bytes(100, 4) >= lib.glove_cooc_route_workspace_bytes(100, 0) > 0
    assert lib.glove_vocab_merge_workspace_bytes(0, 10) > 0 and lib.glove_cooc_csv_workspace_bytes(10) > 0
