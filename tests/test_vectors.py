"""CPU checks of the word-vector text format: the float32 -> shortest decimal formatter (glove_format_float32, the host
build of the routine the export kernel runs) against NumPy's Dragon4 "unique" mode and the decimal parser, the plain-
Python reader of oracle/vectors_oracle.py on hand-made files, the host-side header reader, argument errors of the new C
entries, and CLI argument validation."""
import ctypes

import numpy as np
import pytest

from oracle import vectors_oracle as vo


def _fmt(lib, x):
    buf, n = ctypes.create_string_buffer(16), ctypes.c_int32()
    assert lib.glove_format_float32(float(x), buf, 16, ctypes.byref(n)) == 0
    return buf.raw[:n.value].decode()


def _bit_patterns():
    rng = np.random.default_rng(2024)
    parts = [rng.integers(0, 2 ** 32, 1_000_000, dtype=np.uint64).astype(np.uint32)]    # random over all exponents
    parts.append(rng.integers(1, 1 << 23, 20_000, dtype=np.uint32))                    # subnormals
    pw = (np.arange(1, 255, dtype=np.uint32) << 23)                                     # every normal power of two ...
    parts += [pw, pw | 0x80000000, (1 << np.arange(23, dtype=np.uint32)).astype(np.uint32)]   # ... and subnormal one
    parts.append(np.array([0, 0x80000000, 0x7f7fffff, 0xff7fffff, 1, 0x80000001, 0x00800000, 0x007fffff], np.uint32))
    ints = np.arange(2 ** 24 - 300, 2 ** 24 + 300, dtype=np.float64)                   # the integers near 2^24
    parts.append(ints.astype(np.float32).view(np.uint32))
    for E in (-6, -5, 8, 9):                                                           # around the layout switch
        lo, hi = np.float32(10.0 ** E), np.float32(10.0 ** (E + 1))
        a, b = int(lo.view(np.uint32)), int(hi.view(np.uint32))
        parts += [np.arange(a - 50, a + 50, dtype=np.uint32), np.arange(b - 50, b + 50, dtype=np.uint32),
                  rng.integers(a, b, 5000, dtype=np.uint64).astype(np.uint32)]
    bits = np.concatenate(parts)
    return bits[(bits & 0x7f800000) != 0x7f800000]


def test_format_float32_is_shortest_round_trip():
    from glove_tensorflow_b200 import _lib
    lib = _lib.lib
    bits = _bit_patterns()
    assert len(bits) > 1_000_000
    vals = bits.view(np.float32)
    out = ctypes.c_float()
    for b, x in zip(bits.tolist(), vals.tolist()):
        x32 = np.float32(x)
        s = _fmt(lib, x32)
        assert s == vo.format_f32(x32), hex(b)
        assert len(s) <= 16
        t = s.encode()
        assert lib.glove_parse_float32(t, len(t), ctypes.byref(out)) == 0
        assert np.float32(out.value).view(np.uint32) == b, (hex(b), s)


def test_format_float32_special_values_and_layout():
    from glove_tensorflow_b200 import _lib
    lib = _lib.lib
    cases = [(0.0, "0"), (-0.0, "-0"), (float("inf"), "inf"), (float("-inf"), "-inf"), (float("nan"), "nan"), (1.0, "1"),
             (1e-5, "0.00001"), (-0.05123, "-0.05123"), (123456789.0, "123456790"), (1e9, "1e+09"),
             (1.2345e-6, "1.2345e-06"), (1e-45, "1e-45"), (3.4028234663852886e38, "3.4028235e+38"),
             (343126.125, "343126.12"), (0.1, "0.1")]
    for x, want in cases:
        assert _fmt(lib, np.float32(x)) == want, x
    nan = np.array([0x7fc00001, 0xffc00000, 0x7f800001], np.uint32).view(np.float32)
    assert [_fmt(lib, v) for v in nan] == ["nan"] * 3
    buf, n = ctypes.create_string_buffer(16), ctypes.c_int32()
    assert lib.glove_format_float32(1.0, buf, 15, ctypes.byref(n)) == _lib.EINVAL


@pytest.mark.parametrize("name", sorted(vo.handmade_files()))
def test_oracle_reads_the_handmade_files(name):
    want = {
        "header": ([b"the", b"nan", b"1"], [[0.1, -0.2], [1e-3, 4], [-0.0, 0]]),
        "header_crlf_blank_lines": ([b"x", b"\ty"], [[1, 2, 3], [4, 5, 6]]),
        "no_header_mixed": ([b"a", b"-0", b"inf", b"word with  spaces", "été".encode(), b'"quoted"', b"  lead", b"a"],
                            [[0.5, 1.5], [2, 3], [-100, 0.5], [1, 2], [3, 4], [7, 8], [9, 10], [5, 6]]),
        "number_forms": ([b"x", b"y", b"z", b"w"],
                         [[1, -2.5e-3, 7], [1e38, 3.4028234663852886e38, -0.0],
                          [1.401298464324817e-45, 1.401298464324817e-6, 1.2345678901234568e23], [1, 0.5, -125]]),
    }[name]
    words, rows = vo.read_vectors(vo.handmade_files()[name])
    assert words == want[0]
    np.testing.assert_array_equal(rows.view(np.uint32), np.array(want[1], np.float32).view(np.uint32))


@pytest.mark.parametrize("case", vo.malformed_files(), ids=[c[0] for c in vo.malformed_files()])
def test_oracle_names_the_lowest_bad_line(case):
    name, data, dim, line = case
    with pytest.raises(vo.VectorsFormatError) as e:
        vo.read_vectors(data, dim)
    assert e.value.line == line, str(e.value)


def test_oracle_format_round_trips():
    rng = np.random.default_rng(5)
    rows = rng.normal(0, 0.4, (50, 7)).astype(np.float32)
    rows[0, :3] = [0.0, -0.0, np.float32(1e-45)]
    words = [b"w%d" % i for i in range(50)]
    words[3] = b"two words"
    for header in (False, True):
        w, r = vo.read_vectors(vo.format_vectors(words, rows, header))
        assert w == words
        np.testing.assert_array_equal(r.view(np.uint32), rows.view(np.uint32))


def test_read_header(tmp_path):
    from glove_tensorflow_b200 import vectors
    p = tmp_path / "v.txt"
    for data, dim, want in [(b"3 2\na 1 2\n", None, (3, 2, 4, 2)), (b"\n\na 1 2 3\n", None, (None, 3, 0, 1)),
                            (b"a 1 2 3\n", 3, (None, 3, 0, 1)), (b"12 300\r\n", None, (12, 300, 8, 2))]:
        p.write_bytes(data)
        assert vectors.read_header(str(p), dim) == want
    for data, dim, match in [(b"3 2\n", 4, "line 1: the header declares d = 2"), (b"\na 1\n", None, "line 2: d = 1"),
                             (b"2 511\n", None, "line 1: d = 511"), (b"\n \n", None, "no vector line")]:
        p.write_bytes(data)
        with pytest.raises(ValueError, match=match):
            vectors.read_header(str(p), dim)


def test_vector_entries_refuse_bad_arguments_without_a_gpu():
    from glove_tensorflow_b200 import _lib
    lib = _lib.lib
    n, c = ctypes.c_int64(), ctypes.c_int64()
    buf = ctypes.create_string_buffer(64)
    assert lib.glove_vectors_index(None, 16, buf, 64, ctypes.byref(n), None) == _lib.EINVAL
    assert lib.glove_vectors_index(buf, 0, buf, 64, ctypes.byref(n), None) == _lib.EINVAL
    args = lambda d, ld, text=buf: (text, 16, 1, d, 0, buf, 64, buf, ld, 1, buf, buf, 1, ctypes.byref(n), ctypes.byref(c), None)
    assert lib.glove_vectors_parse(*args(1, 8)) == _lib.EINVAL
    assert b"d = 1" in lib.glove_last_error()
    assert lib.glove_vectors_parse(*args(511, 512)) == _lib.EINVAL
    assert lib.glove_vectors_parse(*args(8, 4)) == _lib.EINVAL
    assert lib.glove_vectors_parse(*args(8, 8, None)) == _lib.EINVAL
    assert lib.glove_vectors_format_size(buf, 8, 1, 4, buf, buf, 64, ctypes.byref(n), None) == _lib.EINVAL
    assert lib.glove_vectors_format_size(buf, 8, 8, 0, buf, buf, 64, ctypes.byref(n), None) == _lib.EINVAL
    assert lib.glove_vectors_format(buf, 8, 8, 4, None, buf, buf, 64, buf, 64, None) == _lib.EINVAL
    assert lib.glove_vectors_workspace_bytes(1 << 20, 1000) > lib.glove_vectors_workspace_bytes(1 << 20, 0) > 0


def test_evaluate_cli_argument_validation(tmp_path, capsys):
    from glove_tensorflow_b200 import evaluate_embeddings as ev
    v = str(tmp_path / "v.txt")
    for argv, msg in [(["--job-dir", "j", "--vectors-txt", v], "not allowed with"),
                      ([], "one of the arguments"),
                      (["--vectors-txt", v], "--vectors-txt needs --output-json"),
                      (["--vectors-txt", v, "--output-json", "o", "--vectors", "row"], "--job-dir only"),
                      (["--vectors-txt", v, "--output-json", "o", "--checkpoint", "c"], "--job-dir only"),
                      (["--job-dir", "j", "--dim", "3"], "--vectors-txt only")]:
        with pytest.raises(SystemExit):
            ev.main(argv)
        assert msg in capsys.readouterr().err, argv

