"""Word vectors in the GloVe text format on the GPU (csrc/glove_vectors.cu, vectors.py): the export formatter over every
float32 bit pattern, import against the plain-Python oracle (oracle/vectors_oracle.py), error lines of malformed files,
export -> import bit-exactness, and the export / evaluate_embeddings CLIs end to end."""
import ctypes
import json
import os

import numpy as np
import pytest

from oracle import analogy_oracle as ao
from oracle import vectors_oracle as vo

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "text8_small")


def _lib():
    from glove_tensorflow_b200 import _lib
    return _lib


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def _format_dev(rows, words_dev, woff_dev):
    """Device text of the rows (every word given by words_dev / woff_dev), 16-byte aligned."""
    import torch
    L = _lib()
    n, d = rows.shape
    ws = torch.empty(L.lib.glove_vectors_workspace_bytes(0, n), dtype=torch.uint8, device=rows.device)
    nb = ctypes.c_int64()
    L.check(L.lib.glove_vectors_format_size(rows.data_ptr(), rows.stride(0), d, n, woff_dev.data_ptr(), ws.data_ptr(), ws.numel(),
                                            ctypes.byref(nb), _stream()), "format_size")
    text = torch.empty(nb.value + 16, dtype=torch.uint8, device=rows.device)
    L.check(L.lib.glove_vectors_format(rows.data_ptr(), rows.stride(0), d, n, words_dev.data_ptr(), woff_dev.data_ptr(),
                                       ws.data_ptr(), ws.numel(), text.data_ptr(), text.numel(), _stream()), "format")
    return text[:nb.value]


def _parse_dev(text, d, n_cap):
    """Rows parsed back from device text (one final chunk)."""
    import torch
    L = _lib()
    nbytes = text.numel()
    ws = torch.empty(L.lib.glove_vectors_workspace_bytes(nbytes, 0), dtype=torch.uint8, device=text.device)
    n_nl = ctypes.c_int64()
    L.check(L.lib.glove_vectors_index(text.data_ptr(), nbytes, ws.data_ptr(), ws.numel(), ctypes.byref(n_nl), _stream()), "index")
    big = torch.empty(L.lib.glove_vectors_workspace_bytes(nbytes, n_nl.value + 1), dtype=torch.uint8, device=text.device)
    big[:ws.numel()].copy_(ws)
    out = torch.empty(n_cap, d, dtype=torch.float32, device=text.device)
    ws_, wl = torch.empty(n_cap, dtype=torch.int64, device=text.device), torch.empty(n_cap, dtype=torch.int32, device=text.device)
    n, consumed = ctypes.c_int64(), ctypes.c_int64()
    L.check(L.lib.glove_vectors_parse(text.data_ptr(), nbytes, 1, d, n_nl.value, big.data_ptr(), big.numel(), out.data_ptr(), d,
                                      n_cap, ws_.data_ptr(), wl.data_ptr(), 1, ctypes.byref(n), ctypes.byref(consumed),
                                      _stream()), "parse")
    assert n.value == n_cap and consumed.value == nbytes
    return out, ws_, wl


def _words_dev(n):
    import torch
    return (torch.full((n,), ord("w"), dtype=torch.uint8, device="cuda"),
            torch.arange(n + 1, dtype=torch.int64, device="cuda"))


def test_every_float32_is_formatted_and_parsed_back_on_the_device():
    """All 2^32 bit patterns: every finite value comes back bit-exact through the export and import kernels, every NaN
    prints 'nan', the infinities 'inf' / '-inf'."""
    import torch
    d, per = 256, 1 << 26
    rows_n = per // d
    words, woff = _words_dev(rows_n)
    for c in range((1 << 32) // per):
        bits = torch.arange(c * per, (c + 1) * per, dtype=torch.int64, device="cuda")
        bits = torch.where(bits >= (1 << 31), bits - (1 << 32), bits).to(torch.int32)
        finite = (bits & 0x7f800000) != 0x7f800000
        vals = torch.where(finite, bits, torch.zeros_like(bits)).view(torch.float32).view(rows_n, d)
        back, _, _ = _parse_dev(_format_dev(vals, words, woff), d, rows_n)
        assert torch.equal(back.view(-1).view(torch.int32)[finite], bits[finite]), c
    nonfinite = torch.cat([torch.arange(0x7f800000, 0x80000000, dtype=torch.int64, device="cuda"),
                           torch.arange(0xff800000, 0x100000000, dtype=torch.int64, device="cuda")])
    nonfinite = torch.where(nonfinite >= (1 << 31), nonfinite - (1 << 32), nonfinite).to(torch.int32)
    n = nonfinite.numel() // d * d
    text = _format_dev(nonfinite[:n].view(torch.float32).view(-1, d), *_words_dev(n // d)).cpu().numpy().tobytes()
    lines = text.split(b"\n")[:-1]
    half = (n // 2) // d            # rows made of +inf / NaN patterns only, then the negative ones
    assert lines[0] == b"w inf" + b" nan" * (d - 1)
    assert all(ln == b"w" + b" nan" * d for ln in lines[1:half])
    assert lines[half] == b"w -inf" + b" nan" * (d - 1)
    assert all(ln == b"w" + b" nan" * d for ln in lines[half + 1:])


def test_device_text_equals_the_host_formatter():
    import torch
    L = _lib()
    rng = np.random.default_rng(9)
    bits = rng.integers(0, 2 ** 32, 1_010_000, dtype=np.uint64).astype(np.uint32)
    bits = bits[(bits & 0x7f800000) != 0x7f800000][:1_000_000]
    d = 250
    text = _format_dev(torch.from_numpy(bits.view(np.float32).reshape(-1, d)).cuda(), *_words_dev(len(bits) // d))
    buf, m = ctypes.create_string_buffer(16), ctypes.c_int32()
    host = []
    for x in bits.view(np.float32).tolist():
        L.lib.glove_format_float32(x, buf, 16, ctypes.byref(m))
        host.append(buf.raw[:m.value])
    want = b"".join(b"w " + b" ".join(host[r * d:(r + 1) * d]) + b"\n" for r in range(len(bits) // d))
    assert text.cpu().numpy().tobytes() == want


def _check_read(path, data, dim=None, **kw):
    from glove_tensorflow_b200 import vectors
    want_w, want_r = vo.read_vectors(data, dim)
    words, rows = vectors.read_vectors(str(path), dim, **kw)
    assert [vectors.word_bytes(w) for w in words] == want_w
    np.testing.assert_array_equal(rows.cpu().numpy().view(np.uint32), want_r.view(np.uint32))
    return words, rows


@pytest.mark.parametrize("name", sorted(vo.handmade_files()))
@pytest.mark.parametrize("chunk", [64 << 20, 64])
def test_import_of_handmade_files_equals_the_oracle(tmp_path, name, chunk):
    data = vo.handmade_files()[name]
    p = tmp_path / "v.txt"
    p.write_bytes(data)
    _check_read(p, data, chunk_bytes=chunk)


def _random_file(rng, V, d, header):
    seps = [b" ", b"  ", b"\t", b" \t "]
    forms = [lambda x: repr(float(x)).encode(), lambda x: b"%.9g" % x, lambda x: b"%.3e" % x, lambda x: b"%+.10f" % x,
             lambda x: vo.format_f32(x).encode(), lambda x: b"%.25f" % x]
    lines = [b"%d %d" % (V, d)] if header else []
    n = 0
    while n < V:
        if rng.random() < 0.05:
            lines.append(rng.choice([b"", b"  ", b"\t\r"]))
            continue
        L = int(rng.integers(1, 21))
        word = bytes(rng.choice(list(b"abcxyz-_.'\"019"), L).tolist())
        if n and rng.random() < 0.05:                     # not on the first line: it decides d without a header
            word = word + b" " + "é".encode()
        vals = rng.normal(0, 0.4, d).astype(np.float32)
        vals[rng.random(d) < 0.02] = np.float32(1e-41)
        line = word + b"".join(seps[int(rng.integers(0, 4))] + forms[int(rng.integers(0, 6))](np.float32(v)) for v in vals)
        if rng.random() < 0.1:
            line += b"  "
        if rng.random() < 0.1:
            line += b"\r"
        lines.append(line)
        n += 1
    return b"\n".join(lines) + (b"\n" if rng.random() < 0.5 else b"")


@pytest.mark.parametrize("d", [2, 50, 300, 510])
@pytest.mark.parametrize("header", [False, True])
def test_import_of_random_files_equals_the_oracle(tmp_path, d, header):
    rng = np.random.default_rng(d * 2 + header)
    data = _random_file(rng, max(20, 12000 // d), d, header)
    p = tmp_path / "v.txt"
    p.write_bytes(data)
    _check_read(p, data)
    _check_read(p, data, chunk_bytes=max(64, len(data) // 300))      # hundreds of chunks: lines, words, numbers split


@pytest.mark.parametrize("case", vo.malformed_files(), ids=[c[0] for c in vo.malformed_files()])
@pytest.mark.parametrize("chunk", [64 << 20, 64])
def test_malformed_files_name_the_lowest_bad_line(tmp_path, case, chunk):
    from glove_tensorflow_b200 import vectors
    name, data, dim, line = case
    p = tmp_path / "v.txt"
    p.write_bytes(data)
    with pytest.raises(ValueError, match="line %d[:, ]" % line):
        vectors.read_vectors(str(p), dim, chunk_bytes=chunk)


def test_a_line_longer_than_the_carry_room_is_refused(tmp_path):
    from glove_tensorflow_b200 import data_utils, vectors
    p = tmp_path / "v.txt"
    p.write_bytes(b"a 1 2\n" + b"x" * (data_utils._HEAD + 100) + b" 1 2\nb 3 4\n")
    with pytest.raises(ValueError, match="line 2 is longer than"):
        vectors.read_vectors(str(p), chunk_bytes=1 << 16)


def _planted_table(rng, V, d):
    W = rng.normal(0, 0.4, (V, d)).astype(np.float32)
    flat = W.reshape(-1)
    idx = rng.integers(0, flat.size, 4000)
    flat[idx[:1000]] = rng.integers(1, 1 << 23, 1000, dtype=np.uint32).view(np.float32)           # subnormals
    flat[idx[1000:1500]] = 0.0
    flat[idx[1500:2000]] = -0.0
    flat[idx[2000:3000]] = (rng.normal(size=1000) * 1e37).astype(np.float32)                       # huge
    flat[idx[3000:]] = np.float32(3.4028235e38) * rng.choice([-1, 1], 1000)
    return W


def test_export_then_import_is_bit_exact(tmp_path):
    import torch
    from glove_tensorflow_b200 import vectors
    rng = np.random.default_rng(1)
    V, d = 40_000, 300
    W = _planted_table(rng, V, d)
    words = ["w%d" % i for i in range(V)]
    words[5], words[6], words[7] = "two words", "été", "w1"          # a space, UTF-8 and a duplicate
    dev = torch.from_numpy(W).cuda()
    for header in (False, True):
        p = str(tmp_path / ("h%d.txt" % header))
        vectors.write_vectors(p, words, dev, header=header, rows_per_chunk=7000)
        got_w, got = vectors.read_vectors(p, chunk_bytes=16 << 20)
        assert got_w == words
        assert torch.equal(got.view(torch.int32), dev.view(torch.int32))
        with open(p, "rb") as f:
            assert (f.readline() == b"40000 300\n") == header
    small = W[:300, :40].copy()
    p = str(tmp_path / "small.txt")
    vectors.write_vectors(p, words[:300], torch.from_numpy(small).cuda()[:, :40], header=True)
    assert open(p, "rb").read() == vo.format_vectors([vectors.word_bytes(w) for w in words[:300]], small, header=True)
    # a strided view (a packed table's rows) is written as its first d columns
    wide = torch.from_numpy(np.ascontiguousarray(np.pad(small, ((0, 0), (0, 8))))).cuda()
    vectors.write_vectors(p + "2", words[:300], wide[:, :40])
    assert open(p + "2", "rb").read() == vo.format_vectors([vectors.word_bytes(w) for w in words[:300]], small)


def test_vectors_engine_fills_the_packed_table_in_place(tmp_path):
    import torch
    from glove_tensorflow_b200 import vectors
    rng = np.random.default_rng(4)
    W = rng.normal(size=(3000, 64)).astype(np.float32)
    words = ["w%d" % i for i in range(3000)]
    for header in (True, False):
        p = str(tmp_path / ("v%d.txt" % header))
        vectors.write_vectors(p, words, torch.from_numpy(W).cuda(), header=header)
        eng, got = vectors.vectors_engine(p)
        assert got == words and (eng.V, eng.d) == (3000, 64)
        np.testing.assert_array_equal(eng.get_state(flush=False)["R"].view(np.uint32), W.view(np.uint32))
        sim, idx = eng.topk([0, 1], 3)
        assert idx[:, 0].tolist() == [0, 1]
        # the normalised copy of the top-k does not survive a replaced table
        eng.row_plane()[:, :64].copy_(torch.from_numpy(W[::-1].copy()).cuda())
        assert eng.topk([0], 1)[1][0, 0] == 0 and abs(eng.pair_cosine([[0, 2999]])[0] - 1.0) > 1e-3
        np.testing.assert_allclose(eng.topk([2999], 1)[0][0, 0], 1.0, atol=1e-6)


def test_text8_export_and_evaluation_of_the_file_match_the_job_dir(tmp_path):
    from glove_tensorflow_b200 import config_utils, estimator, evaluate_embeddings as ev, export_embeddings as ex
    job = str(tmp_path / "job")
    params = config_utils.parse_args(["--train-csv", os.path.join(GOLD, "interaction.csv"), "--vocab-txt",
                                      os.path.join(GOLD, "vocab.txt"), "--job-dir", job, "--disable-datetime-path",
                                      "--embedding-size", "16", "--batch-size", "256", "--learning-rate", "0.05",
                                      "--seed", "2", "--plan-steps", "4", "--train-steps", "40"])
    estimator.train(params)
    qf, sf = tmp_path / "q.txt", tmp_path / "s.txt"
    qf.write_text(": family\nw4 w5 w6 w7\nw8 w9 w10 w11\nNULL none w12 w13\nw14 w15 w16 unknownword\n"
                  ": gram1-x\nw20 w21 w22 w23\nw30 w31 w32 w33\nw4 w4 w40 w41\nthe of and nan\n", encoding="utf8")
    sf.write_text("w4 w5 1.0\nw6 w7 2.5\nw8 w40 0.5\nw9 w41 3.0\nnan null 2.0\nw10 missing 1.0\nw11 w12 4.0\n", encoding="utf8")
    vocab = open(os.path.join(GOLD, "vocab.txt"), encoding="utf8").read().split("\n")
    if vocab[-1] == "":
        vocab.pop()
    for vectors in ("row", "sum"):
        out = str(tmp_path / ("vectors_%s.txt" % vectors))
        ex.main(job, str(tmp_path / "unused.json"), format="glove", vectors=vectors, output=out, word2vec_header=vectors == "sum")
        assert not os.path.exists(str(tmp_path / "unused.json"))
        words, _ = vo.read_vectors(open(out, "rb").read())
        assert [w.decode() for w in words] == vocab                   # every row in id order, <UNK> included
        for restrict in (None, 40):
            extra = ["--restrict-vocab", str(restrict)] if restrict else []
            a = ev.main(["--job-dir", job, "--vectors", vectors, "--analogies", str(qf), "--similarity", str(sf),
                         "--output-json", str(tmp_path / "a.json")] + extra)
            b = ev.main(["--vectors-txt", out, "--analogies", str(qf), "--similarity", str(sf),
                         "--output-json", str(tmp_path / "b.json")] + extra)
            assert a["analogies"] == b["analogies"] and a["similarity"] == b["similarity"]
            assert a["restrict_vocab"] == b["restrict_vocab"]
            assert (b["vectors_txt"], b["rows"], b["dim"]) == (out, len(vocab), 16)
            assert "checkpoint" not in b and json.load(open(str(tmp_path / "b.json"))) == json.loads(json.dumps(b))


def test_a_large_file_through_the_cli(tmp_path):
    import torch
    from glove_tensorflow_b200 import evaluate_embeddings as ev, vectors
    rng = np.random.default_rng(12)
    V, d = 200_000, 100
    W = rng.normal(size=(V, d)).astype(np.float32)
    vocab = ["t%d" % i for i in range(V)]
    p = str(tmp_path / "big.txt")
    vectors.write_vectors(p, vocab, torch.from_numpy(W).cuda())
    pairs = [(int(a), int(b), float(s)) for a, b, s in zip(rng.integers(0, V, 300), rng.integers(0, V, 300), rng.random(300))]
    sf = tmp_path / "s.txt"
    sf.write_text("".join("t%d t%d %r\n" % t for t in pairs), encoding="utf8")
    rep = ev.main(["--vectors-txt", p, "--dim", "100", "--similarity", str(sf), "--output-json", str(tmp_path / "r.json")])
    assert (rep["rows"], rep["dim"]) == (V, d)
    want = ao.similarity_report(W, vocab, [("t%d" % a, "t%d" % b, s) for a, b, s in pairs])
    s = rep["similarity"][0]
    assert s["found"] == want["found"] == 300
    assert abs(s["spearman"] - want["spearman"]) < 1e-9 and abs(s["pearson"] - want["pearson"]) < 1e-5
