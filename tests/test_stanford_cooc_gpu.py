"""GPU checks of corpus.preprocess(scheme="stanford") against oracle/stanford_cooc_oracle.py: vocab.txt byte-identical,
cooccurrence.shuf.bin equal to the oracle's records as a multiset with val bit-exact, the same file bytes however the
corpus is chunked, blocked and partitioned, its import equal to the oracle's COO, the refusals with their offsets, the
memory guard, and the route corpus -> train -> export -> evaluate."""
import os

import numpy as np
import pytest

from oracle import cooc_bin_oracle as cb
from oracle import stanford_cooc_oracle as so

pytestmark = pytest.mark.gpu

CHUNK = 4096
REC = np.dtype([("w1", "<i4"), ("w2", "<i4"), ("val", "<f8")])


def _corpus(seed, n_lines=1500):
    """Short lines, blank lines, CRLF, tabs, repeated words, rare words (out of the vocabulary at min_count 2), non-ASCII
    words, one line longer than a chunk, a '\\n' as the last byte of a chunk and a CRLF across a chunk cut."""
    rng = np.random.default_rng(seed)
    words = [b"w%d" % i for i in range(400)] + ["café".encode(), "中文".encode(), b"<UNK>", b"x" * 300]
    p = 1.0 / np.arange(1, len(words) + 1) ** 1.1
    lines = []
    for i in range(n_lines):
        n = 3000 if i == 700 else int(rng.choice([0, 1, 2, 3, 5, 8, 12, 20, 30]))
        picks = rng.choice(len(words), size=n, p=p / p.sum())
        if n > 4 and rng.random() < 0.2:
            picks[1:4] = picks[0]
        toks = [words[k] for k in picks] + [b"r%d" % int(rng.integers(1 << 20)) for _ in range(int(rng.random() < 0.3))]
        rng.shuffle(toks)
        seps = [rng.choice([b" ", b"\t", b"  "]) for _ in toks]
        lines.append(b"".join(t + s for t, s in zip(toks, seps)) + rng.choice([b"\n", b"\r\n", b" \n", b"\n\n"]))
    data = bytearray(b"".join(lines))
    for c, s in ((3, b"\n"), (5, b"\r\n"), (9, b"\n"), (11, b"\n"), (13, b"\r\n")):   # ascending: later offsets hold
        data[c * CHUNK - 1:c * CHUNK - 1] = s          # byte c * CHUNK - 1: a '\n', or the '\r' of a CRLF across the cut
    return bytes(data)


def _run(path, dest, **kw):
    from glove_tensorflow_b200 import corpus
    stats = {}
    frame, n = corpus.preprocess(str(path), str(dest), scheme="stanford", stats=stats, **kw)
    vocab = open(os.path.join(dest, "vocab.txt"), "rb").read()
    recs = np.fromfile(os.path.join(dest, "cooccurrence.shuf.bin"), REC)
    assert len(recs) == n == stats["records"]
    return vocab, recs, stats


def _sorted(recs):
    order = np.lexsort((recs["w2"], recs["w1"]))
    return recs[order]


@pytest.mark.parametrize("window,symmetric,weighting,min_count,max_vocab", [
    (15, True, True, 2, 0), (15, False, False, 2, 0), (5, False, True, 1, 0), (1, True, False, 3, 0),
    (10, True, True, 2, 150), (8, True, True, 1, 37)])
def test_equals_the_oracle(tmp_path, window, symmetric, weighting, min_count, max_vocab):
    data = _corpus(window)
    path = tmp_path / "c.txt"
    path.write_bytes(data)
    kw = dict(window_size=window, symmetric=symmetric, distance_weighting=weighting, min_count=min_count, max_vocab=max_vocab)
    vocab, recs, _ = _run(path, tmp_path / "out", chunk_bytes=CHUNK, **kw)
    voc = so.vocab(data, min_count, max_vocab)
    assert vocab == so.vocab_txt(voc)
    row, col, val = so.records(so.cooccur(data, voc, window, symmetric, weighting))
    got = _sorted(recs)
    assert np.array_equal(got["w1"], row + 1) and np.array_equal(got["w2"], col + 1)
    assert np.array_equal(got["val"].view(np.int64), val.view(np.int64))


def test_file_bytes_do_not_depend_on_chunks_blocks_or_partitions(tmp_path):
    data = _corpus(99)
    path = tmp_path / "c.txt"
    path.write_bytes(data)
    kw = dict(window_size=15, min_count=2)
    ref = _run(path, tmp_path / "whole", **kw)
    assert ref[2]["partitions"] == 1
    for i, extra in enumerate([{"chunk_bytes": CHUNK}, {"chunk_bytes": 1024, "chunk_positions": 7},
                               {"chunk_bytes": CHUNK, "partition_entries": 2000}, {"chunk_positions": 3}, {}]):
        got = _run(path, tmp_path / ("r%d" % i), **kw, **extra)
        assert got[0] == ref[0] and got[1].tobytes() == ref[1].tobytes(), extra
        if "partition_entries" in extra:
            assert got[2]["partitions"] > 16


def test_import_equals_the_oracle_coo(tmp_path):
    from glove_tensorflow_b200 import data_utils
    data = _corpus(7)
    path = tmp_path / "c.txt"
    path.write_bytes(data)
    _run(path, tmp_path / "out", chunk_bytes=CHUNK, min_count=2, window_size=15)
    voc = so.vocab(data, 2)
    row, col, val = so.records(so.cooccur(data, voc, 15))
    want = cb.read(cb.write(row, col, val), len(voc))
    got = data_utils.load_cooc_bin(str(tmp_path / "out" / "cooccurrence.shuf.bin"), len(voc))
    got = {k: v.cpu().numpy() for k, v in got.items()}
    order = np.lexsort((got["col"], got["row"]))
    for k in ("row", "col", "glove_value", "glove_weight"):
        assert np.array_equal(np.asarray(got[k])[order].view(np.int32), np.asarray(want[k]).view(np.int32)), k


def test_refusals_name_the_offset(tmp_path):
    from glove_tensorflow_b200 import corpus
    p = tmp_path / "c.txt"
    body = b"alpha beta\n" * 1000
    cases = [(body + b"gamma <unk> delta\n" + b"<unk>\n", len(body) + 6, "<unk>"),
             (body + b"ab\rcd\n", len(body) + 2, "carriage return"),
             (body[:CHUNK - 1] + b"\r" + b"x" + body[CHUNK:], CHUNK - 1, "carriage return"),   # '\r' ending a chunk
             (body + b"ab\r", len(body) + 2, "carriage return"),
             (body + b"a\x0bb\n" + b"c\x0cd\n", len(body) + 1, "vertical tab"),
             (body + b"a\x1db\n", len(body) + 1, "separator byte 0x1d"),
             (body + "a　b c\x0bd\n".encode(), len(body) + 1, "non-ASCII Unicode whitespace")]
    for raw, off, what in cases:
        p.write_bytes(raw)
        for kw in ({}, {"chunk_bytes": CHUNK}):
            with pytest.raises(ValueError, match="byte %d: .*%s" % (off, what)):
                corpus.preprocess(str(p), str(tmp_path / "o"), scheme="stanford", **kw)
    # CRLF across a chunk cut is a line end, not a refusal
    p.write_bytes(body[:CHUNK - 1] + b"\r\n" + body[CHUNK:])
    corpus.preprocess(str(p), str(tmp_path / "o"), scheme="stanford", chunk_bytes=CHUNK)


def test_too_small_device_budget_raises_memory_error(tmp_path):
    from glove_tensorflow_b200 import corpus
    p = tmp_path / "c.txt"
    p.write_bytes(_corpus(3))
    with pytest.raises(MemoryError, match="co-occurrence table needs .* GB of device memory"):
        corpus.preprocess(str(p), str(tmp_path / "o"), scheme="stanford", device_bytes=1 << 16)


def test_corpus_to_training_to_export_to_evaluation(tmp_path):
    import torch
    from glove_tensorflow_b200 import corpus, estimator, evaluate_embeddings as ev, export_embeddings as ex, config_utils
    from glove_tensorflow_b200.data_utils import read_stanford_vocab
    data = _corpus(11, 800)
    p = tmp_path / "c.txt"
    p.write_bytes(data)
    dest = tmp_path / "data"
    corpus.main(["--corpus", str(p), "--dest", str(dest), "--scheme", "stanford", "--min-count", "2", "--window-size", "10"])
    tokens, counts = read_stanford_vocab(str(dest / "vocab.txt"))
    voc = so.vocab(data, 2)
    assert tokens == [t.decode() for t, _ in voc] and counts.tolist() == [c for _, c in voc]
    job = str(tmp_path / "job")
    params = config_utils.parse_args(["--train-cooc", str(dest / "cooccurrence.shuf.bin"), "--vocab-txt", str(dest / "vocab.txt"),
                                      "--job-dir", job, "--disable-datetime-path", "--embedding-size", "16", "--batch-size",
                                      "256", "--learning-rate", "0.05", "--seed", "3", "--train-steps", "40",
                                      "--train-csv", str(tmp_path / "missing.csv")])
    eng, hist = estimator.train(params)
    assert eng.host_step == 40 and np.isfinite(hist[-1][1]["loss"])
    del eng
    torch.cuda.empty_cache()
    out = str(tmp_path / "vectors.txt")
    ex.main(job, str(tmp_path / "unused.json"), format="glove", output=out)
    words = [line.split(" ", 1)[0] for line in open(out, encoding="utf8")]
    assert words == tokens                         # the vocabulary survives the round trip, in id order
    sf = tmp_path / "s.txt"
    sf.write_text("w0 w1 1.0\nw2 w3 2.0\nw1 w4 3.0\n", encoding="utf8")
    rep = ev.main(["--vectors-txt", out, "--similarity", str(sf), "--output-json", str(tmp_path / "r.json")])
    assert rep["similarity"][0]["found"] == 3
