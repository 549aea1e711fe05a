"""GPU checks of the Stanford GloVe co-occurrence container (csrc/glove_crec.cu): the import equals the NumPy oracle on
seeded files read whole and in chunks; a bad file names its lowest bad record; the preprocessor's cooccurrence.shuf.bin
is its csv in binary and imports to what the csv ingest gives; the trainer runs from a .bin bit for bit as from the same
arrays given directly."""
import csv
import os
import struct

import numpy as np
import pytest

from oracle import cooc_bin_oracle as cb

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden", "text8_small")


def _seeded_file(path, V, n, seed, x_max=100.0):
    rng = np.random.default_rng(seed)
    val = np.exp(rng.uniform(np.log(1e-300), np.log(1e300), n))
    edge = rng.integers(0, n, max(n // 50, 5))
    val[edge] = rng.choice([x_max, x_max * (1 - 2.0 ** -52), x_max * (1 + 2.0 ** -52), np.nextafter(x_max, 0), 1.0,
                            5e-324, 1.7976931348623157e308], len(edge))
    raw = cb.write(rng.integers(0, V, n), rng.integers(0, V, n), val)
    with open(path, "wb") as f:
        f.write(raw)
    return raw


def _ulps(a, b):
    return np.abs(a.view(np.int32).astype(np.int64) - b.view(np.int32).astype(np.int64))


@pytest.mark.parametrize("V,n,chunks", [(10, 5000, (1, 3, 313)), (1000, 200_000, (1000, 4099)),
                                        (400_000, 1_000_000, (65536, 1 << 20))])
def test_import_equals_the_oracle(tmp_path, V, n, chunks):
    from glove_tensorflow_b200 import data_utils
    path = str(tmp_path / "c.bin")
    raw = _seeded_file(path, V, n, V)
    want = cb.read(raw, V)
    for k in (None,) + chunks:
        kw = {} if k is None else {"chunk_bytes": 16 * k}
        got = {c: t.cpu().numpy() for c, t in data_utils.load_cooc_bin(path, V, **kw).items()}
        assert sorted(got) == ["col", "glove_value", "glove_weight", "row"]
        assert np.array_equal(got["row"], want["row"]) and np.array_equal(got["col"], want["col"])
        for c in ("glove_value", "glove_weight"):
            d = _ulps(got[c], want[c])
            assert d.max() <= 1, (c, k, int(d.max()))
            print("V=%d chunk=%s %s: %d of %d differ from the host by 1 ulp" % (V, k, c, int((d == 1).sum()), n))
        assert got["glove_weight"].max() <= 1.0 and np.all(got["glove_weight"][raw_val(raw) >= 100.0] == 1.0)


def raw_val(raw):
    return np.frombuffer(raw, cb.RECORD)["val"]


def test_import_other_x_max_and_alpha(tmp_path):
    from glove_tensorflow_b200 import data_utils
    path = str(tmp_path / "c.bin")
    raw = _seeded_file(path, 50, 20000, 5, x_max=10.0)
    want = cb.read(raw, 50, x_max=10.0, alpha=0.5)
    got = data_utils.load_cooc_bin(path, 50, x_max=10.0, alpha=0.5, chunk_bytes=16 * 777)
    assert _ulps(got["glove_weight"].cpu().numpy(), want["glove_weight"]).max() <= 1
    assert np.array_equal(got["row"].cpu().numpy(), want["row"])


@pytest.mark.parametrize("w1,w2,val,what", [(0, 1, 1.0, "word1 id 0 outside 1..40"), (41, 1, 1.0, "word1 id 41"),
                                            (-7, 1, 1.0, "word1 id -7"), (1, 0, 1.0, "word2 id 0"),
                                            (1, 41, 1.0, "word2 id 41"), (1, -1, 1.0, "word2 id -1"),
                                            (1, 1, 0.0, "val 0.0"), (1, 1, -3.5, "val -3.5"), (1, 1, float("nan"), "val nan"),
                                            (1, 1, float("inf"), "val inf"), (1, 1, float("-inf"), "val -inf")])
def test_the_lowest_bad_record_is_named(tmp_path, w1, w2, val, what):
    from glove_tensorflow_b200 import data_utils
    V, n = 40, 10000
    rng = np.random.default_rng(3)
    rec = np.frombuffer(bytearray(cb.write(rng.integers(0, V, n), rng.integers(0, V, n), rng.uniform(0.5, 500, n))),
                        cb.RECORD)
    bad = np.frombuffer(struct.pack("<iid", w1, w2, val), cb.RECORD)[0]
    other = np.frombuffer(struct.pack("<iid", 0, 0, -1.0), cb.RECORD)[0]
    path = str(tmp_path / "bad.bin")
    # chunks of 1000 records: the first bad record in chunk 2, a worse kind later in the same chunk, more in later chunks
    for first in (2500, 999, 1000, 9999):
        r = rec.copy()
        r[first] = bad
        for i in (first + 60, 7400, n - 1):
            if first < i < n:
                r[i] = other
        open(path, "wb").write(r.tobytes())
        with pytest.raises(ValueError) as e:
            cb.read(r.tobytes(), V)
        assert "record %d (byte %d): %s" % (first + 1, 16 * first, what) in str(e.value)
        for kw in ({"chunk_bytes": 16 * 1000}, {}, {"chunk_bytes": 16 * 7}):
            with pytest.raises(ValueError) as e:
                data_utils.load_cooc_bin(path, V, **kw)
            assert "bad.bin: record %d (byte %d): %s" % (first + 1, 16 * first, what) in str(e.value)


def test_a_truncated_file_is_refused(tmp_path):
    from glove_tensorflow_b200 import data_utils
    raw = cb.write(np.arange(5000) % 30, np.arange(5000) % 29, np.full(5000, 2.0))
    path = str(tmp_path / "t.bin")
    for cut in (1, 8, 15):
        open(path, "wb").write(raw[:-cut])
        for kw in ({}, {"chunk_bytes": 16 * 100}):
            with pytest.raises(ValueError, match=r"record 5000 \(byte 79984\): the file ends %d bytes into" % (16 - cut)):
                data_utils.load_cooc_bin(path, 30, **kw)
    open(path, "wb").write(raw[:16 * 300] + struct.pack("<iid", 31, 1, 1.0) + raw[16 * 301:-3])
    with pytest.raises(ValueError, match=r"record 301 \(byte 4800\): word1 id 31"):     # a bad whole record comes first
        data_utils.load_cooc_bin(path, 30, chunk_bytes=16 * 100)
    open(path, "wb").write(b"")
    assert data_utils.load_cooc_bin(path, 30)["row"].numel() == 0


def _csv_rows(path):
    with open(path, newline="", encoding="utf8") as f:
        r = csv.reader(f)
        head = next(r)
        rows = list(r)
    c = {name: i for i, name in enumerate(head)}
    return (np.array([int(x[c["row_token_id"]]) for x in rows], np.int64), np.array([int(x[c["col_token_id"]]) for x in rows], np.int64),
            np.array([float(x[c["value"]]) for x in rows], np.float64))


def _check_preprocessed(out):
    import pandas as pd
    from glove_tensorflow_b200 import data_utils
    csv_path, bin_path, voc = (os.path.join(out, n) for n in ("interaction.csv", "cooccurrence.shuf.bin", "vocab.txt"))
    raw = open(bin_path, "rb").read()
    rec = np.frombuffer(raw, cb.RECORD)
    row, col, value = _csv_rows(csv_path)
    assert len(rec) == len(row) > 0
    assert np.array_equal(rec["word1"], row + 1) and np.array_equal(rec["word2"], col + 1)
    assert np.array_equal(rec["val"].view(np.uint64), value.view(np.uint64))
    frame = pd.read_csv(os.path.join(out, "vocab.csv"), keep_default_na=False)
    stanford = open(os.path.join(out, "vocab.stanford.txt"), encoding="utf8").read()
    assert stanford == "".join("%s %d\n" % (t, c) for t, c in zip(frame["token"], frame["count"]))
    tokens, counts = data_utils.read_stanford_vocab(os.path.join(out, "vocab.stanford.txt"))
    assert tokens == data_utils.read_vocab(voc) and counts.tolist() == frame["count"].tolist()
    V = len(tokens)
    got = data_utils.load_cooc_bin(bin_path, V, chunk_bytes=16 * 1000)
    ref = data_utils.ingest_csv(csv_path, voc, row_name="row_token_id", col_name="col_token_id",
                                value_names=("glove_value", "glove_weight"))
    for a, b in (("row", "row"), ("col", "col"), ("glove_value", "glove_value")):
        assert np.array_equal(got[a].cpu().numpy().view(np.int32), ref[b].cpu().numpy().view(np.int32)), a
    want = cb.read(raw, V)
    assert _ulps(got["glove_weight"].cpu().numpy(), want["glove_weight"]).max() <= 1
    return raw


def test_preprocessor_writes_the_csv_table_in_binary(tmp_path):
    from glove_tensorflow_b200 import corpus
    from test_corpus_gpu import _seeded_corpus
    path = os.path.join(GOLD, "corpus.txt")
    frame, n = corpus.preprocess(path, str(tmp_path / "both"), vocab_size=60, coverage=0.9, context_size=5, format="both")
    raw = _check_preprocessed(str(tmp_path / "both"))
    assert len(raw) == 16 * n
    for name in ("vocab.csv", "vocab.txt"):
        assert open(os.path.join(GOLD, name), "rb").read() == open(tmp_path / "both" / name, "rb").read()
    corpus.preprocess(path, str(tmp_path / "st"), vocab_size=60, coverage=0.9, context_size=5, format="stanford")
    assert open(tmp_path / "st" / "cooccurrence.shuf.bin", "rb").read() == raw
    assert not os.path.exists(tmp_path / "st" / "interaction.csv")
    assert sorted(os.listdir(tmp_path / "st")) == ["cooccurrence.shuf.bin", "vocab.csv", "vocab.stanford.txt", "vocab.txt"]
    corpus.preprocess(path, str(tmp_path / "csv"), vocab_size=60, coverage=0.9, context_size=5)
    assert sorted(os.listdir(tmp_path / "csv")) == ["interaction.csv", "vocab.csv", "vocab.txt"]
    assert open(tmp_path / "csv" / "interaction.csv", "rb").read() == open(tmp_path / "both" / "interaction.csv", "rb").read()

    text = _seeded_corpus(8, 40000)
    cp = tmp_path / "c.txt"
    cp.write_bytes(text.encode("utf8"))
    kw = dict(vocab_size=120, coverage=0.95, context_size=5, chunk_bytes=2048, partition_entries=50, records_per_block=333)
    stats = {}
    corpus.preprocess(str(cp), str(tmp_path / "seeded"), format="both", stats=stats, **kw)
    assert stats["partitions"] > 8 and stats["bin_bytes"] == 16 * stats["records"]
    raw = _check_preprocessed(str(tmp_path / "seeded"))
    corpus.main(["--corpus", str(cp), "--dest", str(tmp_path / "seeded_st"), "--vocab-size", "120", "--coverage", "0.95",
                 "--format", "stanford"])
    assert open(tmp_path / "seeded_st" / "cooccurrence.shuf.bin", "rb").read() == raw


def _golden_bin(tmp_path):
    """text8_small's interaction.csv as a Stanford .bin, with vocab.csv as a Stanford vocab.txt."""
    import pandas as pd
    row, col, value = _csv_rows(os.path.join(GOLD, "interaction.csv"))
    binp, vocp = str(tmp_path / "cooccurrence.bin"), str(tmp_path / "vocab.txt")
    open(binp, "wb").write(cb.write(row, col, value))
    frame = pd.read_csv(os.path.join(GOLD, "vocab.csv"), keep_default_na=False)
    with open(vocp, "w", encoding="utf8") as f:
        f.writelines("%s %d\n" % (t, c) for t, c in zip(frame["token"], frame["count"]))
    return binp, vocp


def test_training_from_a_bin_equals_training_from_its_arrays(tmp_path):
    import torch
    from glove_tensorflow_b200 import config_utils, data_utils, estimator, evaluate_embeddings as ev, export_embeddings as ex
    from glove_tensorflow_b200.engine import GloveEngine
    from oracle import glove_oracle as o
    binp, vocp = _golden_bin(tmp_path)
    job = str(tmp_path / "job")
    argv = ["--train-cooc", binp, "--vocab-txt", vocp, "--job-dir", job, "--disable-datetime-path", "--embedding-size", "16",
            "--batch-size", "256", "--learning-rate", "0.05", "--seed", "3", "--plan-steps", "4", "--train-steps", "60",
            "--train-csv", str(tmp_path / "missing.csv")]
    params = config_utils.parse_args(argv)
    assert open(params["vocab_txt"], "rb").read() == open(os.path.join(GOLD, "vocab.txt"), "rb").read()
    V = data_utils.file_lines(params["vocab_txt"])
    want = cb.read(open(binp, "rb").read(), V)

    a = estimator.build_engine(params)
    b = estimator.build_engine(params, load_coo=False)
    b.set_coo(want["row"], want["col"], want["glove_value"], want["glove_weight"], shuffle_key=params["seed"])
    la, lb = a.train(60), b.train(60)
    assert np.array_equal(np.asarray(la).view(np.int32), np.asarray(lb).view(np.int32))
    sa, sb = a.get_state(), b.get_state()
    for k in ("R", "C", "rb", "cb"):
        assert np.array_equal(np.asarray(sa[k]).view(np.int32), np.asarray(sb[k]).view(np.int32)), k

    # loss parity against the training oracle on explicit batches
    coo = {"row": want["row"], "col": want["col"], "target": want["glove_value"], "weight": want["glove_weight"]}
    dev = data_utils.load_cooc_bin(binp, V)
    rng = np.random.default_rng(4)
    steps, B = 12, 256
    batches = rng.integers(0, len(coo["row"]), (steps, B))
    st = o.init_state(V, 16, 1)
    ref = st.copy()
    ref_losses = np.array(o.train(ref, coo, batches, learning_rate=0.01))
    eng = GloveEngine(V, 16, learning_rate=0.01, batch_size=B, plan_steps=4, max_steps=64, device="cuda:0")
    eng.load_state(st.R, st.C, st.rb, st.cb, st.g)
    eng.set_coo(dev["row"], dev["col"], dev["glove_value"], dev["glove_weight"])
    eng.set_batches(batches)
    losses = eng.train(steps)
    assert np.max(np.abs(losses - ref_losses) / np.abs(ref_losses)) < 1e-5
    del a, b, eng
    torch.cuda.empty_cache()

    eng, hist = estimator.train(params)
    assert eng.host_step == 60 and np.isfinite(hist[-1][1]["loss"])
    out = str(tmp_path / "vectors.txt")
    ex.main(job, str(tmp_path / "unused.json"), format="glove", output=out)
    assert sum(1 for _ in open(out, encoding="utf8")) == V
    sf = tmp_path / "s.txt"
    sf.write_text("na null 1.0\nnan the 2.0\nof and 3.0\n", encoding="utf8")
    rep = ev.main(["--job-dir", job, "--similarity", str(sf), "--output-json", str(tmp_path / "r.json")])
    assert rep["similarity"][0]["found"] >= 1
