"""GPU checks of the streamed corpus preprocessor (glove_tensorflow_b200/corpus.py): its files are byte-identical to
text8.save_data(text8.process_data(...)) whole, in hundreds of chunks and with forced small partitions; every float64 it
writes is repr(float); the device formatter equals the host build; a corpus past 2^31 bytes is counted exactly; the csv
trains; bad input fails loudly."""
import ctypes
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden", "text8_small")
FILES = ("vocab.csv", "vocab.txt", "interaction.csv")


def _reference(text, out, vocab_size, context_size, coverage=0.9):
    from glove_tensorflow_b200 import text8
    text8.save_data(text8.process_data(text, vocab_size=vocab_size, coverage=coverage, context_size=context_size), str(out))


def _same_files(a, b):
    for name in FILES:
        with open(os.path.join(a, name), "rb") as fa, open(os.path.join(b, name), "rb") as fb:
            assert fa.read() == fb.read(), name


def _floats_are_repr(path):
    with open(path) as f:
        next(f)
        for line in f:
            fields = line.rstrip("\n").rsplit(",", 3)
            for s in fields[1:] + [line.split(",", 4)[3]]:
                assert repr(float(s)) == s, s


@pytest.mark.parametrize("kw", [{}, {"chunk_bytes": 4096}, {"chunk_bytes": 4096, "partition_entries": 300, "chunk_positions": 5000}])
def test_text8_small_is_byte_identical_to_the_in_memory_path(tmp_path, kw):
    from glove_tensorflow_b200 import corpus
    path = os.path.join(GOLD, "corpus.txt")
    _reference(open(path).read(), tmp_path / "ref", 60, 5)
    stats = {}
    frame, n = corpus.preprocess(path, str(tmp_path / "new"), vocab_size=60, coverage=0.9, context_size=5, stats=stats, **kw)
    _same_files(tmp_path / "ref", tmp_path / "new")
    for name in ("vocab.csv", "vocab.txt"):     # the reference's own records are in its salted-hash order: vocab only
        assert open(os.path.join(GOLD, name), "rb").read() == open(tmp_path / "new" / name, "rb").read()
    assert n == sum(1 for _ in open(tmp_path / "new" / "interaction.csv")) - 1 and len(frame) == 61
    if "partition_entries" in kw:
        assert stats["partitions"] > 8
    _floats_are_repr(tmp_path / "new" / "interaction.csv")


def _seeded_corpus(seed, n):
    rng = np.random.default_rng(seed)
    words = ["w%d" % i for i in range(300)] + ["na", "null", "caf" + chr(0xe9), chr(0x4e2d) + chr(0x6587), "a", "x" * 70,
                                               "<UNK>", '"q"', "a,b", 'x"y,z']
    p = 1.0 / np.arange(1, len(words) + 1)
    seps = [" ", " ", " ", "  ", chr(9), chr(10), chr(13) + chr(10), " " + chr(11) + chr(12) + " ", chr(0x1c), chr(0x1f) + " "]
    picks = rng.choice(len(words), size=n, p=p / p.sum())
    return "  " + chr(10) + "".join(words[i] + seps[rng.integers(len(seps))] for i in picks) + "tail"


@pytest.mark.parametrize("context", [1, 5, 8])
@pytest.mark.parametrize("kw", [{}, {"chunk_bytes": 2048, "partition_entries": 1000}, {"chunk_bytes": 1 << 16, "partition_entries": 50, "chunk_positions": 777}])
def test_seeded_corpora_are_byte_identical(tmp_path, context, kw):
    from glove_tensorflow_b200 import corpus
    text = _seeded_corpus(context, 40000)
    path = tmp_path / "c.txt"
    path.write_bytes(text.encode("utf8"))
    _reference(text, tmp_path / "ref", 120, context, coverage=0.95)
    corpus.preprocess(str(path), str(tmp_path / "new"), vocab_size=120, coverage=0.95, context_size=context, **kw)
    _same_files(tmp_path / "ref", tmp_path / "new")
    _floats_are_repr(tmp_path / "new" / "interaction.csv")


def test_device_formatter_equals_host_build():
    import torch
    from glove_tensorflow_b200 import _lib
    from test_corpus import random_bit_patterns, special_bit_patterns
    lib = _lib.lib
    bits = np.concatenate([random_bit_patterns(1_000_000, seed=7), np.array(special_bit_patterns(), np.uint64)])
    n = len(bits)
    d_bits = torch.from_numpy(bits.view(np.int64)).cuda()
    out = torch.empty(n * 24, dtype=torch.uint8, device="cuda")
    ln = torch.empty(n, dtype=torch.int32, device="cuda")
    _lib.check(lib.glove_format_float64_device(d_bits.data_ptr(), n, out.data_ptr(), ln.data_ptr(),
                                               torch.cuda.current_stream().cuda_stream), "glove_format_float64_device")
    text, ln = out.cpu().numpy().reshape(n, 24), ln.cpu().numpy()
    buf, m = ctypes.create_string_buffer(32), ctypes.c_int32()
    for i, b in enumerate(bits.tolist()):
        x = np.array([b], np.uint64).view(np.float64)[0]
        assert lib.glove_format_float64(float(x), buf, 32, ctypes.byref(m)) == 0
        assert text[i, :ln[i]].tobytes() == buf.raw[:m.value], hex(b)


def test_corpus_past_2_31_bytes(tmp_path):
    """Counted exactly where DeviceCorpus refuses: total count = 2 sum_k n_k, sum of value = 2 sum_k n_k / k (n_k =
    positions whose k-th right neighbour has another id), symmetric, no key twice."""
    import pandas as pd
    import torch
    from glove_tensorflow_b200 import corpus
    rng = np.random.default_rng(31)
    words = np.array([("w%02d" % i).ljust(7, "_").encode() + b" " for i in range(40)])     # 8 bytes a token
    n_tok = (1 << 31) // 8 + 1_000_000
    picks = rng.integers(0, 40, n_tok, dtype=np.int64)
    path = tmp_path / "big.txt"
    with open(path, "wb") as f:
        for s in range(0, n_tok, 1 << 26):
            f.write(np.frombuffer(b"".join(words), np.uint8).reshape(40, 8)[picks[s:s + (1 << 26)]].tobytes())
    assert os.path.getsize(path) > (1 << 31)                      # past what DeviceCorpus (process_data) accepts
    ctx = 3
    frame, n = corpus.preprocess(str(path), str(tmp_path / "out"), vocab_size=30, coverage=1.0, context_size=ctx)
    os.remove(path)
    row_of = {t: i for i, t in enumerate(frame["token"])}
    lut = torch.tensor([row_of.get(w.decode().strip(), 0) for w in words], dtype=torch.int32, device="cuda")
    ids = lut[torch.from_numpy(picks).cuda()]
    n_k = [int((ids[:-k] != ids[k:]).sum()) for k in range(1, ctx + 1)]
    t = pd.read_csv(tmp_path / "out" / "interaction.csv", keep_default_na=False)
    assert len(t) == n and int(t["count"].sum()) == 2 * sum(n_k)
    assert abs(t["value"].sum() - 2 * sum(c / k for k, c in enumerate(n_k, 1))) < 1e-9 * t["value"].sum()
    key = t["row_token_id"].to_numpy(np.int64) * 100 + t["col_token_id"].to_numpy(np.int64)
    assert len(np.unique(key)) == len(key)
    back = dict(zip(t["col_token_id"].to_numpy(np.int64) * 100 + t["row_token_id"].to_numpy(np.int64), zip(t["count"], t["value"])))
    assert all(back[k] == (c, v) for k, c, v in zip(key, t["count"], t["value"]))


def test_streamed_csv_trains(tmp_path):
    from glove_tensorflow_b200 import config_utils, corpus, data_utils, estimator
    frame, n = corpus.preprocess(os.path.join(GOLD, "corpus.txt"), str(tmp_path / "data"), vocab_size=60, coverage=0.9,
                                 context_size=5, chunk_bytes=8192)
    csv, voc = str(tmp_path / "data" / "interaction.csv"), str(tmp_path / "data" / "vocab.txt")
    coo = data_utils.ingest_csv(csv, voc)
    assert len(coo["row"]) == n
    params = config_utils.parse_args(["--train-csv", csv, "--vocab-txt", voc, "--job-dir", str(tmp_path / "job"),
                                      "--disable-datetime-path", "--embedding-size", "16", "--batch-size", "512",
                                      "--learning-rate", "0.05", "--train-steps", "150", "--seed", "1"])
    first = estimator.build_engine(params).eval_metrics(512)["loss"]
    eng, hist = estimator.train(params)
    assert eng.host_step == 150 and hist[-1][1]["loss"] < 0.5 * first


def test_bad_corpora_fail_loudly(tmp_path):
    from glove_tensorflow_b200 import corpus
    p = tmp_path / "c.txt"
    for cp in (0x85, 0xa0, 0x2003, 0x3000):
        raw = ("word " * 3000 + "a" + chr(cp) + "b end").encode("utf8")
        p.write_bytes(raw)
        with pytest.raises(ValueError, match="byte %d: non-ASCII Unicode whitespace" % (3000 * 5 + 1)):
            corpus.preprocess(str(p), str(tmp_path / "o"), chunk_bytes=4096)
    p.write_bytes(b"")
    with pytest.raises(ValueError, match="empty corpus"):
        corpus.preprocess(str(p), str(tmp_path / "o"))
    for raw in (b"  \n\t ", b"  one\n"):
        p.write_bytes(raw)
        with pytest.raises(ValueError, match="at least two tokens"):
            corpus.preprocess(str(p), str(tmp_path / "o"))
    p.write_bytes(_seeded_corpus(3, 20000).encode("utf8"))
    with pytest.raises(MemoryError, match="co-occurrence table needs .* GB of device memory"):
        corpus.preprocess(str(p), str(tmp_path / "o"), vocab_size=120, context_size=5, device_bytes=1 << 20)
