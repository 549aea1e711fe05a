"""GPU checks of Stanford GloVe's trainer (csrc/glove_sgd.cu, stanford_glove.py) against oracle/stanford_glove_oracle:
the links, the parsed records and their refusals, W, gradsq and the epoch cost bit-identical to the kernel-order
oracle on serial, conflict-free and Zipf tables, grid and run invariance, exact resume, and corpus -> train ->
evaluate."""
import os

import numpy as np
import pytest

from oracle import stanford_glove_oracle as sgo

pytestmark = pytest.mark.gpu

REC = np.dtype([("w1", "<i4"), ("w2", "<i4"), ("val", "<f8")])


def write_bin(path, w1, w2, val):
    rec = np.zeros(len(w1), REC)
    rec["w1"], rec["w2"], rec["val"] = w1, w2, val
    rec.tofile(path)
    return str(path)


def make_table(kind, V, n, seed=0):
    rng = np.random.default_rng(seed)
    if kind == "serial":            # every record has word1 = 1: one chain through all of them
        w1, w2 = np.ones(n, np.int64), rng.integers(1, V + 1, n)
    elif kind == "free":            # no two records share word1 or word2
        w1, w2 = rng.permutation(V)[:n] + 1, rng.permutation(V)[:n] + 1
    else:
        p = 1.0 / np.arange(1, V + 1)
        w1, w2 = rng.choice(V, n, p=p / p.sum()) + 1, rng.choice(V, n, p=p / p.sum()) + 1
    return w1, w2, np.exp(rng.uniform(-2, 7, n))


def test_links_and_records_match_numpy(tmp_path):
    from glove_tensorflow_b200.stanford_glove import StanfordGlove
    V = 5000
    w1, w2, val = make_table("zipf", V, 300_000, 1)
    val[:5] = [100.0, np.nextafter(100.0, 200), 1e-300, 1.7e308, 1.0]
    path = write_bin(tmp_path / "c.bin", w1, w2, val)
    sg = StanfordGlove(path, V, 8, alpha=0.75, x_max=100.0, chunk_bytes=16 * 4099)
    words, lf = sg.words.cpu().numpy(), sg.lf.cpu().numpy()
    ref_w, ref_lf = sgo.records(open(path, "rb").read(), 100.0, 0.75)
    np.testing.assert_array_equal(words, ref_w)
    np.testing.assert_array_equal(sg.prev.cpu().numpy(), sgo.links(ref_w))
    for c in range(2):
        ulps = np.abs(lf[:, c].view(np.int64) - ref_lf[:, c].view(np.int64))
        assert ulps.max() <= 1, (c, ulps.max())
    assert lf[0, 1] == 1.0 and lf[1, 1] == 1.0


def test_refusals_match_load_cooc_bin(tmp_path):
    from glove_tensorflow_b200.data_utils import load_cooc_bin
    from glove_tensorflow_b200.stanford_glove import StanfordGlove
    w1, w2, val = make_table("zipf", 50, 1000, 2)
    cases = []
    for k, (a, b, v) in enumerate(((0, 3, 1.0), (3, 51, 1.0), (3, 3, 0.0), (3, 3, np.inf), (3, 3, np.nan))):
        x1, x2, xv = w1.copy(), w2.copy(), val.copy()
        x1[700], x2[700], xv[700] = a, b, v
        x1[900] = 0
        cases.append(write_bin(tmp_path / ("bad%d.bin" % k), x1, x2, xv))
    trunc = tmp_path / "trunc.bin"
    trunc.write_bytes(open(write_bin(tmp_path / "ok.bin", w1, w2, val), "rb").read()[:-5])
    for path in cases + [str(trunc)]:
        with pytest.raises(ValueError) as want:
            load_cooc_bin(path, 50, chunk_bytes=16 * 300)
        with pytest.raises(ValueError) as got:
            StanfordGlove(path, 50, 4, chunk_bytes=16 * 300)
        assert str(got.value) == str(want.value)
    empty = tmp_path / "empty.bin"
    empty.write_bytes(b"")
    with pytest.raises(ValueError, match="no co-occurrence records"):
        StanfordGlove(str(empty), 50, 4)


def _oracle_run(sg, epochs, eta=0.05, clip=100.0):
    W = sgo.init_params(sg.V, sg.d, 7)
    G = np.ones_like(W)
    words, lf = sg.words.cpu().numpy(), sg.lf.cpu().numpy()
    out = []
    for _ in range(epochs):
        out.append(sgo.kernel_cost(sgo.epoch(W, G, words, lf, eta, clip, order=1)))
    return W, G, out


@pytest.mark.parametrize("d", [2, 31, 32, 33, 50, 64, 300, 510])
@pytest.mark.parametrize("kind", ["serial", "free", "zipf"])
def test_bit_identical_to_the_kernel_order_oracle(tmp_path, kind, d):
    from glove_tensorflow_b200.stanford_glove import StanfordGlove
    V, n = {"serial": (3000, 20_000), "free": (40_000, 40_000), "zipf": (50_000, 1_000_000)}[kind]
    path = write_bin(tmp_path / "c.bin", *make_table(kind, V, n, d))
    sg = StanfordGlove(path, V, d, seed=7)
    np.testing.assert_array_equal(sg.W.cpu().numpy(), sgo.init_params(V, d, 7))
    W1, G1, c1 = _oracle_run(sg, 1)
    got1 = sg.epoch()
    np.testing.assert_array_equal(sg.W.cpu().numpy(), W1)
    np.testing.assert_array_equal(sg.gradsq.cpu().numpy(), G1)
    assert got1 == c1[0]
    W3, G3, c3 = _oracle_run(sg, 3)
    got = [got1, sg.epoch(), sg.epoch()]
    np.testing.assert_array_equal(sg.W.cpu().numpy(), W3)
    np.testing.assert_array_equal(sg.gradsq.cpu().numpy(), G3)
    assert got == c3


def test_same_bits_for_one_cta_full_grid_and_reruns(tmp_path):
    from glove_tensorflow_b200.stanford_glove import StanfordGlove
    V = 20_000
    path = write_bin(tmp_path / "c.bin", *make_table("zipf", V, 400_000, 5))
    runs = []
    for grid in (0, 1, 0, 37):
        sg = StanfordGlove(path, V, 50, seed=3)
        costs = [sg.epoch(grid=grid) for _ in range(2)]
        runs.append((sg.W.cpu().numpy(), sg.gradsq.cpu().numpy(), costs))
    for W, G, c in runs[1:]:
        np.testing.assert_array_equal(W, runs[0][0])
        np.testing.assert_array_equal(G, runs[0][1])
        assert c == runs[0][2]


def test_resume_is_exact(tmp_path):
    from glove_tensorflow_b200 import stanford_glove as sg
    V = 300
    path = write_bin(tmp_path / "c.bin", *make_table("zipf", V, 20_000, 6))
    vocab = tmp_path / "vocab.txt"
    vocab.write_text("".join("w%d %d\n" % (i, 1000 - i) for i in range(V)))
    common = ["--input-file", path, "--vocab-file", str(vocab), "--vector-size", "33", "--seed", "4"]
    full = sg.main(common + ["--iter", "2", "--binary", "2", "--save-file", str(tmp_path / "full"), "--save-gradsq",
                             "--gradsq-file", str(tmp_path / "gfull")])
    one = sg.main(common + ["--iter", "1", "--binary", "1", "--save-file", str(tmp_path / "one"), "--save-gradsq",
                            "--gradsq-file", str(tmp_path / "g1")])
    two = sg.main(common + ["--iter", "1", "--binary", "2", "--save-file", str(tmp_path / "two"), "--save-gradsq",
                            "--gradsq-file", str(tmp_path / "g2"), "--init-param-file", str(tmp_path / "one.bin"),
                            "--init-gradsq-file", str(tmp_path / "g1.bin")])
    assert one == full[:1] and two == full[1:]
    for a, b in (("full.bin", "two.bin"), ("gfull.bin", "g2.bin"), ("full.txt", "two.txt")):
        assert open(tmp_path / a, "rb").read() == open(tmp_path / b, "rb").read()
    W = np.fromfile(tmp_path / "full.bin", "<f8").reshape(2 * V, 34)
    assert not os.path.exists(tmp_path / "one.txt")
    words = [ln.split(" ", 1)[0] for ln in open(tmp_path / "full.txt")]
    assert words == ["w%d" % i for i in range(V)] + ["<unk>"]
    from glove_tensorflow_b200.vectors import read_vectors
    _, rows = read_vectors(str(tmp_path / "full.txt"))
    np.testing.assert_array_equal(rows.cpu().numpy(), sgo.rows(W, 2))
    with pytest.raises(ValueError, match="bytes"):
        sg.main(common + ["--iter", "1", "--vector-size", "32", "--init-param-file", str(tmp_path / "one.bin")])


@pytest.mark.parametrize("model", [0, 1, 2])
def test_model_rows_and_header(tmp_path, model):
    from glove_tensorflow_b200 import stanford_glove as sg
    from glove_tensorflow_b200.vectors import read_vectors
    V = 150
    path = write_bin(tmp_path / "c.bin", *make_table("zipf", V, 5000, 8))
    vocab = tmp_path / "vocab.txt"
    vocab.write_text("".join("w%d\n" % i for i in range(V)))      # plain one-token lines
    sg.main(["--input-file", path, "--vocab-file", str(vocab), "--vector-size", "6", "--iter", "2", "--model", str(model),
             "--binary", "2", "--write-header", "--save-file", str(tmp_path / "v")])
    W = np.fromfile(tmp_path / "v.bin", "<f8").reshape(2 * V, 7)
    first = open(tmp_path / "v.txt").readline().split()
    assert first == [str(V + 1), str(14 if model == 0 else 6)]
    _, rows = read_vectors(str(tmp_path / "v.txt"))
    np.testing.assert_array_equal(rows.cpu().numpy(), sgo.rows(W, model))
    sg.main(["--input-file", path, "--vocab-file", str(vocab), "--vector-size", "6", "--iter", "1", "--model", str(model),
             "--no-unk-vector", "--save-file", str(tmp_path / "n")])
    assert sum(1 for _ in open(tmp_path / "n.txt")) == V


def test_corpus_to_stanford_glove_to_evaluation(tmp_path, capsys):
    from glove_tensorflow_b200 import corpus, evaluate_embeddings as ev, stanford_glove as sg
    from glove_tensorflow_b200.data_utils import read_stanford_vocab
    from glove_tensorflow_b200.vectors import read_vectors
    rng = np.random.default_rng(12)
    p = 1.0 / np.arange(1, 501) ** 1.1
    lines = [" ".join("w%d" % k for k in rng.choice(500, int(rng.integers(3, 30)), p=p / p.sum())) for _ in range(4000)]
    (tmp_path / "c.txt").write_text("\n".join(lines) + "\n")
    dest = tmp_path / "data"
    corpus.main(["--corpus", str(tmp_path / "c.txt"), "--dest", str(dest), "--scheme", "stanford", "--min-count", "3"])
    tokens, _ = read_stanford_vocab(str(dest / "vocab.txt"))
    out = str(tmp_path / "vectors")
    costs = sg.main(["--input-file", str(dest / "cooccurrence.shuf.bin"), "--vocab-file", str(dest / "vocab.txt"),
                     "--vector-size", "20", "--iter", "6", "--save-file", out])
    assert all(b < a for a, b in zip(costs, costs[1:])), costs
    assert "iter: 006, cost: " in capsys.readouterr().out
    words, rows = read_vectors(out + ".txt")
    assert words == list(tokens) + ["<unk>"]
    state = sg.StanfordGlove(str(dest / "cooccurrence.shuf.bin"), len(tokens), 20)
    for _ in range(6):
        state.epoch()
    np.testing.assert_array_equal(rows.cpu().numpy(), state.rows(2, True).cpu().numpy())
    sf = tmp_path / "s.txt"
    sf.write_text("w0 w1 1.0\nw2 w3 2.0\nw1 w4 3.0\n", encoding="utf8")
    rep = ev.main(["--vectors-txt", out + ".txt", "--similarity", str(sf), "--output-json", str(tmp_path / "r.json")])
    assert rep["similarity"][0]["found"] == 3
