"""CPU checks of the intrinsic evaluation: the analogy / similarity file parsers, the word lookup, the report
aggregation (with a NumPy stand-in for the GPU engine), the float64 oracle against a transcription of Stanford GloVe's
evaluate.py and against scipy, and the argument errors of the C entries."""
import ctypes

import numpy as np
import pytest
import scipy.stats

from glove_tensorflow_b200 import evaluate_embeddings as ev
from oracle import analogy_oracle as ao


def _write(tmp_path, name, text):
    p = tmp_path / name
    p.write_text(text, encoding="utf8")
    return str(p)


# ---- parsers ---------------------------------------------------------------------------------------------------------
def test_parse_analogies_sections_blank_lines_and_headerless_start(tmp_path):
    p = _write(tmp_path, "q.txt", "a b c d\n\n: capital-common\nAthens Greece Baghdad Iraq\n  \n"
                                  ": gram1-adjective-to-adverb\namazing amazingly apparent apparently\n")
    got = ev.parse_analogies(p)
    assert [s for s, _ in got] == ["q.txt", "capital-common", "gram1-adjective-to-adverb"]
    assert got[0][1] == [(1, ("a", "b", "c", "d"))]
    assert got[1][1] == [(4, ("Athens", "Greece", "Baghdad", "Iraq"))]
    assert got[2][1] == [(7, ("amazing", "amazingly", "apparent", "apparently"))]
    assert [ev.is_syntactic(s) for s, _ in got] == [False, False, True]


@pytest.mark.parametrize("bad", ["a b c", "a b c d e"])
def test_parse_analogies_reports_malformed_line_number(tmp_path, bad):
    p = _write(tmp_path, "q.txt", ": s\na b c d\n\n%s\n" % bad)
    with pytest.raises(ValueError, match=r"q\.txt:4:"):
        ev.parse_analogies(p)


def test_parse_similarity_comments_extra_fields_and_errors(tmp_path):
    p = _write(tmp_path, "s.txt", "# word1 word2 score\n\ntiger cat 7.35\nbook paper 7.46 extra fields\n")
    assert ev.parse_similarity(p) == [(3, "tiger", "cat", 7.35), (4, "book", "paper", 7.46)]
    with pytest.raises(ValueError, match=r"s2\.txt:2:"):
        ev.parse_similarity(_write(tmp_path, "s2.txt", "a b 1\nonly two\n"))
    with pytest.raises(ValueError, match=r"s3\.txt:1: score"):
        ev.parse_similarity(_write(tmp_path, "s3.txt", "a b high\n"))


def test_word_lookup_case_folding_lowest_id_and_restrict():
    vocab = ["<UNK>", "the", "Paris", "paris", "France", "the", "PARIS"]
    w = ev.WordIds(vocab)
    assert w.get("paris") == 2 and w.get("PARIS") == 2 and w.get("the") == 1 and w.get("france") == 4
    assert w.get("berlin") is None
    cs = ev.WordIds(vocab, case_sensitive=True)
    assert cs.get("paris") == 3 and cs.get("PARIS") == 6 and cs.get("Paris") == 2 and cs.get("the") == 1
    assert cs.get("france") is None
    r = ev.WordIds(vocab, restrict=3)
    assert r.n == 3 and r.get("paris") == 2 and r.get("France") is None
    assert ev.WordIds(vocab, restrict=100).n == len(vocab)
    assert w.same_word(6, "paris") and not cs.same_word(6, "paris")


# ---- report with a NumPy stand-in for the engine -----------------------------------------------------------------------
class OracleEngine:
    """engine.analogy / engine.pair_cosine answered by the float64 oracle (the GPU tests hold the kernels to it)."""

    def __init__(self, W):
        self.W = W

    def analogy(self, abc, k=1, method="add", restrict=None):
        s, i = ao.analogy_topk(self.W, abc, k, method, restrict)
        return s.astype(np.float32), i.astype(np.int32)

    def pair_cosine(self, pairs):
        return ao.pair_cosine(self.W, pairs).astype(np.float32)


def test_report_aggregation_matches_the_oracle_report(tmp_path):
    vocab, W = ao.planted_analogies(6, 24)
    lines = [": capital-world", "w0 w0_off w1 w1_off", "w2 W2_OFF w3 w3_off", "w4 w4_off nope w5_off",
             ": gram2-opposite", "w1 w1_off w5 w5_off", "w3 w3_off w4 missing", "", ": family", "w0 w1 w2 w3"]
    p = _write(tmp_path, "q.txt", "\n".join(lines) + "\n")
    s = _write(tmp_path, "s.txt", "# pairs\nw0 w0_off 3\nw1 w2 1\nw3 absent 2\nw4 w5 2.5\n")
    rep = ev.evaluate(OracleEngine(W), vocab, [p], [s])
    a = rep["analogies"][0]
    assert a["file"] == p
    assert [(x["name"], x["total"], x["seen"]) for x in a["sections"]] == [("capital-world", 3, 2), ("gram2-opposite", 2, 1),
                                                                           ("family", 1, 1)]
    assert a["sections"][0]["correct"] == {"add": 2, "mul": 2} and a["sections"][0]["accuracy"]["add"] == 1.0
    assert (a["semantic"]["total"], a["semantic"]["seen"]) == (4, 3) and (a["syntactic"]["total"], a["syntactic"]["seen"]) == (2, 1)
    assert a["overall"]["seen"] == 4 and a["overall"]["correct"]["add"] == a["semantic"]["correct"]["add"] + a["syntactic"]["correct"]["add"]
    assert a["overall"]["accuracy"]["add"] == a["overall"]["correct"]["add"] / 4
    want = ao.analogy_report(W, vocab, [(n, [q for _, q in qs]) for n, qs in ev.parse_analogies(p)])
    assert {k: a[k] for k in want} == want
    sim = rep["similarity"][0]
    assert (sim["total"], sim["found"]) == (4, 3)
    want = ao.similarity_report(W, vocab, [(x, y, z) for _, x, y, z in ev.parse_similarity(s)])
    assert sim["file"] == s and sim["spearman"] == want["spearman"] and abs(sim["pearson"] - want["pearson"]) < 1e-6
    # restricted vocabulary: words past the first N lines are unseen, candidates are the first N rows
    rep = ev.evaluate(OracleEngine(W), vocab, [p], [], restrict_vocab=7)
    want = ao.analogy_report(W, vocab, [(n, [q for _, q in qs]) for n, qs in ev.parse_analogies(p)], restrict=7)
    assert {k: rep["analogies"][0][k] for k in want} == want and want["overall"]["seen"] == 1


def test_aggregate_with_nothing_seen():
    out = ev.aggregate_analogies([("gram1-x", 5, 0, {"add": 0, "mul": 0})])
    assert out["syntactic"]["accuracy"] == {"add": None, "mul": None}
    assert out["semantic"] == {"total": 0, "seen": 0, "correct": {"add": 0, "mul": 0}, "accuracy": {"add": None, "mul": None}}


# ---- oracle ------------------------------------------------------------------------------------------------------------
def stanford_evaluate_top1(W, indices, split_size=100):
    """The argmax loop of Stanford GloVe eval/python/evaluate.py (evaluate_vectors), transcribed."""
    d = (np.sum(W ** 2, 1) ** 0.5)
    W = (W.T / d).T
    ind1, ind2, ind3 = indices.T[:3]
    predictions = np.zeros((len(indices),))
    num_iter = int(np.ceil(len(indices) / float(split_size)))
    for j in range(num_iter):
        subset = np.arange(j * split_size, min((j + 1) * split_size, len(ind1)))
        pred_vec = (W[ind2[subset], :] - W[ind1[subset], :] + W[ind3[subset], :])
        dist = np.dot(W, pred_vec.T)
        for k in range(len(subset)):
            dist[ind1[subset[k]], k] = -np.inf
            dist[ind2[subset[k]], k] = -np.inf
            dist[ind3[subset[k]], k] = -np.inf
        predictions[subset] = np.argmax(dist, 0).flatten()
    return predictions.astype(np.int64)


def test_oracle_add_top1_matches_stanford_loop():
    rng = np.random.default_rng(1)
    W = rng.normal(size=(500, 20))
    W[7] = W[3] * 2.5                     # a duplicate direction under a higher id: a tie, the lower id wins
    abc = rng.integers(0, 500, (257, 3))
    abc[:5] = [[3, 4, 5], [4, 3, 3], [1, 1, 1], [9, 7, 2], [5, 5, 8]]
    _, idx = ao.analogy_topk(W, abc, 1, "add")
    np.testing.assert_array_equal(idx[:, 0], stanford_evaluate_top1(W, abc))


def test_oracle_mul_excludes_ties_and_formula():
    rng = np.random.default_rng(2)
    W = rng.normal(size=(60, 8))
    W[11] = W[10]                         # exact duplicate candidates: the lower id comes first
    abc = np.array([[0, 1, 2], [3, 3, 4]])
    s, idx = ao.analogy_topk(W, abc, 59 - 3, "mul")
    for q in range(2):
        assert not set(idx[q]) & set(abc[q])
        assert np.all(np.diff(s[q]) <= 0)
        i10, i11 = list(idx[q]).index(10), list(idx[q]).index(11)
        assert i11 == i10 + 1
    Wn = ao.normalise(W)
    x = Wn[20]
    ca, cb, cc = Wn[0] @ x, Wn[1] @ x, Wn[2] @ x
    want = ((1 + cb) / 2) * ((1 + cc) / 2) / ((1 + ca) / 2 + 1e-3)
    assert abs(s[0][list(idx[0]).index(20)] - want) < 1e-15


def test_oracle_normalisation_floor():
    W = np.zeros((3, 4))
    W[1] = [1e-8, 0, 0, 0]
    n = ao.normalise(W)
    assert np.all(n[0] == 0) and abs(n[1][0] - 1e-8 / 1e-6) < 1e-18


def test_mul_plan_restates_the_kernel():
    """The 3CosMul slicing the edge tests plant ties against: the constants are the kernel's, every row is in exactly one
    non-empty slice, and the extremes fall where the GPU tests expect them."""
    import os
    import re
    csrc = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "glove_tensorflow_b200", "csrc")
    src = open(os.path.join(csrc, "glove_analogy.cu")).read()
    assert int(re.search(r"constexpr int kMulQT = (\d+);", src).group(1)) == ao.MUL_QT
    assert int(re.search(r"constexpr int kMulTV = (\d+);", src).group(1)) == ao.MUL_TV
    assert "if (slices > 64) slices = 64;" in src and "(2 * kNumSMs + p.q_tiles - 1) / p.q_tiles" in src
    common = open(os.path.join(csrc, "glove_common.cuh")).read()
    assert int(re.search(r"constexpr int kNumSMs = (\d+);", common).group(1)) == ao.NUM_SMS
    for V in (4, 31, 255, 256, 257, 1023, 1024, 5249, 16384, 16411, 20000, 400000):
        for n in (1, 7, 8, 9, 300, 2368, 2369, 2500):
            q_tiles, slices, rps = ao.mul_plan(V, n)
            assert q_tiles * ao.MUL_QT >= n > (q_tiles - 1) * ao.MUL_QT
            assert 1 <= slices <= 64 and (slices - 1) * rps < V <= slices * rps
            assert slices <= (V + ao.MUL_TV - 1) // ao.MUL_TV     # no more slices than 256-row tiles
    assert ao.mul_plan(16384, 1) == (1, 64, 256) and ao.mul_plan(20000, 9) == (2, 64, 313)
    assert ao.mul_plan(20000, 2368)[1] == 1 and ao.mul_plan(5249, 2369)[1] == 1 and ao.mul_plan(5249, 2360)[1] == 2
    assert ao.mul_plan(255, 1) == (1, 1, 255) and ao.mul_plan(257, 1) == (1, 2, 129)


def test_correlations_match_scipy():
    rng = np.random.default_rng(3)
    for n in (2, 5, 40, 300):
        x = np.round(rng.normal(size=n), 1)          # many ties
        y = x + rng.normal(size=n)
        y[: n // 4] = y[0]
        for f_ours in (ao, ev):
            assert abs(f_ours.spearman(x, y) - scipy.stats.spearmanr(x, y).statistic) < 1e-12
            assert abs(f_ours.pearson(x, y) - scipy.stats.pearsonr(x, y).statistic) < 1e-12
        np.testing.assert_array_equal(ev.average_ranks(x), scipy.stats.rankdata(x))
        np.testing.assert_array_equal(ao.average_ranks(x), scipy.stats.rankdata(x))
    assert ev.spearman([1.0], [2.0]) is None and ev.pearson([1, 1, 1], [1, 2, 3]) is None


# ---- C entries: argument errors before the device is touched -------------------------------------------------------
def test_analogy_entries_argument_errors_without_a_gpu():
    from glove_tensorflow_b200 import _lib
    lib = _lib.lib
    nz = ctypes.c_void_p(256)        # non-null, never dereferenced
    ADD, MUL = _lib.ANALOGY_METHODS["add"], _lib.ANALOGY_METHODS["mul"]

    def call(table=nz, V=1000, d=16, planes=1, nb=None, inv=nz, abc=nz, n=4, method=ADD, k=1, score=nz, idx=nz, ws=nz,
             wsb=1 << 40):
        return lib.glove_analogy_topk(table, V, d, planes, nb, inv, abc, n, method, k, score, idx, ws, wsb, None)

    for kw in (dict(table=None), dict(inv=None), dict(abc=None), dict(score=None), dict(idx=None), dict(ws=None)):
        assert call(**kw) == _lib.EINVAL and b"glove_analogy_topk" in lib.glove_last_error()
    assert call(n=0) == _lib.EINVAL and call(V=0) == _lib.EINVAL and call(planes=0) == _lib.EINVAL
    assert call(method=2) == _lib.EUNSUPPORTED and b"method" in lib.glove_last_error()
    for k in (0, 30, -1):
        assert call(k=k) == _lib.EUNSUPPORTED and b"k=" in lib.glove_last_error()
    assert call(V=5, k=3) == _lib.EUNSUPPORTED and call(method=MUL, V=5, k=3) == _lib.EUNSUPPORTED
    assert call(d=511) == _lib.EUNSUPPORTED
    assert call(wsb=16) == _lib.EWORKSPACE
    need = lib.glove_analogy_workspace_bytes(1000, 16, 4, 1, ADD)
    assert need > 0 and lib.glove_analogy_workspace_bytes(1000, 16, 4, 1, MUL) > 0
    assert call(wsb=need - 1) == _lib.EWORKSPACE
    assert lib.glove_analogy_workspace_bytes(1000, 16, 4, 1, 7) == 0 and lib.glove_analogy_workspace_bytes(0, 16, 4, 1, ADD) == 0
    pc = lib.glove_pair_cosine
    assert pc(None, 10, 16, 1, nz, nz, 3, nz, None) == _lib.EINVAL and b"glove_pair_cosine" in lib.glove_last_error()
    assert pc(nz, 10, 16, 1, None, nz, 3, nz, None) == _lib.EINVAL and pc(nz, 10, 16, 1, nz, None, 3, nz, None) == _lib.EINVAL
    assert pc(nz, 10, 16, 1, nz, nz, 0, nz, None) == _lib.EINVAL and pc(nz, 10, 16, 0, nz, nz, 3, nz, None) == _lib.EINVAL
    assert pc(nz, 10, 511, 1, nz, nz, 3, nz, None) == _lib.EUNSUPPORTED



def test_get_analogies_strings_and_scores():
    from glove_tensorflow_b200.model_utils import get_analogies
    vocab, W = ao.planted_analogies(6, 24)
    out = get_analogies(OracleEngine(W), [("w0", "W0_off", "w1"), ("w2", "W2_off", "w5")], vocab, top_k=2, method="mul")
    assert out["input_strings"] == [["w0", "W0_off", "w1"], ["w2", "W2_off", "w5"]]
    assert [r[0] for r in out["top_k_string"]] == ["W1_off", "W5_off"] and out["top_k_score"].shape == (2, 2)
    with pytest.raises(KeyError, match="w0_off"):
        get_analogies(OracleEngine(W), [("w0", "w0_off", "w1")], vocab)      # exact lookup: the vocab spells W0_off
