"""Word analogies (3CosAdd, 3CosMul) and pair cosines on the GPU against the float64 oracle (oracle/analogy_oracle.py),
and the evaluate_embeddings CLI end to end."""
import json
import os

import numpy as np
import pytest

from oracle import analogy_oracle as ao

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "text8_small")


def _engine(W, optimizer="SGD"):
    from glove_tensorflow_b200.engine import GloveEngine
    V, d = W.shape
    eng = GloveEngine(V, d, optimizer=optimizer, batch_size=64, plan_steps=1, max_steps=4)
    z = np.zeros(V, np.float32)
    eng.load_state(W, np.zeros_like(W), z, z)
    return eng


def _check(W, abc, k, method, restrict, score, idx):
    """Scores within 1e-5 (relative above 1) of the float64 oracle; ids equal, except where the oracle's own scores of
    the two ids are within fp32 noise of each other."""
    want_s, want_i = ao.analogy_topk(W, abc, k, method, restrict)
    full = ao.analogy_scores(W, abc, method, restrict)
    tol = 1e-5 * np.maximum(1.0, np.abs(want_s))
    assert np.all(np.abs(score - want_s) <= tol), float(np.max(np.abs(score - want_s) / np.maximum(1.0, np.abs(want_s))))
    V = W.shape[0] if restrict is None else restrict
    assert idx.min() >= 0 and idx.max() < V
    for q in range(len(abc)):
        assert len(set(idx[q])) == k and not set(idx[q]) & set(abc[q])
        for j in np.nonzero(idx[q] != want_i[q])[0]:
            assert abs(full[q, idx[q, j]] - want_s[q, j]) <= tol[q, j], (q, j, idx[q, j], want_i[q, j])


@pytest.mark.parametrize("V", [700, 5000, 40000])
@pytest.mark.parametrize("d", [30, 64, 300])
def test_analogy_matches_oracle(V, d):
    rng = np.random.default_rng(V + d)
    W = rng.normal(size=(V, d)).astype(np.float32)
    eng = _engine(W, optimizer="Adam" if (V, d) == (5000, 64) else "SGD")   # a three-plane table once
    n = 37
    for restrict in (None, V // 3):
        R = V if restrict is None else restrict
        abc = rng.integers(0, R, (n, 3))
        abc[0, 2] = abc[0, 0]                                  # a repeated word
        for k in (1, 5, 21, 29):
            for method, exact in (("add", False), ("add", True), ("mul", False)):
                s, i = eng.analogy(abc, k, method, restrict=restrict, exact_fp32=exact)
                assert s.shape == i.shape == (n, k)
                _check(W, abc, k, method, restrict, s, i)


def test_exclusion_duplicates_and_ties():
    rng = np.random.default_rng(7)
    V, d = 3000, 64
    W = rng.normal(size=(V, d)).astype(np.float32)
    x, e = 10, rng.normal(size=d).astype(np.float32) * 1e-2
    W[11], W[12] = W[x] + e, W[x] - e          # b^ + c^ ~ 2 a^: the query's top-1 is a (or b, c)
    W[2001] = W[20]                            # a duplicate row of b under a higher id
    W[2500] = W[2600] = W[30] * 3              # exact duplicate candidates (the answer to (40, 30, 40))
    eng = _engine(W)
    abc = np.array([[x, 11, 12],               # a (and b, c) nearest to the query
                    [5, 20, 5],                # a == c: the query is b^, its top-1 is b itself
                    [6, 6, 21],                # a == b: the query is c^
                    [40, 30, 40]])             # best outside {30, 40}: the two copies of row 30, lower id first
    assert eng.topk([20], 2)[1][0].tolist() == [20, 2001]
    for method, exact in (("add", False), ("add", True), ("mul", False)):
        s, i = eng.analogy(abc, 5, method, exact_fp32=exact)
        _check(W, abc, 5, method, None, s, i)
        if method == "add":
            assert i[1, 0] == 2001 and abs(s[1, 0] - 1.0) < 1e-6
            assert i[3, :2].tolist() == [2500, 2600] and s[3, 0] == s[3, 1]
    with pytest.raises(ValueError, match="word ids"):
        eng.analogy([[0, 1, V]], 1)
    with pytest.raises(ValueError, match="word ids"):
        eng.analogy([[0, 1, 1000]], 1, restrict=1000)
    with pytest.raises(ValueError, match="method"):
        eng.analogy([[0, 1, 2]], 1, "sub")


def test_pair_cosine_is_the_topk_similarity_bit_for_bit():
    rng = np.random.default_rng(3)
    for V, d in ((800, 30), (5000, 300), (3000, 510)):
        W = rng.normal(size=(V, d)).astype(np.float32)
        eng = _engine(W)
        q = rng.integers(0, V, 40)
        for exact in (False, True):
            sim, idx = eng.topk(q, 8, exact_fp32=exact)
            pairs = np.stack([np.repeat(q, 8), idx.reshape(-1)], 1)
            got = eng.pair_cosine(pairs)
            np.testing.assert_array_equal(got.view(np.uint32), sim.reshape(-1).view(np.uint32))
        np.testing.assert_allclose(got, ao.pair_cosine(W, pairs), rtol=0, atol=1e-6)


def test_mul_is_deterministic():
    rng = np.random.default_rng(11)
    W = rng.normal(size=(20000, 300)).astype(np.float32)
    eng = _engine(W)
    abc = rng.integers(0, 20000, (300, 3))
    s1, i1 = eng.analogy(abc, 10, "mul")
    s2, i2 = eng.analogy(abc, 10, "mul")
    np.testing.assert_array_equal(s1.view(np.uint32), s2.view(np.uint32))
    np.testing.assert_array_equal(i1, i2)


def _job_with_table(tmp_path, vocab, W):
    from glove_tensorflow_b200 import config_utils, estimator, train_utils
    vt = tmp_path / "vocab.txt"
    vt.write_text("\n".join(vocab), encoding="utf8")
    job = str(tmp_path / "job")
    params = config_utils.parse_args(["--vocab-txt", str(vt), "--job-dir", job, "--disable-datetime-path", "--optimizer",
                                      "SGD", "--embedding-size", str(W.shape[1]), "--train-steps", "1"])
    eng = estimator.build_engine(params, load_coo=False)
    z = np.zeros(len(vocab), np.float32)
    eng.load_state(W, np.zeros_like(W), z, z)
    train_utils.save_checkpoint(eng, job)
    return job


def test_planted_analogies_score_100_percent_through_the_cli(tmp_path):
    from glove_tensorflow_b200 import evaluate_embeddings as ev
    vocab, W = ao.planted_analogies(600, 30)          # V = 1201: the tensor-core path of 3CosAdd
    rng = np.random.default_rng(0)
    gh = [(g, h) for g, h in rng.integers(0, 600, (400, 2)) if g != h]
    lines = [": capital-planted"] + ["w%d W%d_off w%d W%d_off" % (g, g, h, h) for g, h in gh[:200]]
    lines += [": gram3-planted"] + ["W%d w%d_OFF w%d w%d_off" % (g, g, h, h) for g, h in gh[200:]]
    lines += [": unseen-words", "w1 w1_off w2 absent", "nowhere w1_off w2 w2_off"]
    qf = tmp_path / "questions.txt"
    qf.write_text("\n".join(lines) + "\n", encoding="utf8")
    job = _job_with_table(tmp_path, vocab, W)
    out = str(tmp_path / "report.json")
    ev.main(["--job-dir", job, "--analogies", str(qf), "--output-json", out])
    rep = json.load(open(out))
    a = rep["analogies"][0]
    n_seen = len(gh)
    assert a["overall"]["seen"] == n_seen and a["overall"]["total"] == n_seen + 2
    assert a["overall"]["correct"] == {"add": n_seen, "mul": n_seen}
    assert a["sections"][2] == {"name": "unseen-words", "total": 2, "seen": 0, "correct": {"add": 0, "mul": 0},
                                "accuracy": {"add": None, "mul": None}}
    want = ao.analogy_report(W, vocab, [(n, [q for _, q in qs]) for n, qs in ev.parse_analogies(str(qf))])
    assert {k: a[k] for k in want} == want
    assert rep["global_step"] == 0 and rep["vectors"] == "row"


def test_text8_training_then_evaluation_matches_the_oracle(tmp_path):
    from glove_tensorflow_b200 import config_utils, data_utils, estimator, evaluate_embeddings as ev
    job = str(tmp_path / "job")
    params = config_utils.parse_args(["--train-csv", os.path.join(GOLD, "interaction.csv"), "--vocab-txt",
                                      os.path.join(GOLD, "vocab.txt"), "--job-dir", job, "--disable-datetime-path",
                                      "--embedding-size", "16", "--batch-size", "256", "--learning-rate", "0.05",
                                      "--seed", "2", "--plan-steps", "4", "--train-steps", "40"])
    estimator.train(params)
    vocab = data_utils.read_vocab(os.path.join(job, "vocab.txt"))
    qf, sf = tmp_path / "q.txt", tmp_path / "s.txt"
    qf.write_text(": family\nw4 w5 w6 w7\nw8 w9 w10 w11\nNULL none w12 w13\nw14 w15 w16 unknownword\n"
                  ": gram1-x\nw20 w21 w22 w23\nw30 w31 w32 w33\nw4 w4 w40 w41\n", encoding="utf8")
    sf.write_text("# handmade\nw4 w5 1.0\nw6 w7 2.5\nw8 w40 0.5\nw9 w41 3.0\nnan null 2.0\nw10 missing 1.0\n"
                  "w11 w12 4.0\nw13 w14 1.5\n", encoding="utf8")
    from glove_tensorflow_b200 import train_utils
    with np.load(train_utils.latest_checkpoint(job)) as z:
        tables = {"row": z["R"], "sum": z["R"] + z["C"]}
    for vectors in ("row", "sum"):
        for restrict in (None, 30):
            argv = ["--job-dir", job, "--analogies", str(qf), "--similarity", str(sf), "--vectors", vectors]
            if restrict:
                argv += ["--restrict-vocab", str(restrict)]
            rep = ev.main(argv)
            assert json.load(open(os.path.join(job, "intrinsic_eval.json"))) == json.loads(json.dumps(rep))
            W = tables[vectors]
            want = ao.analogy_report(W, vocab, [(n, [q for _, q in qs]) for n, qs in ev.parse_analogies(str(qf))], restrict)
            a = rep["analogies"][0]
            assert {k: a[k] for k in want} == want
            s = rep["similarity"][0]
            ws = ao.similarity_report(W, vocab, [(x, y, v) for _, x, y, v in ev.parse_similarity(str(sf))], restrict)
            assert (s["total"], s["found"]) == (ws["total"], ws["found"])
            assert abs(s["spearman"] - ws["spearman"]) < 1e-9 and abs(s["pearson"] - ws["pearson"]) < 1e-5
            assert a["overall"]["seen"] == (4 if restrict else 6) and s["found"] == (5 if restrict else 7)
