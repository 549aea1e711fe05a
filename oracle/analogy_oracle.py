"""NumPy float64 restatement of the intrinsic evaluation (glove_tensorflow_b200/evaluate_embeddings.py and
glove_analogy.cu): word analogies by 3CosAdd (Stanford GloVe eval/python/evaluate.py) and 3CosMul (Levy & Goldberg
2014), word-pair cosines and the two correlations.  Test infrastructure only: the product never imports it."""
import numpy as np

EPS_MUL = 1e-3


def normalise(W):
    """Rows scaled by 1 / sqrt(max(sum x^2, 1e-12)) -- tf.math.l2_normalize, as the top-k normalises."""
    W = np.asarray(W, np.float64)
    return W / np.sqrt(np.maximum((W * W).sum(1, keepdims=True), 1e-12))


def _topk_excluding(score, exclude, k):
    """k best columns per row, descending, ties -> lower id, the ids in ``exclude`` [n, 3] skipped."""
    score = score.copy()
    np.put_along_axis(score, np.asarray(exclude, np.int64), -np.inf, axis=1)
    idx = np.argsort(-score, axis=1, kind="stable")[:, :k]
    return np.take_along_axis(score, idx, 1), idx


def analogy_scores(W, abc, method="add", restrict=None):
    """[n, V'] scores of every candidate row (the first ``restrict`` rows) for each question (a, b, c)."""
    Wn = normalise(W)
    cand = Wn if restrict is None else Wn[:restrict]
    abc = np.asarray(abc, np.int64).reshape(-1, 3)
    a, b, c = Wn[abc[:, 0]], Wn[abc[:, 1]], Wn[abc[:, 2]]
    if method == "add":
        q = normalise(b - a + c)             # the cosine with q; the argmax is that of evaluate.py's W_norm @ q
        return q @ cand.T
    if method == "mul":
        ca, cb, cc = a @ cand.T, b @ cand.T, c @ cand.T
        return ((1 + cb) / 2) * ((1 + cc) / 2) / ((1 + ca) / 2 + EPS_MUL)
    raise ValueError(method)


def analogy_topk(W, abc, k=1, method="add", restrict=None):
    """(scores [n, k], ids [n, k]): the k best candidates outside {a, b, c}, descending, ties -> lower id."""
    abc = np.asarray(abc, np.int64).reshape(-1, 3)
    return _topk_excluding(analogy_scores(W, abc, method, restrict), abc, k)


def pair_cosine(W, pairs):
    Wn = normalise(W)
    pairs = np.asarray(pairs, np.int64).reshape(-1, 2)
    return (Wn[pairs[:, 0]] * Wn[pairs[:, 1]]).sum(1)


def average_ranks(x):
    """Ranks 1..n, ties share their average rank (scipy.stats.rankdata 'average')."""
    x = np.asarray(x, np.float64)
    lt = (x[None, :] < x[:, None]).sum(1)
    eq = (x[None, :] == x[:, None]).sum(1)
    return lt + (eq + 1) / 2.0


def pearson(x, y):
    x, y = np.asarray(x, np.float64), np.asarray(y, np.float64)
    if len(x) < 2:
        return None
    dx, dy = x - x.mean(), y - y.mean()
    den = np.sqrt((dx * dx).sum() * (dy * dy).sum())
    return float((dx * dy).sum() / den) if den > 0 else None


def spearman(x, y):
    if len(x) < 2:
        return None
    return pearson(average_ranks(x), average_ranks(y))


def analogy_report(W, vocab, sections, restrict=None, case_sensitive=False, methods=("add", "mul")):
    """The analogy part of the evaluation report from a table W [V, d] and string questions:
    ``sections`` = [(name, [(a, b, c, d), ...])].  Lookup: first line wins, lower() on both sides unless case_sensitive;
    only the first ``restrict`` words; a question with an unknown word is not seen; correct = top-1 spells d."""
    n = len(vocab) if restrict is None else min(restrict, len(vocab))
    fold = (lambda w: w) if case_sensitive else (lambda w: w.lower())
    ids = {}
    for i in range(n):
        ids.setdefault(fold(vocab[i]), i)
    rows, groups = [], {g: [0, 0, {m: 0 for m in methods}] for g in ("semantic", "syntactic", "overall")}
    for name, qs in sections:
        known = [q for q in qs if all(fold(w) in ids for w in q)]
        correct = {m: 0 for m in methods}
        if known:
            abc = np.array([[ids[fold(w)] for w in q[:3]] for q in known])
            for m in methods:
                _, top = analogy_topk(W, abc, 1, m, n)
                correct[m] = int(sum(fold(vocab[i]) == fold(q[3]) for i, q in zip(top[:, 0], known)))
        rows.append({"name": name, "total": len(qs), "seen": len(known), "correct": correct,
                     "accuracy": {m: (correct[m] / len(known) if known else None) for m in methods}})
        for g in ("syntactic" if name.startswith("gram") else "semantic", "overall"):
            groups[g][0] += len(qs)
            groups[g][1] += len(known)
            for m in methods:
                groups[g][2][m] += correct[m]
    out = {"sections": rows}
    for g, (total, seen, correct) in groups.items():
        out[g] = {"total": total, "seen": seen, "correct": correct,
                  "accuracy": {m: (c / seen if seen else None) for m, c in correct.items()}}
    return out


def similarity_report(W, vocab, pairs, restrict=None, case_sensitive=False):
    """``pairs`` = [(w1, w2, human score)] -> total / found / spearman / pearson."""
    n = len(vocab) if restrict is None else min(restrict, len(vocab))
    fold = (lambda w: w) if case_sensitive else (lambda w: w.lower())
    ids = {}
    for i in range(n):
        ids.setdefault(fold(vocab[i]), i)
    found = [(ids[fold(a)], ids[fold(b)], s) for a, b, s in pairs if fold(a) in ids and fold(b) in ids]
    cos = pair_cosine(W, [(a, b) for a, b, _ in found]) if found else np.zeros(0)
    human = [s for _, _, s in found]
    return {"total": len(pairs), "found": len(found), "spearman": spearman(human, cos), "pearson": pearson(human, cos)}


def planted_analogies(n_groups, D, seed=0):
    """A vocabulary and table [1 + 2 n_groups, D + 2] in which "w<g>" : "W<g>_off" :: "w<h>" : "W<h>_off" holds exactly:
    w<g> = [base_g, 1, 0], W<g>_off = [base_g, 0, 1] with |base_g| = 3 for every g, so b^ - a^ + c^ is the unit vector
    of the answer itself.  Row 0 is "<UNK>" (random)."""
    rng = np.random.default_rng(seed)
    vocab, rows = ["<UNK>"], [np.concatenate([rng.normal(size=D), [0.3, 0.3]])]
    for g in range(n_groups):
        base = rng.normal(size=D)
        base *= 3.0 / np.linalg.norm(base)
        vocab += ["w%d" % g, "W%d_off" % g]
        rows += [np.concatenate([base, [1.0, 0.0]]), np.concatenate([base, [0.0, 1.0]])]
    return vocab, np.array(rows, np.float32)


MUL_QT, MUL_TV, NUM_SMS = 8, 256, 148      # kMulQT, kMulTV (glove_analogy.cu), kNumSMs (glove_common.cuh)


def mul_plan(V, n):
    """(question tiles, table slices, rows per slice) of the 3CosMul scan for n questions over V rows -- mul_plan of
    glove_analogy.cu: at least two CTAs per SM, at most 64 slices and no more slices than 256-row tiles.  Slice s holds
    rows [s * rows_per_slice, min((s + 1) * rows_per_slice, V)) and sweeps them in 256-row tiles from its first row, one
    32-row warp list per tile section; the tests plant exact ties on these edges."""
    q_tiles = (n + MUL_QT - 1) // MUL_QT
    slices = min((2 * NUM_SMS + q_tiles - 1) // q_tiles, 64)
    if slices * MUL_TV > V:
        slices = (V + MUL_TV - 1) // MUL_TV
    slices = max(slices, 1)
    return q_tiles, slices, (V + slices - 1) // slices
