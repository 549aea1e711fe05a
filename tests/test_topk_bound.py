"""The tensor-core top-k ranks candidates with bf16 products and re-scores them in fp32; a query whose k-th exact score is
not safely above the bf16 cut-off goes to the exact scan.  This file builds the adversarial table the GPU test of that
check uses (tests/test_kernel_edges_gpu.py) and proves on the CPU, by emulating the bf16 candidate pass, that the table
is adversarial: the query loses ~2^-7 of its self-similarity to bf16 rounding, 32 other rows outrank it, and a bound of
4e-3 on |bf16 score - exact score| would accept the wrong answer while the true bound (2^-7 + 2^-16 + slack = 8e-3)
sends the query to the exact scan.  If someone changes the generator so that it stops being adversarial, this fails."""
import numpy as np
import pytest

KP = 32                 # candidates kept per (query, table slice) by the tensor-core pass (TC_KP)
OLD_DELTA = 4.0e-3      # the bound the check used to assume ("2^-8 + slack")
DELTA = 8.0e-3          # 2^-7 + 2^-16 + slack (TC_DELTA)
MARGIN = 1e-4           # every quantity that decides the outcome is at least this far from its rival


def bf16_round(x):
    """fp32 -> bf16 -> fp32 with round-to-nearest-even (__float2bfloat16 for finite values)."""
    b = np.ascontiguousarray(x, np.float32).view(np.uint32).astype(np.uint64)
    b = (b + 0x7FFF + ((b >> 16) & 1)) & 0xFFFF0000
    return b.astype(np.uint32).view(np.float32)


def normalise_fp32(T):
    """tf.math.l2_normalize in fp32, as the normalisation kernel computes it (up to summation order)."""
    T = np.asarray(T, np.float32)
    ss = np.sum(T * T, axis=1, dtype=np.float32, keepdims=True)
    return T * (np.float32(1) / np.sqrt(np.maximum(ss, np.float32(1e-12))))


def adversarial_table(V=2048, d=256, k=1, start=0, stride=1, seed=0, near_cos=0.9985, filler_bf16=0.9935):
    """Table whose row `start` (and, for k > 1, its k - 1 exact copies) is misranked by the bf16 candidate pass.

    Block layout, at ids start + stride * (0, 1, ...):
      k copies of the query q: all but two of its 256 normalised components are +-2^-4 (1 + 2^-8 - 2^-13), just below a
        bf16 rounding midpoint, so every one of them rounds DOWN by ~2^-8 and bf16(q).bf16(q) ~ 1 - 2^-7 = 0.9925;
      k "near" rows at exact cosine `near_cos` to q (bf16 score ~0.9948);
      KP - k fillers at a slightly lower exact cosine, chosen so that their bf16 score is `filler_bf16`.
    KP rows outrank the query in bf16, so the query is not among its own candidates; the k-th exact candidate score is a
    near row at 0.9985, more than 4e-3 but less than 8e-3 above the cut-off.  Every other row is N(0, 0.05^2).
    Returns (T [V, d] fp32, ids of the query copies, ids of the near rows, ids of the fillers)."""
    assert d == 256, "the query construction needs components of 2^-4"
    rng = np.random.default_rng(seed)
    T = rng.normal(0.0, 0.05, (V, d))
    a = 2.0 ** -4 * (1 + 2.0 ** -8 - 2.0 ** -13)
    q = np.empty(d)
    q[: d - 2] = a * rng.choice([-1.0, 1.0], d - 2)
    q[d - 2:] = np.sqrt((1.0 - (d - 2) * a * a) / 2.0)        # the rest of the unit norm
    q = q.astype(np.float32).astype(np.float64)
    qb = bf16_round(normalise_fp32(q[None]))[0].astype(np.float64)
    c_fill = filler_bf16 / float(qb @ q)                       # bf16(q) . x ~ (bf16(q) . q) cos(q, x) for x = cos q + sin u, u _|_ q

    def at_cos(c):
        u = rng.normal(size=d)
        u -= (u @ q) / (q @ q) * q
        u /= np.linalg.norm(u)
        return c * q / np.linalg.norm(q) + np.sqrt(1.0 - c * c) * u

    ids = start + stride * np.arange(KP + k)
    assert ids[-1] < V
    T[ids[:k]] = q
    for i in ids[k:2 * k]:
        T[i] = at_cos(near_cos)
    for i in ids[2 * k:]:
        T[i] = at_cos(c_fill)
    return T.astype(np.float32), ids[:k], ids[k:2 * k], ids[2 * k:]


def emulate_candidate_pass(T, qid, k):
    """What the tensor-core pass and the guarantee check decide for query `qid` with the whole table in one slice:
    bf16 scores (exact products, fp64 sums), the top-KP candidate list, its cut-off, the exact (fp64) scores."""
    tn = normalise_fp32(T)
    tb = bf16_round(tn).astype(np.float64)
    bf = tb @ tb[qid]
    order = np.argsort(-bf, kind="stable")
    cand, rest = order[:KP], order[KP:]
    t64 = T.astype(np.float64)
    t64 /= np.linalg.norm(t64, axis=1, keepdims=True)
    exact = t64 @ t64[qid]
    cand_exact = np.sort(exact[cand])[::-1]
    return {"bf16": bf, "exact": exact, "cand": cand, "cut": float(bf[cand[-1]]), "best_outside": float(bf[rest[0]]),
            "kth_cand_exact": float(cand_exact[k - 1]), "next_cand_exact": float(cand_exact[k])}


@pytest.mark.parametrize("k,start,stride", [(1, 0, 1), (5, 0, 1), (1, 120, 1), (5, 120, 1), (1, 0, 2)])
def test_adversarial_table_defeats_the_old_bound(k, start, stride):
    T, queries, near, fill = adversarial_table(k=k, start=start, stride=stride)
    for qid in queries:
        e = emulate_candidate_pass(T, qid, k)
        deficit = 1.0 - e["bf16"][qid]
        assert deficit > 6e-3, deficit                          # ~2^-7: twice what a 2^-8 bound allows for
        assert not set(queries) & set(e["cand"])                # the query and its copies are not candidates ...
        assert set(e["cand"]) == set(near) | set(fill)          # ... the near rows and the fillers are
        assert e["cut"] - e["best_outside"] >= MARGIN           # (33rd bf16 score = the query's own)
        assert np.all(e["exact"][near] - e["exact"][fill].max() >= MARGIN)   # the wrong answer would be the near rows
        assert e["exact"][qid] - e["kth_cand_exact"] >= MARGIN  # which are wrong: the query itself is the top-1
        # the old check accepts the candidates' answer, the new one sends the query to the exact scan
        assert e["kth_cand_exact"] - (e["cut"] + OLD_DELTA) >= MARGIN, (e["kth_cand_exact"], e["cut"])
        assert (e["cut"] + DELTA) - e["kth_cand_exact"] >= MARGIN, (e["kth_cand_exact"], e["cut"])
        # rows outside the block are far away: no other table slice can raise the cut-off
        outside = np.setdiff1d(np.arange(len(T)), np.concatenate([queries, near, fill]))
        assert e["bf16"][outside].max() < 0.5


def test_bound_covers_the_worst_case_rounding():
    """2^-7 + 2^-16 is attained: x rounded down by a relative 2^-8 (minus a hair) on every component of both factors."""
    worst = (1 + 2.0 ** -8) ** 2 - 1
    assert worst == pytest.approx(2.0 ** -7 + 2.0 ** -16)
    assert OLD_DELTA < worst < DELTA
    x = np.float32(2.0 ** -4 * (1 + 2.0 ** -8 - 2.0 ** -13))
    assert bf16_round(np.array([x]))[0] == np.float32(2.0 ** -4)                 # just below the midpoint: rounds down
    assert bf16_round(np.array([np.float32(2.0 ** -4 * (1 + 2.0 ** -8))]))[0] == np.float32(2.0 ** -4)  # tie -> even
    assert bf16_round(np.array([np.float32(2.0 ** -4 * (1 + 3 * 2.0 ** -8))]))[0] == np.float32(2.0 ** -4 * (1 + 2.0 ** -6))


def test_kernel_uses_this_bound():
    import os
    import re
    src = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "glove_tensorflow_b200", "csrc",
                       "glove_topk_tc.cu")
    m = re.search(r"constexpr float TC_DELTA = ([0-9.eE+-]+)f;", open(src).read())
    assert m and float(m.group(1)) == DELTA
