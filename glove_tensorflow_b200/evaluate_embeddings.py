"""``python -m glove_tensorflow_b200.evaluate_embeddings`` -- intrinsic evaluation of trained embeddings on the GPU:
word analogies (``questions-words.txt`` format, 3CosAdd and 3CosMul) and word-similarity rank correlation (WordSim-353 /
SimLex / MEN style ``w1 w2 score`` files), from a checkpoint of a job directory.

    python -m glove_tensorflow_b200.evaluate_embeddings --job-dir J [--checkpoint P] [--analogies FILE ...]
        [--similarity FILE ...] [--restrict-vocab N] [--vectors row|sum] [--case-sensitive] [--output-json PATH]
    python -m glove_tensorflow_b200.evaluate_embeddings --vectors-txt FILE [--dim D] --output-json PATH [...]

``--vectors-txt`` evaluates any word-vectors file in the GloVe text format (Stanford's trainer, the published glove.*
files, gensim's word2vec text format; see vectors.py), parsed on the GPU; the candidates and ``--restrict-vocab`` follow
the file's order (published files are in frequency order).

Conventions (Stanford GloVe ``eval/python/evaluate.py``; 3CosMul after Levy & Goldberg 2014): rows are l2-normalised,
the answer to a : b :: c : ? is the best row outside the ids of a, b and c, ties go to the lower id.  ``--restrict-vocab
N`` keeps the first N lines of vocab.txt (the most frequent words: the preprocessor writes it in frequency order) both as
candidates and for the lookup of the question words.  A question or pair with a word outside that vocabulary is skipped
and counted; accuracy is over the questions seen."""
import json
import logging
import os
import sys
from argparse import ArgumentParser

import numpy as np

logger = logging.getLogger(__name__)
METHODS = ("add", "mul")


# ---- files ------------------------------------------------------------------------------------------------------------
def parse_analogies(path):
    """``questions-words.txt`` format: ``a b c d`` per line, ``: name`` starts a section, blank lines are ignored.
    Returns [(section name, [(line number, (a, b, c, d)), ...]), ...]; questions before the first header go to a section
    named after the file.  A line without exactly four words raises ValueError naming the file and line."""
    sections = []
    with open(path, encoding="utf8") as f:
        for no, line in enumerate(f, 1):
            s = line.strip()
            if not s:
                continue
            if s.startswith(":"):
                sections.append((s[1:].strip(), []))
                continue
            words = s.split()
            if len(words) != 4:
                raise ValueError("%s:%d: an analogy line holds 4 words, found %d: %r" % (path, no, len(words), s))
            if not sections:
                sections.append((os.path.basename(path), []))
            sections[-1][1].append((no, tuple(words)))
    return sections


def parse_similarity(path):
    """``w1 w2 score`` per line (further fields ignored), ``#`` starts a comment line, blank lines are ignored.
    Returns [(line number, w1, w2, score), ...]; a line with fewer than three fields or a score that is not a number
    raises ValueError naming the file and line."""
    out = []
    with open(path, encoding="utf8") as f:
        for no, line in enumerate(f, 1):
            s = line.strip()
            if not s or s.startswith("#"):
                continue
            fields = s.split()
            if len(fields) < 3:
                raise ValueError("%s:%d: a similarity line holds 'w1 w2 score', found %r" % (path, no, s))
            try:
                score = float(fields[2])
            except ValueError:
                raise ValueError("%s:%d: score %r is not a number" % (path, no, fields[2])) from None
            out.append((no, fields[0], fields[1], score))
    return out


def is_syntactic(section):
    """``questions-words.txt`` convention: the syntactic sections are named gram1-... to gram9-..."""
    return section.startswith("gram")


class WordIds:
    """Token -> row id over the first ``restrict`` lines of vocab.txt: the first line holding a token wins; unless
    ``case_sensitive``, both sides are lower()-ed and the lowest id wins (gensim's case-insensitive lookup)."""

    def __init__(self, vocab, restrict=None, case_sensitive=False):
        self.vocab = list(vocab)
        self.n = len(self.vocab) if restrict is None else min(int(restrict), len(self.vocab))
        self.fold = (lambda w: w) if case_sensitive else (lambda w: w.lower())
        self.ids = {}
        for i in range(self.n):
            self.ids.setdefault(self.fold(self.vocab[i]), i)

    def get(self, word):
        return self.ids.get(self.fold(word))

    def same_word(self, i, word):
        """Row i spells ``word`` (under the case rule)."""
        return 0 <= i < len(self.vocab) and self.fold(self.vocab[i]) == self.fold(word)


# ---- statistics ---------------------------------------------------------------------------------------------------------
def average_ranks(x):
    """Ranks 1..n, ties share the average of their ranks."""
    x = np.asarray(x, np.float64)
    order = np.argsort(x, kind="mergesort")
    xs = x[order]
    ranks = np.empty(len(x), np.float64)
    i = 0
    while i < len(x):
        j = i
        while j + 1 < len(x) and xs[j + 1] == xs[i]:
            j += 1
        ranks[order[i:j + 1]] = (i + j) / 2.0 + 1.0
        i = j + 1
    return ranks


def pearson(x, y):
    """Pearson r, None when undefined (fewer than two points or a constant side)."""
    x, y = np.asarray(x, np.float64), np.asarray(y, np.float64)
    if len(x) < 2:
        return None
    dx, dy = x - x.mean(), y - y.mean()
    den = np.sqrt(np.dot(dx, dx) * np.dot(dy, dy))
    return float(np.dot(dx, dy) / den) if den > 0 else None


def spearman(x, y):
    """Spearman rho = Pearson r of the average ranks."""
    if len(x) < 2:
        return None
    return pearson(average_ranks(x), average_ranks(y))


# ---- report -------------------------------------------------------------------------------------------------------------
def _tally(total, seen, correct):
    return {"total": total, "seen": seen, "correct": dict(correct),
            "accuracy": {m: (c / seen if seen else None) for m, c in correct.items()}}


def aggregate_analogies(sections, methods=METHODS):
    """``sections``: [(name, total, seen, {method: correct})] -> per-section, semantic, syntactic and overall counts,
    accuracy = correct / seen (None when nothing was seen)."""
    out = {"sections": []}
    groups = {g: [0, 0, {m: 0 for m in methods}] for g in ("semantic", "syntactic", "overall")}
    for name, total, seen, correct in sections:
        out["sections"].append(dict(name=name, **_tally(total, seen, correct)))
        for g in ("syntactic" if is_syntactic(name) else "semantic", "overall"):
            acc = groups[g]
            acc[0] += total
            acc[1] += seen
            for m, c in correct.items():
                acc[2][m] += c
    for g, (total, seen, correct) in groups.items():
        out[g] = _tally(total, seen, correct)
    return out


def evaluate_analogies(engine, sections, words, methods=METHODS):
    """Answers every question whose four words ``words`` knows, over the candidates [0, words.n)."""
    abc, expect, where = [], [], []
    for s, (_, qs) in enumerate(sections):
        for _, q in qs:
            ids = [words.get(w) for w in q]
            if all(i is not None for i in ids):
                abc.append(ids[:3])
                expect.append(q[3])
                where.append(s)
    correct = {m: np.zeros(len(sections), np.int64) for m in methods}
    if abc:
        for m in methods:
            _, idx = engine.analogy(np.array(abc, np.int64), 1, m, restrict=words.n)
            hit = np.array([words.same_word(int(i), e) for i, e in zip(idx[:, 0], expect)], bool)
            np.add.at(correct[m], np.array(where)[hit], 1)
    seen = np.bincount(np.array(where, np.int64), minlength=len(sections)) if where else np.zeros(len(sections), np.int64)
    return aggregate_analogies([(name, len(qs), int(seen[s]), {m: int(correct[m][s]) for m in methods})
                                for s, (name, qs) in enumerate(sections)], methods)


def evaluate_similarity(engine, pairs, words):
    """Spearman rho and Pearson r of the human scores against the cosines of the pairs ``words`` knows."""
    found = [(words.get(a), words.get(b), s) for _, a, b, s in pairs]
    found = [(a, b, s) for a, b, s in found if a is not None and b is not None]
    cos = engine.pair_cosine(np.array([[a, b] for a, b, _ in found], np.int64)) if found else np.zeros(0, np.float32)
    human = [s for _, _, s in found]
    return {"total": len(pairs), "found": len(found), "spearman": spearman(human, cos), "pearson": pearson(human, cos)}


def load_engine(job_dir, checkpoint=None, vectors="row"):
    """Engine with the checkpoint's tables on one GPU; ``vectors="sum"`` puts W + W~ (R + C in fp32, no biases) in the
    row table, what GloVe's own tools evaluate."""
    from . import data_utils, estimator, train_utils
    with open(os.path.join(job_dir, "params.json")) as f:
        params = json.load(f)
    ckpt = checkpoint or train_utils.latest_checkpoint(job_dir)
    if ckpt is None:
        raise FileNotFoundError("no checkpoint in %s" % job_dir)
    eng = estimator.build_engine(params, load_coo=False)
    step = train_utils.load_checkpoint(eng, ckpt)
    if vectors == "sum":
        with np.load(ckpt, allow_pickle=False) as z:
            eng.load_state(z["R"] + z["C"], z["C"], z["rb"], z["cb"], float(z["g"]))
    elif vectors != "row":
        raise ValueError("vectors must be 'row' or 'sum', not %r" % vectors)
    return eng, data_utils.read_vocab(params["vocab_txt"]), ckpt, step


def evaluate(engine, vocab, analogies=(), similarity=(), restrict_vocab=None, case_sensitive=False):
    words = WordIds(vocab, restrict_vocab, case_sensitive)
    report = {"restrict_vocab": words.n, "case_sensitive": bool(case_sensitive), "analogies": [], "similarity": []}
    for path in analogies:
        r = evaluate_analogies(engine, parse_analogies(path), words)
        report["analogies"].append(dict(file=path, **r))
    for path in similarity:
        r = evaluate_similarity(engine, parse_similarity(path), words)
        report["similarity"].append(dict(file=path, **r))
    return report


def _pct(x):
    return "n/a" if x is None else "%.2f%%" % (100.0 * x)


def log_report(report):
    for a in report["analogies"]:
        for s in a["sections"]:
            logger.info("%s [%s]: %s", a["file"], s["name"], ", ".join("%s %d/%d (%s)" % (m, c, s["seen"], _pct(s["accuracy"][m]))
                                                                      for m, c in s["correct"].items()))
        for g in ("semantic", "syntactic", "overall"):
            t = a[g]
            logger.info("%s %s: seen %d of %d questions, %s", a["file"], g, t["seen"], t["total"],
                        ", ".join("%s %s" % (m, _pct(acc)) for m, acc in t["accuracy"].items()))
    for s in report["similarity"]:
        logger.info("%s: %d of %d pairs found, spearman %s, pearson %s", s["file"], s["found"], s["total"],
                    "n/a" if s["spearman"] is None else "%.4f" % s["spearman"],
                    "n/a" if s["pearson"] is None else "%.4f" % s["pearson"])


def main(argv=None):
    ap = ArgumentParser(description="Word-analogy and word-similarity evaluation of a trained job's embeddings.")
    src = ap.add_mutually_exclusive_group(required=True)
    src.add_argument("--job-dir", help="job directory (params.json, vocab.txt, checkpoints)")
    src.add_argument("--vectors-txt", metavar="FILE", help="word vectors in the GloVe text format (optional word2vec header)")
    ap.add_argument("--dim", type=int, default=None, metavar="D",
                    help="with --vectors-txt: the number of values per line (default: from the header or the first line)")
    ap.add_argument("--checkpoint", default=None, help="checkpoint file (default: the latest in the job directory)")
    ap.add_argument("--analogies", nargs="+", action="extend", default=[], metavar="FILE",
                    help="analogy files in questions-words.txt format")
    ap.add_argument("--similarity", nargs="+", action="extend", default=[], metavar="FILE",
                    help="word-similarity files: 'w1 w2 score' per line")
    ap.add_argument("--restrict-vocab", type=int, default=None, metavar="N",
                    help="only the first N words of vocab.txt (the most frequent) are looked up and ranked")
    ap.add_argument("--vectors", choices=("row", "sum"), default=None,
                    help="row (default): the row embeddings (PREDICT and export use them); sum: row + column embeddings")
    ap.add_argument("--case-sensitive", action="store_true", help="match words exactly (default: lower() on both sides)")
    ap.add_argument("--output-json", default=None,
                    help="report path (default: <job-dir>/intrinsic_eval.json; required with --vectors-txt)")
    args = ap.parse_args(argv)
    if args.restrict_vocab is not None and args.restrict_vocab < 1:
        ap.error("--restrict-vocab must be at least 1")
    if args.vectors_txt is not None:
        if args.output_json is None:
            ap.error("--vectors-txt needs --output-json")
        if args.vectors is not None or args.checkpoint is not None:
            ap.error("--vectors and --checkpoint apply to --job-dir only")
        from .vectors import vectors_engine
        eng, vocab = vectors_engine(args.vectors_txt, args.dim)
        report = {"vectors_txt": args.vectors_txt, "rows": eng.V, "dim": eng.d}
    else:
        if args.dim is not None:
            ap.error("--dim applies to --vectors-txt only")
        vectors = args.vectors or "row"
        eng, vocab, ckpt, step = load_engine(args.job_dir, args.checkpoint, vectors)
        report = {"checkpoint": ckpt, "global_step": step, "vectors": vectors}
    report.update(evaluate(eng, vocab, args.analogies, args.similarity, args.restrict_vocab, args.case_sensitive))
    log_report(report)
    out = args.output_json or os.path.join(args.job_dir, "intrinsic_eval.json")
    with open(out, "w") as f:
        json.dump(report, f, indent=2)
    logger.info("report saved: %s.", out)
    return report


if __name__ == "__main__":
    logging.basicConfig(level=logging.INFO, format="%(asctime)s - %(levelname)s - %(name)s - %(message)s")
    logger.info("call: %s.", " ".join(sys.argv))
    main()
