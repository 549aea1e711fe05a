"""PREDICT-side helpers mirroring the reference's src/models/model_utils.py:81-136."""
import numpy as np


def get_id_string_table(vocab):
    """id -> string with default '<UNK>' (ref model_utils.py:130-136)."""
    def lookup(ids):
        return [vocab[i] if 0 <= i < len(vocab) else "<UNK>" for i in np.asarray(ids).reshape(-1)]
    return lookup


def get_predictions(engine, input_ids, vocab, top_k=20):
    """ref get_predictions (model_utils.py:81-110): cosine similarity of the ROW embedding of each input id against the
    whole row table, tf.math.top_k(sorted) -- values descending, ties -> lower id.  Returns the reference's prediction
    keys: input_string, input_embedding, top_k_similarity, top_k_string."""
    input_ids = np.asarray(input_ids, dtype=np.int32).reshape(-1)
    sim, idx = engine.topk(input_ids, top_k)
    table = engine.row_embeddings()
    lookup = get_id_string_table(vocab)
    return {
        "input_string": lookup(input_ids),
        "input_embedding": table[input_ids.astype(np.int64)].cpu().numpy(),
        "top_k_similarity": sim,
        "top_k_string": [lookup(r) for r in idx],
    }


def get_analogies(engine, triples, vocab, top_k=1, method="add"):
    """Word analogies a : b :: c : ? for string triples (a, b, c): the ``top_k`` best rows outside {a, b, c} by 3CosAdd
    (``method="add"``) or 3CosMul (``"mul"``).  Words are looked up exactly in ``vocab`` (the first line holding a token
    wins); an unknown word raises KeyError.  Returns input_strings, top_k_score, top_k_string."""
    first = {}
    for i, tok in enumerate(vocab):
        first.setdefault(tok, i)
    triples = [tuple(t) for t in triples]
    missing = sorted({w for t in triples for w in t if w not in first})
    if missing:
        raise KeyError("get_analogies: not in the vocabulary: %s" % ", ".join(missing[:10]))
    abc = np.array([[first[w] for w in t] for t in triples], np.int64).reshape(-1, 3)
    score, idx = engine.analogy(abc, top_k, method)
    lookup = get_id_string_table(vocab)
    return {
        "input_strings": [list(t) for t in triples],
        "top_k_score": score,
        "top_k_string": [lookup(r) for r in idx],
    }
