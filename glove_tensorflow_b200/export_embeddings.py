"""``python -m glove_tensorflow_b200.export_embeddings`` -- drop-in for src/models/export_embeddings.py:13-64:
reload params.json from the job dir, read the ROW embedding of every vocab token from the latest checkpoint and write
{token: {"item_id": token, "item_embedding": [d floats]}} (indent 2), skipping '<UNK>'.

``--format glove`` writes the GloVe text format instead (vectors.py; formatted on the GPU), the format Stanford's trainer
and the published vectors use: every vocabulary row in id order, '<UNK>' included (as Stanford writes its '<unk>'), so
that row ids survive the round trip, each value as the shortest decimal that reads back to the same float32.
``--vectors sum`` writes W + W~ (row + column embeddings, fp32), Stanford's default output; ``--word2vec-header`` adds the
first line ``V d``."""
import json
import logging
import os
import sys
from argparse import ArgumentParser

import numpy as np

from .config import EMBEDDINGS_JSON, JOB_DIR
from . import data_utils, train_utils

logger = logging.getLogger(__name__)


def format_predictions(tokens, embeddings):
    out = {}
    for tok, emb in zip(tokens, embeddings):
        if tok != "<UNK>":
            out[tok] = {"item_id": tok, "item_embedding": [float(x) for x in emb]}
    logger.info("embedding dict size: %s.", len(out))
    return out


def main(job_dir=JOB_DIR, embeddings_json=EMBEDDINGS_JSON, format="json", vectors="row", output=None, word2vec_header=False,
         **kwargs):
    with open(os.path.join(job_dir, "params.json")) as f:
        params = json.load(f)
    ckpt = train_utils.latest_checkpoint(job_dir)
    if ckpt is None:
        raise FileNotFoundError("no checkpoint in %s" % job_dir)
    if format == "glove":
        return export_glove(params, ckpt, output or os.path.join(job_dir, "vectors.txt"), vectors, word2vec_header)
    if format != "json":
        raise ValueError("format must be 'json' or 'glove', not %r" % format)
    # the checkpoint holds the flushed (dense-Keras-exact) tables in the reference's layout: the export needs no GPU
    table = np.load(ckpt, allow_pickle=False)["R"]
    vocab = data_utils.read_vocab(params["vocab_txt"])
    embeddings = format_predictions(vocab, table)
    os.makedirs(os.path.dirname(os.path.abspath(embeddings_json)), exist_ok=True)
    with open(embeddings_json, "w") as f:
        json.dump(embeddings, f, indent=2)
    logger.info("json saved: %s.", embeddings_json)
    return embeddings_json


def export_glove(params, ckpt, output, vectors="row", header=False):
    """Every vocabulary row of the checkpoint as a GloVe text file; ``vectors="sum"`` is R + C in fp32, exactly the table
    ``evaluate_embeddings --vectors sum`` evaluates."""
    import torch
    from . import vectors as vec
    with np.load(ckpt, allow_pickle=False) as z:
        if vectors == "sum":
            table = z["R"] + z["C"]
        elif vectors == "row":
            table = z["R"]
        else:
            raise ValueError("vectors must be 'row' or 'sum', not %r" % vectors)
    vocab = data_utils.read_vocab(params["vocab_txt"])
    os.makedirs(os.path.dirname(os.path.abspath(output)), exist_ok=True)
    vec.write_vectors(output, vocab, torch.from_numpy(np.ascontiguousarray(table, np.float32)).to("cuda"), header=header)
    logger.info("vectors saved: %s (%d x %d).", output, table.shape[0], table.shape[1])
    return output


if __name__ == "__main__":
    logging.basicConfig(level=logging.INFO)
    ap = ArgumentParser()
    ap.add_argument("--job-dir", default=JOB_DIR, help="job directory (default: %(default)s)")
    ap.add_argument("--embeddings-json", default=EMBEDDINGS_JSON, help="path to the embeddings json (default: %(default)s)")
    ap.add_argument("--format", choices=("json", "glove"), default="json",
                    help="json: the reference's embeddings json; glove: the GloVe text format (default: %(default)s)")
    ap.add_argument("--vectors", choices=("row", "sum"), default="row",
                    help="--format glove: row embeddings, or row + column embeddings (default: %(default)s)")
    ap.add_argument("--output", default=None, help="--format glove: output path (default: <job-dir>/vectors.txt)")
    ap.add_argument("--word2vec-header", action="store_true", help="--format glove: first line 'V d' (word2vec text format)")
    args = ap.parse_args()
    logger.info("call: %s.", " ".join(sys.argv))
    try:
        main(**args.__dict__)
    except KeyboardInterrupt:
        pass
    except Exception as e:
        logger.exception(e)
        raise e
