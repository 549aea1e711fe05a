"""``python -m glove_tensorflow_b200.estimator`` -- drop-in for ``python -m src.models.estimator`` (ref Makefile:93-98,
src/models/estimator.py:79-95): same flags, same inputs (interaction.csv + vocab.txt), same job-dir artefacts
(params.json, vocab.txt copy, checkpoints), the GloVe weighted-least-squares head (RegressionHead with weight column).
``--train-cooc`` trains from a Stanford GloVe cooccurrence.bin instead (data_utils.load_cooc_bin)."""
import logging

from . import config_utils, data_utils, train_utils

HEAD = "glove"


def build_engine(params, head=HEAD, value_names=None, load_coo=True):
    """``load_coo=False``: tables only (PREDICT needs the checkpoint and vocab.txt, not interaction.csv).  With
    ``params["train_cooc"]`` the COO comes from that Stanford GloVe co-occurrence file (``--train-csv`` is ignored)."""
    from .engine import GloveEngine
    cooc = params.get("train_cooc")
    if cooc and head != "glove":
        raise ValueError("--train-cooc trains the glove head only: a Stanford co-occurrence file has no neg_weight column "
                         "for the %s head (use --train-csv)" % head)
    value_names = value_names or (params["target_name"], params["weight_name"])
    vocab_size = data_utils.file_lines(params["vocab_txt"])
    coo = None
    if load_coo and cooc:
        coo = data_utils.load_cooc_bin(cooc, vocab_size, params.get("x_max", 100.0), params.get("alpha", 0.75),
                                       device=params.get("device", "cuda:0"))
        value_names = ("glove_value", "glove_weight")
    elif load_coo:
        coo = data_utils.load_interaction_csv(params["train_csv"], params["vocab_txt"], params["row_name"],
                                              params["col_name"], value_names, device=params.get("device", "cuda:0"))
    reg_scale = params.get("reg_scale")
    if reg_scale is None:
        reg_scale = 2.0  # estimator.py / logistic_matrix_factorisation.py under TF 2.11 (SURVEY A4)
    eng = GloveEngine(vocab_size, params["embedding_size"], optimizer=params["optimizer"],
                      learning_rate=params["learning_rate"], l2_reg=params["l2_reg"], reg_scale=reg_scale,
                      neg_factor=params["neg_factor"], head=head, adam_mode=params.get("adam_mode", "replay"),
                      batch_size=params["batch_size"], plan_steps=params.get("plan_steps", 16),
                      max_steps=params["train_steps"] + 1, device=params.get("device", "cuda:0"))
    eng.init_uniform(params.get("seed", 0))
    if coo is not None:
        eng.set_coo(coo["row"], coo["col"], coo[value_names[0]], coo[value_names[1]], shuffle_key=params.get("seed", 0))
    return eng


def train(params, head=HEAD, value_names=None):
    eng = build_engine(params, head, value_names)
    ckpt = train_utils.latest_checkpoint(params["job_dir"])
    if ckpt:
        train_utils.load_checkpoint(eng, ckpt)
    history = train_utils.train_and_evaluate(eng, params["train_steps"], params["job_dir"],
                                             eval_fn=lambda e: e.eval_metrics(params["batch_size"]))
    return eng, history


def estimator_predict(params, input_ids=None):
    """ref estimator_predict (src/models/estimator.py:59-76): PREDICT over every vocab line from the latest checkpoint."""
    import numpy as np
    from .model_utils import get_predictions
    eng = build_engine(params, load_coo=False)
    ckpt = train_utils.latest_checkpoint(params["job_dir"])
    if ckpt is None:
        raise FileNotFoundError("no checkpoint in %s" % params["job_dir"])
    train_utils.load_checkpoint(eng, ckpt)
    vocab = data_utils.read_vocab(params["vocab_txt"])
    ids = np.arange(len(vocab), dtype=np.int32) if input_ids is None else input_ids
    return get_predictions(eng, ids, vocab, params["top_k"])


def main(argv=None):
    logging.basicConfig(level=logging.INFO, format="%(asctime)s - %(levelname)s - %(name)s - %(message)s")
    params = config_utils.parse_args(argv)
    train(params)


if __name__ == "__main__":
    try:
        main()
    except KeyboardInterrupt:
        pass
