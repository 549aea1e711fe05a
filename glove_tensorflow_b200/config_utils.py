"""CLI + job-dir bookkeeping of the trainer: same 19 flags, names, types and defaults as the reference's
src/models/config_utils.py:76-180, same derived ``input_fn_args`` / ``dataset_args`` / ``serving_input_fn_args`` (:20-45),
same ``params.json`` (indent 2, :48-52) and vocab copy into the job dir (:55-73).  Flags that only exist here
(--adam-mode, --reg-scale, --plan-steps, --seed, --device, --train-cooc, --x-max, --alpha) default to the reference's
behaviour.  A --vocab-txt of Stanford GloVe's ``word count`` lines is copied into the job dir as one token per line."""
import json
import logging
import os
import shutil
import sys
from argparse import ArgumentParser
from datetime import datetime

from .config import (
    BATCH_SIZE, COL_NAME, EMBEDDING_SIZE, JOB_DIR, L2_REG, LEARNING_RATE, NEG_FACTOR, NEG_NAME, OPTIMIZER, POS_NAME,
    ROW_NAME, STEPS_PER_EPOCH, TARGET_NAME, TOP_K, TRAIN_CSV, TRAIN_STEPS, VOCAB_TXT, WEIGHT_NAME,
)
from .data_utils import read_stanford_vocab

logger = logging.getLogger(__name__)


def get_function_args(params):
    row_name, col_name = params["row_name"], params["col_name"]
    target_name, weight_name = params["target_name"], params["weight_name"]
    input_fn_args = {
        "file_pattern": params["train_csv"],
        "batch_size": params["batch_size"],
        "select_columns": [row_name, col_name, weight_name, target_name],
        "target_names": [target_name],
    }
    dataset_args = {
        "row_col_names": [row_name, col_name],
        "vocab_txt": params["vocab_txt"],
        **input_fn_args,
        "weight_names": [weight_name],
    }
    serving_input_fn_args = {"string_features": [row_name, col_name]}
    return {"input_fn_args": input_fn_args, "dataset_args": dataset_args,
            "serving_input_fn_args": serving_input_fn_args}


def save_params(params, params_json="params.json"):
    path = os.path.join(params["job_dir"], params_json)
    with open(path, "w") as f:
        json.dump(params, f, indent=2)
    return path


def init_params(params):
    if not params["disable_datetime_path"]:
        params["job_dir"] = "{job_dir}-{datetime:%Y%m%d-%H%M%S}".format(job_dir=params["job_dir"], datetime=datetime.now())
    os.makedirs(params["job_dir"], exist_ok=True)
    output_vocab_txt = os.path.join(params["job_dir"], os.path.basename(params["vocab_txt"]))
    tokens, counts = read_stanford_vocab(params["vocab_txt"])
    if counts is not None:
        # Stanford's `word count` lines: the job-dir copy is one token per line, the vocab.txt every other tool reads
        with open(output_vocab_txt + ".tmp", "w", encoding="utf8") as f:
            f.write("\n".join(tokens))
        os.replace(output_vocab_txt + ".tmp", output_vocab_txt)
    elif os.path.abspath(params["vocab_txt"]) != os.path.abspath(output_vocab_txt):
        shutil.copyfile(params["vocab_txt"], output_vocab_txt)
    params["vocab_txt"] = output_vocab_txt
    params.update(get_function_args(params))
    save_params(params)
    return params


def build_parser():
    p = ArgumentParser()
    p.add_argument("--train-csv", default=TRAIN_CSV, help="path to the training csv data (default: %(default)s)")
    p.add_argument("--vocab-txt", default=VOCAB_TXT, help="path to the vocab txt (default: %(default)s)")
    p.add_argument("--row-name", default=ROW_NAME, help="row id name (default: %(default)s)")
    p.add_argument("--col-name", default=COL_NAME, help="column id name (default: %(default)s)")
    p.add_argument("--target-name", default=TARGET_NAME, help="target name (default: %(default)s)")
    p.add_argument("--weight-name", default=WEIGHT_NAME, help="weight name (default: %(default)s)")
    p.add_argument("--pos-name", default=POS_NAME, help="positive name (default: %(default)s)")
    p.add_argument("--neg-name", default=NEG_NAME, help="negative name (default: %(default)s)")
    p.add_argument("--job-dir", default=JOB_DIR, help="job directory (default: %(default)s)")
    p.add_argument("--disable-datetime-path", action="store_true",
                   help="flag whether to disable appending datetime in job_dir path (default: %(default)s)")
    p.add_argument("--embedding-size", type=int, default=EMBEDDING_SIZE, help="embedding size (default: %(default)s)")
    p.add_argument("--l2-reg", type=float, default=L2_REG, help="scale of l2 regularisation (default: %(default)s)")
    p.add_argument("--neg-factor", type=float, default=NEG_FACTOR, help="negative loss factor (default: %(default)s)")
    p.add_argument("--optimizer", default=OPTIMIZER, help="name of optimzer (default: %(default)s)")
    p.add_argument("--learning-rate", type=float, default=LEARNING_RATE, help="learning rate (default: %(default)s)")
    p.add_argument("--batch-size", type=int, default=BATCH_SIZE, help="batch size (default: %(default)s)")
    p.add_argument("--train-steps", type=int, default=TRAIN_STEPS, help="number of training steps (default: %(default)s)")
    p.add_argument("--steps-per-epoch", type=int, default=STEPS_PER_EPOCH,
                   help="number of steps per checkpoint (default: %(default)s)")
    p.add_argument("--top-k", type=int, default=TOP_K, help="number of similar items (default: %(default)s)")
    # --- B200-only knobs (defaults = reference semantics) ---
    p.add_argument("--adam-mode", default="replay", choices=["replay", "replay_exact", "dense", "lazy"],
                   help="replay / replay_exact / dense = legacy Keras Adam (reference): idle steps applied in closed form / "
                        "replayed step by step / swept after every step; lazy = LazyAdam (default: %(default)s)")
    p.add_argument("--reg-scale", type=float, default=None,
                   help="activity-L2 multiplicity; default 2 for the estimator trainers under TF 2.11 (SURVEY A4)")
    p.add_argument("--plan-steps", type=int, default=16, help="batches planned per prepare call (default: %(default)s)")
    p.add_argument("--seed", type=int, default=0, help="seed of the table initialiser and the epoch shuffle")
    p.add_argument("--device", default="cuda:0")
    # --- Stanford GloVe co-occurrence input (glove head only) ---
    p.add_argument("--train-cooc", default=None,
                   help="Stanford GloVe cooccurrence.bin / cooccurrence.shuf.bin to train from instead of --train-csv; ids "
                        "are 1-based lines of --vocab-txt (default: %(default)s)")
    p.add_argument("--x-max", type=float, default=100.0,
                   help="with --train-cooc: weight cutoff of glove.c, weight = min(1, (X / x_max)^alpha) (default: %(default)s)")
    p.add_argument("--alpha", type=float, default=0.75, help="with --train-cooc: weight exponent (default: %(default)s)")
    return p


def parse_args(argv=None):
    args = build_parser().parse_args(argv)
    logger.info("call: %s.", " ".join(sys.argv))
    logger.info("ArgumentParser: %s.", args.__dict__)
    return init_params(dict(args.__dict__))
