"""CPU checks of the Stanford GloVe co-occurrence container: the oracle (oracle/cooc_bin_oracle.py) on hand-made files,
Stanford-vocabulary detection, argument errors of glove_cooc_bin_parse / glove_cooc_bin_format, the trainer flags and
the job-dir vocabulary."""
import ctypes
import json
import os
import struct

import numpy as np
import pytest

from oracle import cooc_bin_oracle as cb

GOLD = os.path.join(os.path.dirname(__file__), "golden", "text8_small")


def test_record_is_16_packed_little_endian_bytes():
    raw = struct.pack("<iid", 3, 7, 2.5)
    assert len(raw) == 16 and cb.RECORD.itemsize == 16
    assert raw == cb.write([2], [6], [2.5])
    rec = np.frombuffer(raw, cb.RECORD)[0]
    assert (rec["word1"], rec["word2"], rec["val"]) == (3, 7, 2.5)


def test_oracle_reads_a_three_record_file():
    raw = struct.pack("<iid", 1, 2, 1.0) + struct.pack("<iid", 2, 1, 1e4) + struct.pack("<iid", 3, 3, 0.5)
    got = cb.read(raw, 3)
    assert got["row"].tolist() == [0, 1, 2] and got["col"].tolist() == [1, 0, 2]
    assert got["row"].dtype == np.int32 and got["glove_value"].dtype == np.float32
    assert got["glove_value"].tolist() == [0.0, np.float32(np.log(1e4)), np.float32(np.log(0.5))]
    assert got["glove_weight"].tolist() == [np.float32(0.01 ** 0.75), 1.0, np.float32(0.005 ** 0.75)]
    assert cb.read(raw, 3, x_max=10.0, alpha=0.5)["glove_weight"][0] == np.float32(0.1 ** 0.5)


def test_oracle_weight_at_the_x_max_boundary():
    below, above = 100.0 * (1 - 2.0 ** -52), 100.0 * (1 + 2.0 ** -52)
    vals = np.array([below, 100.0, above, np.nextafter(100.0, 0), np.nextafter(100.0, 200)])
    got = cb.read(cb.write([0] * 5, [1] * 5, vals), 2)
    assert got["glove_weight"][1:3].tolist() == [1.0, 1.0]
    w = np.power(vals / 100.0, 0.75)                                      # rounded once from float64
    assert got["glove_weight"][0] == np.float32(w[0]) and got["glove_weight"][3] == np.float32(w[3])
    assert got["glove_weight"][0] <= 1.0


@pytest.mark.parametrize("w1,w2,val,what", [(0, 1, 1.0, "word1 id 0"), (5, 1, 1.0, "word1 id 5"), (-3, 1, 1.0, "word1 id -3"),
                                            (1, 0, 1.0, "word2 id 0"), (1, 5, 1.0, "word2 id 5"), (1, -1, 1.0, "word2 id -1"),
                                            (1, 1, 0.0, "val 0.0"), (1, 1, -2.0, "val -2.0"), (1, 1, float("nan"), "val nan"),
                                            (1, 1, float("inf"), "val inf"), (1, 1, -0.0, "val -0.0")])
def test_oracle_refusals_name_the_lowest_record(w1, w2, val, what):
    good = cb.write(np.zeros(10, int), np.ones(10, int), np.full(10, 3.0))
    bad = struct.pack("<iid", w1, w2, val)
    raw = good[:7 * 16] + bad + good[:2 * 16] + bad + good
    with pytest.raises(ValueError, match=r"record 8 \(byte 112\): %s" % what):
        cb.read(raw, 4)


def test_oracle_truncated_file():
    raw = cb.write([0, 1, 2], [1, 2, 0], [1.0, 2.0, 3.0])
    for cut in (1, 8, 15):
        with pytest.raises(ValueError, match=r"record 3 \(byte 32\): truncated"):
            cb.read(raw[:-cut], 3)
    with pytest.raises(ValueError, match=r"record 2 \(byte 16\): word1"):   # a bad whole record comes first
        cb.read(raw[:16] + struct.pack("<iid", 9, 1, 1.0) + raw[32:-3], 3)
    assert len(cb.read(b"", 3)["row"]) == 0


def test_stanford_vocabulary_is_detected(tmp_path):
    from glove_tensorflow_b200 import data_utils
    p = tmp_path / "vocab.txt"
    p.write_text("the 1061396\nof 593677\ncafé 12\n<UNK> 7\n", encoding="utf8")
    tokens, counts = data_utils.read_stanford_vocab(str(p))
    assert tokens == ["the", "of", "café", "<UNK>"] and counts.tolist() == [1061396, 593677, 12, 7]
    o_tokens, o_counts = cb.read_vocab(p.read_text(encoding="utf8"))
    assert o_tokens == tokens and o_counts.tolist() == counts.tolist()
    tokens, counts = data_utils.read_stanford_vocab(os.path.join(GOLD, "vocab.txt"))
    assert counts is None and tokens == data_utils.read_vocab(os.path.join(GOLD, "vocab.txt"))
    for bad, line in (("the 10\nof\nand 3\n", 2), ("the 10\nof 3\na b 4\n", 3), ("the 10\nof -3\n", 2),
                      ("the 10\nof 3 \n", 2), ("the 10\n\nof 3\n", 2)):
        p.write_text(bad)
        with pytest.raises(ValueError, match="line %d is not 'word count'" % line):
            data_utils.read_stanford_vocab(str(p))
        with pytest.raises(ValueError, match="line %d" % line):
            cb.read_vocab(bad)
    p.write_text("the 10 x\nof 3\n")                                        # first line is not 'word count': one token a line
    assert data_utils.read_stanford_vocab(str(p)) == (["the 10 x", "of 3"], None)


def test_cooc_bin_entries_refuse_bad_arguments_without_a_gpu():
    from glove_tensorflow_b200 import _lib
    lib, E = _lib.lib, _lib.EINVAL
    f = ctypes.c_void_p(1 << 20)
    cols = [f] * 4
    assert lib.glove_cooc_bin_parse(None, 4, 0, 10, 100.0, 0.75, *cols, f, None) == E
    assert lib.glove_cooc_bin_parse(f, 4, 0, 10, 100.0, 0.75, None, f, f, f, f, None) == E
    assert lib.glove_cooc_bin_parse(f, 4, 0, 10, 100.0, 0.75, *cols, None, None) == E
    assert lib.glove_cooc_bin_parse(ctypes.c_void_p((1 << 20) + 8), 4, 0, 10, 100.0, 0.75, *cols, f, None) == E
    assert b"16-byte aligned" in lib.glove_last_error()
    assert lib.glove_cooc_bin_parse(f, 0, 0, 10, 100.0, 0.75, *cols, f, None) == E
    assert lib.glove_cooc_bin_parse(f, 4, -1, 10, 100.0, 0.75, *cols, f, None) == E
    assert lib.glove_cooc_bin_parse(f, 4, 1 << 62, 10, 100.0, 0.75, *cols, f, None) == E
    assert lib.glove_cooc_bin_parse(f, 4, 0, 0, 100.0, 0.75, *cols, f, None) == E
    assert lib.glove_cooc_bin_parse(f, 4, 0, 1 << 31, 100.0, 0.75, *cols, f, None) == E
    for x_max, alpha in ((0.0, 0.75), (-1.0, 0.75), (float("inf"), 0.75), (float("nan"), 0.75), (100.0, float("nan"))):
        assert lib.glove_cooc_bin_parse(f, 4, 0, 10, x_max, alpha, *cols, f, None) == E
    assert lib.glove_cooc_bin_format(None, f, f, 4, f, None) == E
    assert lib.glove_cooc_bin_format(f, f, f, 4, None, None) == E
    assert lib.glove_cooc_bin_format(f, f, f, 0, f, None) == E
    assert lib.glove_cooc_bin_format(f, f, f, 4, ctypes.c_void_p((1 << 20) + 4), None) == E


def test_trainer_flags_and_defaults():
    from glove_tensorflow_b200 import config_utils
    d = vars(config_utils.build_parser().parse_args([]))
    assert (d["train_cooc"], d["x_max"], d["alpha"]) == (None, 100.0, 0.75)
    a = vars(config_utils.build_parser().parse_args(["--train-cooc", "c.bin", "--x-max", "10", "--alpha", "0.5"]))
    assert (a["train_cooc"], a["x_max"], a["alpha"]) == ("c.bin", 10.0, 0.5)


def test_job_dir_vocabulary_is_converted_and_flags_are_saved(tmp_path):
    from glove_tensorflow_b200 import config_utils, data_utils
    sv = tmp_path / "vocab.stanford.txt"
    sv.write_text("the 50\nof 20\ncafé 3\n", encoding="utf8")
    job = tmp_path / "job"
    params = config_utils.parse_args(["--train-cooc", str(tmp_path / "c.bin"), "--vocab-txt", str(sv), "--job-dir", str(job),
                                      "--disable-datetime-path", "--x-max", "10"])
    assert params["vocab_txt"] == str(job / "vocab.stanford.txt")
    assert (job / "vocab.stanford.txt").read_text(encoding="utf8") == "the\nof\ncafé"
    assert data_utils.read_vocab(params["vocab_txt"]) == ["the", "of", "café"] and data_utils.file_lines(params["vocab_txt"]) == 3
    saved = json.load(open(job / "params.json"))
    assert (saved["train_cooc"], saved["x_max"], saved["alpha"]) == (str(tmp_path / "c.bin"), 10.0, 0.75)
    again = config_utils.parse_args(["--vocab-txt", params["vocab_txt"], "--job-dir", str(job), "--disable-datetime-path"])
    assert (job / "vocab.stanford.txt").read_text(encoding="utf8") == "the\nof\ncafé" and again["train_cooc"] is None


def test_logistic_trainer_refuses_train_cooc(tmp_path):
    from glove_tensorflow_b200 import logistic_matrix_factorisation
    sv = tmp_path / "vocab.txt"
    sv.write_text("the 50\nof 20\n")
    with pytest.raises(ValueError, match="--train-cooc trains the glove head only"):
        logistic_matrix_factorisation.main(["--train-cooc", str(tmp_path / "c.bin"), "--vocab-txt", str(sv), "--job-dir",
                                            str(tmp_path / "job"), "--disable-datetime-path"])


def test_preprocess_refuses_an_unknown_format(tmp_path):
    from glove_tensorflow_b200 import corpus
    with pytest.raises(ValueError, match="format must be one of csv, stanford, both"):
        corpus.preprocess(os.path.join(GOLD, "corpus.txt"), str(tmp_path / "out"), format="bin")
