"""Stanford GloVe's trainer on the GPU: glove.c's per-record AdaGrad over a co-occurrence file in file order, exactly
as its sequential run (-threads 1) computes it, run in parallel along the records' dependencies (csrc/glove_sgd.cu,
DESIGN.md section 3, "Stanford GloVe's trainer").

    python -m glove_tensorflow_b200.stanford_glove --input-file cooccurrence.shuf.bin --vocab-file vocab.txt \\
        [--save-file vectors] [--vector-size 50] [--iter 25] [--eta 0.05] [--alpha 0.75] [--x-max 100] \\
        [--grad-clip 100] [--seed 1] [--model 2] [--binary 0] [--write-header] [--no-unk-vector] \\
        [--save-gradsq] [--gradsq-file gradsq] [--init-param-file F.bin] [--init-gradsq-file G.bin]

Flags mirror glove.c's.  ``--model``: 0 = word and context rows with their biases (2d + 2 values a line), 1 = word
vectors, 2 = word + context vectors.  ``--binary``: 0 = ``<save-file>.txt``, 1 = ``<save-file>.bin`` (W in glove.c's
layout, 2V rows of d + 1 little-endian doubles), 2 = both.  ``--save-gradsq`` writes ``<gradsq-file>.bin`` in the same
layout; ``--init-param-file`` / ``--init-gradsq-file`` read that layout, so a run resumes bit for bit.  The text file
holds float32 values in the shortest decimals that read back exactly (vectors.write_vectors), not glove.c's %lf, and
ends with glove.c's ``<unk>`` line unless ``--no-unk-vector`` is given.  Initialisation is seeded (``--seed``) where
glove.c seeds rand() from the clock."""
import argparse
import os
import sys

import numpy as np

from . import _lib
from .data_utils import COOC_RECORD, _check_vocab_size, read_stanford_vocab, stream_cooc_bin

DEFAULTS = {"save_file": "vectors", "vector_size": 50, "iter": 25, "eta": 0.05, "alpha": 0.75, "x_max": 100.0,
            "grad_clip": 100.0, "seed": 1, "model": 2, "binary": 0, "write_header": False, "unk_vector": True,
            "save_gradsq": False, "gradsq_file": "gradsq", "init_param_file": None, "init_gradsq_file": None}
MAX_VECTOR_SIZE = 512     # csrc/glove_sgd.cu: 32 lanes x 16 elements per lane
MAX_TEXT_VALUES = 510     # vectors.write_vectors
UNK = "<unk>"


def text_values(vector_size, model):
    return 2 * vector_size + 2 if model == 0 else vector_size


class StanfordGlove:
    """The trainer's device state for one co-occurrence file: records (words int32 [n, 2], lf float64 [n, 2]), links
    (prev int32 [n, 2]), W and gradsq (float64 [2V, d + 1], glove.c's layout) and the per-record done flags."""

    def __init__(self, input_file, vocab_size, vector_size=50, alpha=0.75, x_max=100.0, seed=1, device="cuda:0",
                 chunk_bytes=64 << 20):
        import torch
        self.V, self.d = _check_vocab_size(vocab_size), int(vector_size)
        if not 1 <= self.d <= MAX_VECTOR_SIZE:
            raise ValueError("vector_size must be 1 .. %d, got %d" % (MAX_VECTOR_SIZE, self.d))
        self.dev = torch.device(device)
        size = os.path.getsize(input_file)
        n = size // COOC_RECORD
        if n == 0:
            raise ValueError("%s holds no co-occurrence records" % input_file)
        if n >= 1 << 31:
            raise ValueError("%s holds %d records; the trainer takes at most 2^31 - 1" % (input_file, n))
        self.n = n
        lib = _lib.lib
        links_ws, epoch_ws = lib.glove_sgd_links_workspace_bytes(n), lib.glove_sgd_epoch_workspace_bytes(n)
        tables = 2 * 2 * self.V * (self.d + 1) * 8
        need = tables + n * (24 + 8 + 4) + max(links_ws, epoch_ws) + (chunk_bytes + 4096)
        with torch.cuda.device(self.dev):
            free, _ = torch.cuda.mem_get_info()
            if need > free:
                raise MemoryError("training %s needs %.3g GB of device memory (W and gradsq %.3g GB for V = %d, d = %d; "
                                  "%d records at 36 bytes; %.3g GB of workspace); %.3g GB are free"
                                  % (input_file, need / 1e9, tables / 1e9, self.V, self.d, n,
                                     max(links_ws, epoch_ws) / 1e9, free / 1e9))
            st = torch.cuda.current_stream().cuda_stream
            self.words = torch.empty((n, 2), dtype=torch.int32, device=self.dev)
            self.lf = torch.empty((n, 2), dtype=torch.float64, device=self.dev)

            def parse(raw, m, first, err, stream):
                _lib.check(lib.glove_sgd_parse(raw, m, first, self.V, float(x_max), float(alpha),
                                               self.words[first:].data_ptr(), self.lf[first:].data_ptr(), err, stream),
                           "glove_sgd_parse")

            stream_cooc_bin(input_file, self.V, parse, self.dev, chunk_bytes)
            self.prev = torch.empty((n, 2), dtype=torch.int32, device=self.dev)
            ws = torch.empty(links_ws, dtype=torch.uint8, device=self.dev)
            _lib.check(lib.glove_sgd_links(self.words.data_ptr(), n, self.V, self.prev.data_ptr(), ws.data_ptr(), links_ws,
                                           st), "glove_sgd_links")
            del ws
            self.ws = torch.empty(epoch_ws, dtype=torch.uint8, device=self.dev)
            self.done = torch.zeros(n, dtype=torch.int32, device=self.dev)
            self.cost = torch.zeros(1, dtype=torch.float64, device=self.dev)
            self.W = torch.empty((2 * self.V, self.d + 1), dtype=torch.float64, device=self.dev)
            self.gradsq = torch.ones_like(self.W)
            _lib.check(lib.glove_sgd_init(self.W.data_ptr(), self.V, self.d, int(seed) & (2 ** 64 - 1), st), "glove_sgd_init")
        self.epochs = 0

    def load(self, which, path):
        """Replaces W ('W') or gradsq ('gradsq') by a .bin file of glove.c's layout."""
        t = self.W if which == "W" else self.gradsq
        want = t.numel() * 8
        if os.path.getsize(path) != want:
            raise ValueError("%s: %d bytes, but 2V(d + 1) doubles for V = %d, d = %d are %d bytes"
                             % (path, os.path.getsize(path), self.V, self.d, want))
        import torch
        t.copy_(torch.from_numpy(np.fromfile(path, "<f8").reshape(t.shape)))

    def save(self, which, path):
        t = self.W if which == "W" else self.gradsq
        t.cpu().numpy().astype("<f8", copy=False).tofile(path)
        return path

    def epoch(self, eta=0.05, grad_clip=100.0, grid=0):
        """One pass over the records in file order; returns glove.c's cost (summed record costs / n)."""
        import torch
        self.epochs += 1
        with torch.cuda.device(self.dev):
            st = torch.cuda.current_stream().cuda_stream
            _lib.check(_lib.lib.glove_sgd_epoch(self.W.data_ptr(), self.gradsq.data_ptr(), self.V, self.d,
                                                self.words.data_ptr(), self.lf.data_ptr(), self.prev.data_ptr(), self.n,
                                                float(eta), float(grad_clip), self.epochs, self.done.data_ptr(),
                                                int(grid), self.ws.data_ptr(), self.ws.numel(), self.cost.data_ptr(), st),
                       "glove_sgd_epoch")
            return float(self.cost.item())

    def rows(self, model=2, unk=True):
        """float32 [V + unk, values] device rows of the vectors file (model 0: 2d + 2 values, 1 and 2: d)."""
        import torch
        with torch.cuda.device(self.dev):
            out = torch.empty((self.V + int(unk), text_values(self.d, model)), dtype=torch.float32, device=self.dev)
            _lib.check(_lib.lib.glove_sgd_rows(self.W.data_ptr(), self.V, self.d, int(model), int(unk), out.data_ptr(),
                                               torch.cuda.current_stream().cuda_stream), "glove_sgd_rows")
            return out


def train(input_file, vocab_file, save_file="vectors", vector_size=50, iter=25, eta=0.05, alpha=0.75, x_max=100.0,
          grad_clip=100.0, seed=1, model=2, binary=0, write_header=False, unk_vector=True, save_gradsq=False,
          gradsq_file="gradsq", init_param_file=None, init_gradsq_file=None, device="cuda:0", grid=0, log=print):
    """Trains ``iter`` epochs and writes the files glove.c writes; returns the per-epoch costs."""
    from . import vectors
    if model not in (0, 1, 2) or binary not in (0, 1, 2):
        raise ValueError("model must be 0, 1 or 2 and binary 0, 1 or 2")
    if iter < 0:
        raise ValueError("iter must be >= 0")
    if not (eta == eta and grad_clip == grad_clip and x_max > 0):
        raise ValueError("eta and grad_clip must not be NaN and x_max must be > 0")
    if binary != 1 and not 2 <= text_values(vector_size, model) <= MAX_TEXT_VALUES:
        raise ValueError("a text file of model %d holds %d values a line; the text writer takes 2 .. %d"
                         % (model, text_values(vector_size, model), MAX_TEXT_VALUES))
    words, _ = read_stanford_vocab(vocab_file)
    if unk_vector and UNK in words:
        raise ValueError("%s: the vocabulary holds %s, which the <unk> vector line would repeat (use --no-unk-vector)"
                         % (vocab_file, UNK))
    sg = StanfordGlove(input_file, len(words), vector_size, alpha, x_max, seed, device)
    if init_param_file:
        sg.load("W", init_param_file)
    if init_gradsq_file:
        sg.load("gradsq", init_gradsq_file)
    costs = []
    for it in range(iter):
        costs.append(sg.epoch(eta, grad_clip, grid))
        log("iter: %03d, cost: %.6f" % (it + 1, costs[-1]))
    if binary > 0:
        sg.save("W", save_file + ".bin")
    if binary != 1:
        vectors.write_vectors(save_file + ".txt", list(words) + ([UNK] if unk_vector else []), sg.rows(model, unk_vector),
                              header=write_header)
    if save_gradsq:
        sg.save("gradsq", gradsq_file + ".bin")
    return costs


def parser():
    ap = argparse.ArgumentParser(prog="python -m glove_tensorflow_b200.stanford_glove", description=__doc__.split("\n")[0])
    ap.add_argument("--input-file", required=True, help="cooccurrence.shuf.bin (16-byte records, read in file order)")
    ap.add_argument("--vocab-file", required=True, help="vocab.txt: 'word count' lines, or one token a line")
    ap.add_argument("--save-file", default=DEFAULTS["save_file"], help="writes <save-file>.txt and/or <save-file>.bin")
    ap.add_argument("--vector-size", type=int, default=DEFAULTS["vector_size"])
    ap.add_argument("--iter", type=int, default=DEFAULTS["iter"])
    ap.add_argument("--eta", type=float, default=DEFAULTS["eta"])
    ap.add_argument("--alpha", type=float, default=DEFAULTS["alpha"])
    ap.add_argument("--x-max", type=float, default=DEFAULTS["x_max"])
    ap.add_argument("--grad-clip", type=float, default=DEFAULTS["grad_clip"])
    ap.add_argument("--seed", type=int, default=DEFAULTS["seed"])
    ap.add_argument("--model", type=int, choices=(0, 1, 2), default=DEFAULTS["model"])
    ap.add_argument("--binary", type=int, choices=(0, 1, 2), default=DEFAULTS["binary"])
    ap.add_argument("--write-header", action="store_true", help="first line 'rows values' (word2vec)")
    ap.add_argument("--no-unk-vector", dest="unk_vector", action="store_false", help="omit the <unk> line")
    ap.add_argument("--save-gradsq", action="store_true", help="also write <gradsq-file>.bin")
    ap.add_argument("--gradsq-file", default=DEFAULTS["gradsq_file"])
    ap.add_argument("--init-param-file", default=None, help="W to start from (.bin layout)")
    ap.add_argument("--init-gradsq-file", default=None, help="gradsq to start from (.bin layout)")
    return ap


def main(argv=None):
    ap = parser()
    args = ap.parse_args(argv)
    if not 1 <= args.vector_size <= MAX_VECTOR_SIZE:
        ap.error("--vector-size must be 1 .. %d" % MAX_VECTOR_SIZE)
    if args.iter < 0:
        ap.error("--iter must be >= 0")
    if not (args.x_max > 0 and args.eta == args.eta and args.grad_clip == args.grad_clip and args.alpha == args.alpha):
        ap.error("--x-max must be > 0, and --eta, --grad-clip and --alpha must be numbers")
    if args.binary != 1 and not 2 <= text_values(args.vector_size, args.model) <= MAX_TEXT_VALUES:
        ap.error("--model %d --vector-size %d gives %d values a text line; the text writer takes 2 .. %d"
                 % (args.model, args.vector_size, text_values(args.vector_size, args.model), MAX_TEXT_VALUES))
    return train(**vars(args))


if __name__ == "__main__":
    main()
    sys.exit(0)
