"""``python -m glove_tensorflow_b200.text8`` -- drop-in for ``python -m src.data.text8`` (ref src/data/text8.py:154-196):
corpus text -> vocab.csv, vocab.txt, interaction.csv with the reference's schema (SURVEY §8 f.4).

The vocabulary (a few thousand strings) is counted on the host; the pair counting -- the position cross-join, groupby
and symmetrisation that take minutes and tens of GB in pandas -- runs on the GPU (csrc/glove_cooc.cu): token ids are
uploaded once, pairs are emitted / radix-sorted / reduced per chunk of positions, chunks are merged, and the final
kernel writes the reference's numeric columns.  ``cooccurrence_table`` also hands the result over as device tensors, so a
trainer can skip the csv altogether."""
import ctypes
import logging
import os
import sys
from argparse import ArgumentParser
from collections import Counter

import numpy as np

logger = logging.getLogger(__name__)

from .config import CONTEXT_SIZE, COVERAGE, DATA_DIR, TEXT8_URL, VOCAB_SIZE   # ref src/data/text8.py:12 (VOCAB_SIZE = None)


def download_data(url=TEXT8_URL, dest_dir=DATA_DIR):
    """Fetch and unzip the corpus unless ``<dest_dir>/text8`` is already there (ref text8.py:18-35)."""
    import shutil
    import urllib.request
    from zipfile import ZipFile
    os.makedirs(dest_dir, exist_ok=True)
    if os.path.exists(os.path.join(dest_dir, "text8")):
        return
    dest = os.path.join(dest_dir, os.path.basename(url))
    if not os.path.exists(dest):
        logger.info("downloading file: %s.", url)
        with urllib.request.urlopen(url) as r, open(dest, "wb") as f:
            shutil.copyfileobj(r, f)
    with ZipFile(dest) as zf:
        zf.extractall(dest_dir)


def load_data(src_dir=DATA_DIR):
    with open(os.path.join(src_dir, "text8")) as f:
        return f.read()


def create_vocabulary(text_tokens, vocab_size=VOCAB_SIZE, coverage=COVERAGE):
    """Frame (token, count, proportion): '<UNK>' plus at most ``vocab_size`` tokens whose count reaches the cut-off at
    which the cumulative token share passes ``coverage``; ordered by count (ref text8.py:61-81)."""
    freq = Counter(text_tokens)                    # insertion order = order of first occurrence
    return _frame_from_counts(list(freq.keys()), np.fromiter(freq.values(), np.int64, len(freq)), vocab_size, coverage)


def token_ids(text_tokens, vocab_tokens):
    """token -> row of the vocabulary frame, unknown -> 0 (ref text8.py:85-86)."""
    lut = {t: i for i, t in enumerate(vocab_tokens)}
    get = lut.get
    return np.fromiter((get(t, 0) for t in text_tokens), np.int32, len(text_tokens))


def _frame_from_counts(tokens, counts, vocab_size, coverage):
    """The vocabulary frame from (token, count) pairs listed in order of first occurrence -- the part of
    create_vocabulary that comes after Counter (ref text8.py:64-81)."""
    import pandas as pd
    counts = np.asarray(counts, np.int64)
    by_count = np.sort(counts)[::-1]
    total = int(by_count.sum())
    cutoff = by_count[np.searchsorted(np.cumsum(by_count) / total, coverage)]
    logger.info("count cufoff: %s; token coverage: %s.", cutoff, coverage)
    top = np.argsort(-counts, kind="stable")[:vocab_size]        # most_common: by count, ties in order of first occurrence
    top = top[counts[top] >= cutoff]
    kept = counts[top].tolist()
    frame = pd.DataFrame({"token": ["<UNK>"] + [tokens[i] for i in top], "count": [total - int(np.sum(kept))] + kept})
    frame["proportion"] = frame["count"] / total
    return frame.sort_values("count", ascending=False).reset_index(drop=True)


class DeviceCorpus:
    """Corpus text resident on the GPU with its token index (glove_tokens_scan): what ``text8.split()`` is to the
    reference (ref text8.py:47), without materialising Python strings."""

    def __init__(self, text, device="cuda:0"):
        import torch
        from . import _lib
        self.lib, self.check = _lib.lib, _lib.check
        self.dev = torch.device(device)
        raw = text.encode("utf8") if isinstance(text, str) else bytes(text)
        if not 0 < len(raw) < (1 << 31):
            raise ValueError("corpus must hold 1 .. 2^31-1 bytes (split larger corpora at whitespace)")
        self.raw, self.nbytes = raw, len(raw)
        with torch.cuda.device(self.dev):
            self.st = torch.cuda.current_stream().cuda_stream
            self.text = torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(self.dev)
            ws = torch.empty(self.lib.glove_tokens_workspace_bytes(self.nbytes, 0), dtype=torch.uint8, device=self.dev)
            cap = self.nbytes // 2 + 1
            starts = torch.empty(cap, dtype=torch.int64, device=self.dev)
            lens = torch.empty(cap, dtype=torch.int32, device=self.dev)
            n = ctypes.c_int64()
            self.check(self.lib.glove_tokens_scan(self.text.data_ptr(), self.nbytes, ws.data_ptr(), ws.numel(), starts.data_ptr(),
                                                  lens.data_ptr(), cap, ctypes.byref(n), self.st), "glove_tokens_scan")
            self.n_tokens = n.value
            self.starts, self.lens = starts[:self.n_tokens].clone(), lens[:self.n_tokens].clone()

    def distinct(self):
        """(tokens, counts) of the distinct tokens in order of first occurrence -- Counter(text.split()) (ref text8.py:62)."""
        import torch
        with torch.cuda.device(self.dev):
            n = self.n_tokens
            ws = torch.empty(self.lib.glove_tokens_workspace_bytes(self.nbytes, n), dtype=torch.uint8, device=self.dev)
            first = torch.empty(n, dtype=torch.int64, device=self.dev)
            flen = torch.empty(n, dtype=torch.int32, device=self.dev)
            cnt = torch.empty(n, dtype=torch.int64, device=self.dev)
            m = ctypes.c_int64()
            self.check(self.lib.glove_tokens_count(self.text.data_ptr(), self.nbytes, self.starts.data_ptr(), n, ws.data_ptr(),
                                                   ws.numel(), first.data_ptr(), flen.data_ptr(), cnt.data_ptr(), n,
                                                   ctypes.byref(m), self.st), "glove_tokens_count")
            first, flen, cnt = (t[:m.value].cpu().numpy() for t in (first, flen, cnt))
        order = np.argsort(first, kind="stable")
        tokens = [self.raw[s:s + l].decode("utf8") for s, l in zip(first[order].tolist(), flen[order].tolist())]
        return tokens, cnt[order]

    def ids(self, vocab_tokens):
        """Device int32 id of every token: row of the vocabulary frame, unknown -> 0 (ref text8.py:85-86)."""
        import torch
        lines = [t.encode("utf8") for t in vocab_tokens]
        blob = b"".join(t + b"\n" for t in lines)
        off = np.zeros(len(lines) + 1, np.int64)
        np.cumsum([len(t) + 1 for t in lines], out=off[1:])
        with torch.cuda.device(self.dev):
            vb = torch.frombuffer(bytearray(blob), dtype=torch.uint8).to(self.dev)
            voff = torch.from_numpy(off).to(self.dev)
            slots = self.lib.glove_vocab_slots(len(lines))
            table = torch.empty(slots, dtype=torch.int32, device=self.dev)
            self.check(self.lib.glove_vocab_build(table.data_ptr(), slots, vb.data_ptr(), voff.data_ptr(), len(lines), self.st),
                       "glove_vocab_build")
            out = torch.empty(self.n_tokens, dtype=torch.int32, device=self.dev)
            self.check(self.lib.glove_tokens_lookup(self.text.data_ptr(), self.starts.data_ptr(), self.lens.data_ptr(),
                                                    self.n_tokens, table.data_ptr(), slots, vb.data_ptr(), voff.data_ptr(),
                                                    out.data_ptr(), self.st), "glove_tokens_lookup")
            torch.cuda.current_stream().synchronize()
        return out


def cooccurrence_table(ids, vocab_count, context_size=CONTEXT_SIZE, count_minimum=10, device="cuda:0",
                       chunk_positions=32 << 20, order_key=0, as_numpy=True):
    """Symmetric co-occurrence table of an id stream on the GPU.  Returns the numeric columns of interaction.csv
    (row_token_id, col_token_id int32; count int64; value, neg_weight, glove_weight, glove_value float64)."""
    import torch
    from . import _lib
    lib, check = _lib.lib, _lib.check
    dev = torch.device(device)
    V, T = len(vocab_count), len(ids)
    if T < 2:
        raise ValueError("need at least two tokens")
    with torch.cuda.device(dev):
        st = torch.cuda.current_stream().cuda_stream
        if torch.is_tensor(ids):
            d_ids = ids.to(device=dev, dtype=torch.int32).contiguous()
        else:
            d_ids = torch.as_tensor(np.array(ids, np.int32)).to(dev)
        d_vc = torch.as_tensor(np.array(vocab_count, np.int64)).to(dev)
        total = int(np.asarray(vocab_count, np.int64).sum())
        chunk = int(min(chunk_positions, T, ((1 << 31) - 1) // context_size))
        n_items = chunk * context_size
        ws = torch.empty(lib.glove_cooc_workspace_bytes(n_items), dtype=torch.uint8, device=dev)
        acc_k = acc_a = None
        n_acc = 0
        got = ctypes.c_int64()
        for p0 in range(0, T, chunk):
            n_pos = min(chunk, T - p0)
            n_tok = min(n_pos + context_size, T - p0)
            cap = n_pos * context_size
            k = torch.empty(cap, dtype=torch.int64, device=dev)
            a = torch.empty(2 * cap, dtype=torch.int64, device=dev)
            check(lib.glove_cooc_chunk(d_ids[p0:].data_ptr(), n_pos, n_tok, V, context_size, ws.data_ptr(), ws.numel(),
                                       k.data_ptr(), a.data_ptr(), cap, ctypes.byref(got), st), "glove_cooc_chunk")
            n = got.value
            k, a = k[:n].clone(), a[:2 * n].clone()
            if acc_k is None:
                acc_k, acc_a, n_acc = k, a, n
                continue
            if n == 0:
                continue
            m = n_acc + n
            if lib.glove_cooc_workspace_bytes(m) > ws.numel():
                ws = torch.empty(lib.glove_cooc_workspace_bytes(m), dtype=torch.uint8, device=dev)
            ok_, oa = torch.empty(m, dtype=torch.int64, device=dev), torch.empty(2 * m, dtype=torch.int64, device=dev)
            check(lib.glove_cooc_merge(acc_k.data_ptr(), acc_a.data_ptr(), n_acc, k.data_ptr(), a.data_ptr(), n, V,
                                       ws.data_ptr(), ws.numel(), ok_.data_ptr(), oa.data_ptr(), m, ctypes.byref(got), st),
                  "glove_cooc_merge")
            n_acc = got.value
            acc_k, acc_a = ok_[:n_acc].clone(), oa[:2 * n_acc].clone()
        names = ("row_token_id", "col_token_id", "count", "value", "neg_weight", "glove_weight", "glove_value")
        dts = (torch.int32, torch.int32, torch.int64, torch.float64, torch.float64, torch.float64, torch.float64)
        if n_acc == 0:
            out = [torch.empty(0, dtype=dt, device=dev) for dt in dts]
        else:
            if lib.glove_cooc_workspace_bytes(2 * n_acc) > ws.numel():
                ws = torch.empty(lib.glove_cooc_workspace_bytes(2 * n_acc), dtype=torch.uint8, device=dev)
            cap = 2 * n_acc
            out = [torch.empty(cap, dtype=dt, device=dev) for dt in dts]
            check(lib.glove_cooc_finish(acc_k.data_ptr(), acc_a.data_ptr(), n_acc, V, context_size, count_minimum,
                                        d_vc.data_ptr(), total, order_key, ws.data_ptr(), ws.numel(),
                                        *[t.data_ptr() for t in out], cap, ctypes.byref(got), st), "glove_cooc_finish")
            out = [t[:got.value] for t in out]
    if as_numpy:
        return {n: t.cpu().numpy() for n, t in zip(names, out)}
    return dict(zip(names, out))


def create_interaction_dataframe(text_tokens, df_vocab, context_size=CONTEXT_SIZE, count_minimum=10, device="cuda:0"):
    """interaction frame in the reference's column order, GloVe columns included (ref text8.py:84-139: the reference builds
    it in two steps, create_interaction_dataframe + create_glove_dataframe; the GPU kernel writes all columns at once)."""
    import pandas as pd
    vocab_tokens = df_vocab["token"].to_numpy()
    ids = token_ids(text_tokens, vocab_tokens)
    t = cooccurrence_table(ids, df_vocab["count"].to_numpy(), context_size, count_minimum, device)
    frame = interaction_frame(t, vocab_tokens)
    logger.info("dataframe shape: %s.", frame.shape)
    return frame


def interaction_frame(table, vocab_tokens):
    """The reference's interaction.csv columns, in its order, from the numeric table (ref text8.py:113-114 for the tokens)."""
    import pandas as pd
    vocab_tokens = np.asarray(vocab_tokens, dtype=object)
    return pd.DataFrame({"row_token_id": table["row_token_id"], "col_token_id": table["col_token_id"], "count": table["count"],
                         "value": table["value"], "row_token": vocab_tokens[table["row_token_id"]],
                         "col_token": vocab_tokens[table["col_token_id"]], "neg_weight": table["neg_weight"],
                         "glove_weight": table["glove_weight"], "glove_value": table["glove_value"]})


def process_data(text8, vocab_size=VOCAB_SIZE, coverage=COVERAGE, context_size=CONTEXT_SIZE, device="cuda:0"):
    """ref text8.py:46-58, with the token stream kept on the GPU from the split to the table: tokenise, count distinct
    tokens, (host: pick the vocabulary among them), map tokens to ids, count pairs, write the columns."""
    corpus = DeviceCorpus(text8, device)
    tokens, counts = corpus.distinct()
    df_vocab = _frame_from_counts(tokens, counts, None if vocab_size is None else int(vocab_size), coverage)
    logger.info("vocab created, size: %s.", df_vocab.shape[0])
    vocab_tokens = df_vocab["token"].to_numpy()
    table = cooccurrence_table(corpus.ids(vocab_tokens), df_vocab["count"].to_numpy(), context_size, 10, device)
    frame = interaction_frame(table, vocab_tokens)
    logger.info("dataframe shape: %s.", frame.shape)
    return {"vocabulary": df_vocab, "interaction": frame}


def save_data(data, save_dir=DATA_DIR):
    """vocab.csv, vocab.txt (one token per line, no trailing newline), interaction.csv (ref text8.py:142-156)."""
    os.makedirs(save_dir, exist_ok=True)
    data["vocabulary"].to_csv(os.path.join(save_dir, "vocab.csv"), index=False)
    with open(os.path.join(save_dir, "vocab.txt"), "w") as f:
        f.write("\n".join(data["vocabulary"]["token"]))
    data["interaction"].to_csv(os.path.join(save_dir, "interaction.csv"), index=False)
    return data


def main(argv=None):
    logging.basicConfig(level=logging.INFO, format="%(asctime)s - %(levelname)s - %(name)s - %(message)s")
    ap = ArgumentParser(description="Download, extract and prepare text8 data.")
    ap.add_argument("--url", default=TEXT8_URL, help="url of text8 data (default: %(default)s)")
    ap.add_argument("--dest", default=DATA_DIR, help="destination directory for downloaded and extracted files (default: %(default)s)")
    ap.add_argument("--vocab-size", type=int, default=VOCAB_SIZE, help="maximum size of vocab (default: %(default)s)")
    ap.add_argument("--coverage", type=float, default=COVERAGE, help="token coverage to set token count cutoff (default: %(default)s)")
    ap.add_argument("--context-size", type=int, default=CONTEXT_SIZE, help="size of context window (default: %(default)s)")
    ap.add_argument("--device", default="cuda:0")
    args = ap.parse_args(argv)
    logger.info("call: %s.", " ".join(sys.argv))
    download_data(args.url, args.dest)
    from .corpus import preprocess     # the streamed preprocessor: same files as save_data(process_data(...))
    preprocess(os.path.join(args.dest, "text8"), args.dest, args.vocab_size, args.coverage, args.context_size, args.device)


if __name__ == "__main__":
    main()
