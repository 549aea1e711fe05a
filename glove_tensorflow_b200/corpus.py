"""``python -m glove_tensorflow_b200.corpus --corpus PATH --dest DIR``: corpus text of any size -> vocab.csv, vocab.txt,
interaction.csv, streamed through the GPU in two passes.

The output is byte for byte what ``text8.save_data(text8.process_data(text))`` writes for the same text: tokens of
``str.split()``, the vocabulary of ``text8._frame_from_counts``, right context 1..context_size, count >= 10, the reference's
columns, records in the keyed-hash order.  Unlike that in-memory path it never holds the corpus, its token stream or the
whole pair table on the device at once:

- the file is read in chunks cut after their last ASCII whitespace byte (UTF-8 puts no ASCII byte inside a multi-byte
  sequence); the cut-off tail is carried in front of the next chunk;
- pass 1 counts the distinct tokens of every chunk and merges them on the device into one table of distinct tokens
  (csrc/glove_corpus.cu); only those go to the host, which picks the vocabulary;
- pass 2 maps tokens to ids and counts right-context pairs per block of positions (glove_cooc_chunk), routes both
  orientations of every pair to one of 2^k partitions by the top bits of its record-order hash (glove_cooc_route) and
  merges them into that partition's accumulator (glove_cooc_merge); each partition is then finished on its own
  (glove_cooc_finish_sorted) and, in ascending partition order, its records are formatted into csv lines on the device
  (glove_cooc_csv_*) and written by a thread while the next block is formatted.  With ``--format stanford`` / ``both``
  the same records also go out as Stanford GloVe's binary cooccurrence.shuf.bin (glove_cooc_bin_format).

With ``--scheme stanford`` the same two passes follow Stanford GloVe's vocab_count and cooccur instead and write
vocab.txt (``word count`` lines) and cooccurrence.shuf.bin: vocabulary by count (ties in byte order), out-of-vocabulary
words removed from the stream, windows of up to 15 words that never cross a line end, self pairs kept, every pair
written (DESIGN.md §3, "Stanford GloVe preprocessing").

The device must hold the pair table: about 24 bytes per directed pair plus one merge workspace.  A table that does not
fit is refused with the figure (DESIGN.md §3, "Streamed corpus preprocessing")."""
import contextlib
import csv
import ctypes
import io
import logging
import math
import os
import re
import sys
from argparse import ArgumentParser
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from .config import CONTEXT_SIZE, COVERAGE, VOCAB_SIZE
from .data_utils import _HEAD, _ChunkReader

logger = logging.getLogger(__name__)

COLUMNS = ("row_token_id", "col_token_id", "count", "value", "row_token", "col_token", "neg_weight", "glove_weight",
           "glove_value")
_SPACE = np.zeros(256, bool)                      # the ASCII whitespace of str.split()
_SPACE[[0x09, 0x0a, 0x0b, 0x0c, 0x0d, 0x20, 0x1c, 0x1d, 0x1e, 0x1f]] = True
# UTF-8 of the non-ASCII separators str.split() knows (the token scanner refuses them)
_UNICODE_SPACE = re.compile(rb"\xc2[\x85\xa0]|\xe1\x9a\x80|\xe2\x80[\x80-\x8a\xa8\xa9\xaf]|\xe2\x81\x9f|\xe3\x80\x80")
_PAIR_BYTES = 24                                  # one accumulated directed pair: u64 key + {count, numer}
_MAX_PART_BITS = 12
FORMATS = ("csv", "stanford", "both")             # table containers preprocess() writes
SCHEMES = ("reference", "stanford")               # counting rules: text8.process_data's, or vocab_count + cooccur's
STANFORD_MAX_WINDOW = 15
# bytes Stanford's tokenizer glues into tokens but the vocabulary readers split on (glove_text_refused)
_REFUSED = {0x0b: "a vertical tab", 0x0c: "a form feed", 0x0d: "a carriage return not followed by a line feed",
            **{b: "the separator byte 0x%02x" % b for b in range(0x1c, 0x20)}}


def text_chunks(path, chunk_bytes, bufs):
    """Yields ``(k, lo, hi, origin, final)`` for the chunks of the file: ``bufs[k % 2][lo:hi]`` is the chunk's text, which
    ends after its last ASCII whitespace byte (the final chunk: at the end of the file), and ``origin`` is the file offset
    of ``bufs[k % 2][lo]``.  A chunk without whitespace is carried whole into the next one.  The text starts 16-byte
    aligned; bytes in front of the carried tail are padded with '\\n'.  ``bufs``: two uint8 arrays of ``_HEAD +
    chunk_bytes`` (the same one twice for a file of one chunk).  The caller must be done with a chunk, asynchronous copies
    included, before it asks for the next.  A token longer than the carry area (``_HEAD - 16`` bytes) fails with its byte
    offset."""
    head = _HEAD
    size = os.path.getsize(path)
    reader = _ChunkReader(path, 0, size, chunk_bytes, bufs)
    try:
        n_chunks, carry = reader.n_chunks(), 0
        reader.start(0)
        for k in range(n_chunks):
            n_new = reader.wait(k)
            reader.start(k + 1)
            buf = bufs[k % 2]
            lo = (head - carry) // 16 * 16
            buf[lo:head - carry] = 0x0A
            end = head + n_new
            pos = k * chunk_bytes                   # file offset of buf[head]
            final = k == n_chunks - 1
            hi = end if final else _cut(buf, head - carry, end)
            if end - hi > head - 16:
                raise ValueError("%s: the token at byte %d is longer than %d bytes" % (path, pos + hi - head, head - 16))
            if hi > head - carry:
                yield k, lo, hi, pos - (head - lo), final
            carry = end - hi
            if carry:   # the tail goes in front of the next chunk (which is being read into the other buffer)
                bufs[(k + 1) % 2][head - carry:head] = buf[hi:end]
    finally:
        reader.close()


def _cut(buf, lo, end, window=4096):
    """One past the last whitespace byte of buf[lo:end]; lo when there is none."""
    while True:
        w0 = max(lo, end - window)
        hit = np.flatnonzero(_SPACE[buf[w0:end]])
        if len(hit):
            return w0 + int(hit[-1]) + 1
        if w0 == lo:
            return lo
        window *= 16


def csv_quote(token):
    """A token as pandas' to_csv writes it (csv.QUOTE_MINIMAL)."""
    out = io.StringIO()
    csv.writer(out, lineterminator="\n").writerow([token])
    return out.getvalue()[:-1]


class _Device:
    """The library, the device and its stream, and the device-memory budget of the pair table."""

    def __init__(self, device, device_bytes):
        import torch
        from . import _lib
        self.torch, self.lib, self.check = torch, _lib.lib, _lib.check
        self.dev = torch.device(device)
        self.device_bytes = device_bytes

    def free_bytes(self):
        torch = self.torch
        free, _ = torch.cuda.mem_get_info(self.dev)
        return free + torch.cuda.memory_reserved(self.dev) - torch.cuda.memory_allocated(self.dev)

    def empty(self, n, dtype):
        return self.torch.empty(max(int(n), 1), dtype=dtype, device=self.dev)


def _scan(d, path, text, fill, host_text, origin):
    """Token starts and lengths of one chunk on the device."""
    torch, lib = d.torch, d.lib
    st = torch.cuda.current_stream().cuda_stream
    ws = d.empty(lib.glove_tokens_workspace_bytes(fill, 0), torch.uint8)
    cap = fill // 2 + 1
    starts, lens = d.empty(cap, torch.int64), d.empty(cap, torch.int32)
    n = ctypes.c_int64()
    rc = lib.glove_tokens_scan(text.data_ptr(), fill, ws.data_ptr(), ws.numel(), starts.data_ptr(), lens.data_ptr(), cap,
                               ctypes.byref(n), st)
    if rc != 0:
        m = _UNICODE_SPACE.search(host_text.tobytes())
        if m is not None:
            raise ValueError("%s: byte %d: non-ASCII Unicode whitespace, which str.split() would split on"
                             % (path, origin + m.start()))
        d.check(rc, "glove_tokens_scan")
    return starts, lens, n.value


def _chunk_loop(d, path, chunk_bytes):
    """Yields (device text, fill, host text view, origin, final) for every chunk (pass 1 and pass 2 read the file
    alike)."""
    torch = d.torch
    size = os.path.getsize(path)
    chunk = int(max(64, min(chunk_bytes, size, (1 << 30)))) // 16 * 16
    pinned = [torch.empty(_HEAD + chunk, dtype=torch.uint8, pin_memory=True) for _ in range(2 if size > chunk else 1)]
    host = [t.numpy() for t in pinned]
    text = torch.empty(_HEAD + chunk, dtype=torch.uint8, device=d.dev)
    for k, lo, hi, origin, final in text_chunks(path, chunk, host * (2 // len(host))):
        fill = hi - lo
        text[:fill].copy_(pinned[k % len(pinned)][lo:hi], non_blocking=True)
        yield text, fill, host[k % len(host)][lo:hi], origin, final
        torch.cuda.current_stream().synchronize()


def _refuse_bytes(d, path, text, fill, host_text, origin, final, scratch):
    """Raises ValueError naming the lowest offset of a byte glove_text_refused refuses, or of a non-ASCII separator
    before it."""
    first = ctypes.c_int64()
    nxt = -1
    if not final and host_text[-1] == 0x0d:          # the byte after the chunk decides a \r at its end
        with open(path, "rb") as f:
            f.seek(origin + fill)
            nxt = f.read(1)[0]
    d.check(d.lib.glove_text_refused(text.data_ptr(), fill, nxt, scratch.data_ptr(), ctypes.byref(first),
                                     d.torch.cuda.current_stream().cuda_stream), "glove_text_refused")
    if first.value < 0:
        return
    m = _UNICODE_SPACE.search(host_text[:first.value].tobytes())
    if m is not None:
        raise ValueError("%s: byte %d: non-ASCII Unicode whitespace, which str.split() would split on"
                         % (path, origin + m.start()))
    raise ValueError("%s: byte %d: %s, which Stanford GloVe's tokenizer would keep inside a token"
                     % (path, origin + first.value, _REFUSED[int(host_text[first.value])]))


def count_tokens(d, path, chunk_bytes, stanford=False):
    """Pass 1: (tokens in order of first occurrence, their counts), and with ``stanford`` also the file offset of each
    token's first occurrence; ``stanford`` also refuses the bytes of ``_REFUSED``."""
    torch, lib, check = d.torch, d.lib, d.check
    st = torch.cuda.current_stream().cuda_stream
    g = None                     # global table: hash, count, first, off, len
    n_g, pool_used = 0, 0
    pool = d.empty(1 << 20, torch.uint8)
    scratch = d.empty(1, torch.int64)
    for text, fill, host_text, origin, final in _chunk_loop(d, path, chunk_bytes):
        if stanford:
            _refuse_bytes(d, path, text, fill, host_text, origin, final, scratch)
        starts, _, n = _scan(d, path, text, fill, host_text, origin)
        if n == 0:
            continue
        ws = d.empty(lib.glove_tokens_workspace_bytes(fill, n), torch.uint8)
        first, flen, cnt = d.empty(n, torch.int64), d.empty(n, torch.int32), d.empty(n, torch.int64)
        m = ctypes.c_int64()
        check(lib.glove_tokens_count(text.data_ptr(), fill, starts.data_ptr(), n, ws.data_ptr(), ws.numel(), first.data_ptr(),
                                     flen.data_ptr(), cnt.data_ptr(), n, ctypes.byref(m), st), "glove_tokens_count")
        m = m.value
        if pool.numel() < pool_used + fill:          # new token bytes of a chunk never exceed its size
            bigger = d.empty(max(2 * pool.numel(), pool_used + fill), torch.uint8)
            bigger[:pool_used].copy_(pool[:pool_used])
            pool = bigger
        cap = n_g + m
        out = (d.empty(cap, torch.int64), d.empty(cap, torch.int64), d.empty(cap, torch.int64), d.empty(cap, torch.int64),
               d.empty(cap, torch.int32))
        ws = d.empty(lib.glove_vocab_merge_workspace_bytes(n_g, m), torch.uint8)
        gp = [t.data_ptr() for t in g] if g is not None else [None] * 5
        n_out, used = ctypes.c_int64(), ctypes.c_int64()
        check(lib.glove_vocab_merge(text.data_ptr(), origin, first.data_ptr(), flen.data_ptr(), cnt.data_ptr(), m, *gp, n_g,
                                    pool.data_ptr(), pool_used, pool.numel(), ws.data_ptr(), ws.numel(),
                                    *[t.data_ptr() for t in out], cap, ctypes.byref(n_out), ctypes.byref(used), st),
              "glove_vocab_merge")
        g, n_g, pool_used = out, n_out.value, used.value
    if n_g == 0:
        return ([], np.zeros(0, np.int64)) + ((np.zeros(0, np.int64),) if stanford else ())
    _, count, first, off, ln = (t[:n_g].cpu().numpy() for t in g)
    blob = pool[:pool_used].cpu().numpy().tobytes()
    order = np.argsort(first, kind="stable")
    tokens = [blob[s:s + n].decode("utf8") for s, n in zip(off[order].tolist(), ln[order].tolist())]
    return (tokens, count[order]) + ((first[order],) if stanford else ())


def stanford_vocab(tokens, counts, min_count=1, max_vocab=0):
    """Stanford vocab_count's vocabulary: the tokens with count >= min_count, by count descending and equal counts in
    byte order (strcmp), the first max_vocab of them (0: all).  Returns (tokens, int64 counts); a token's id is its
    rank."""
    keep = [i for i in range(len(tokens)) if counts[i] >= min_count]
    keep.sort(key=lambda i: (-int(counts[i]), tokens[i].encode("utf8")))
    if max_vocab:
        keep = keep[:max_vocab]
    return [tokens[i] for i in keep], np.array([counts[i] for i in keep], np.int64)


def _part_bits(vocab_size, n_tokens, context_size, partition_entries, diagonal=False):
    """Smallest k such that 2^k partitions of the largest possible table (every position pair distinct, or every
    ordered pair of vocabulary rows, the diagonal included when self pairs are kept) hold at most ``partition_entries``
    directed pairs each."""
    bound = min(vocab_size * (vocab_size if diagonal else vocab_size - 1), 2 * n_tokens * context_size)
    k = 0
    while (bound >> k) > partition_entries and k < _MAX_PART_BITS:
        k += 1
    return k


class _Pairs:
    """Pass 2 accumulators: one sorted, reduced table of directed pairs per partition.  ``stanford``: None for the
    reference rules, or (window, distance_weighting, symmetric)."""

    def __init__(self, d, V, part_bits, order_key, stanford=None):
        self.d, self.V, self.part_bits, self.order_key, self.stanford = d, V, part_bits, order_key, stanford
        self.acc = [None] * (1 << part_bits)
        self.n = [0] * (1 << part_bits)
        self.ws = d.empty(0, d.torch.uint8)

    def _workspace(self, n_items):
        need = self.d.lib.glove_cooc_workspace_bytes(n_items)
        if self.ws.numel() < need:
            self.ws = None
            self.ws = self.d.empty(need, self.d.torch.uint8)
        return self.ws

    def require(self, out_bytes, n_work):
        """Refuses, with the figure, a step that would not fit the device: out_bytes of new buffers and a workspace of
        n_work items next to the pairs held so far."""
        d = self.d
        held = sum(self.n) * _PAIR_BYTES + self.ws.numel()
        ws_bytes = d.lib.glove_cooc_workspace_bytes(n_work)
        need = out_bytes + max(ws_bytes - self.ws.numel(), 0)
        budget = d.device_bytes if d.device_bytes is not None else d.free_bytes() + held
        if held + need > budget:
            raise MemoryError("the co-occurrence table needs %.3g GB of device memory (%d directed pairs at %d bytes, "
                              "%.3g GB of new buffers and a %.3g GB merge workspace); %.3g GB are available"
                              % ((held + need) / 1e9, sum(self.n), _PAIR_BYTES, out_bytes / 1e9, ws_bytes / 1e9,
                                 budget / 1e9))

    def add(self, keys, agg, n):
        """Routes both orientations of a right-context table (n entries), or only (left, right) for an asymmetric
        Stanford table, and merges them into the partitions."""
        d, torch, lib, check = self.d, self.d.torch, self.d.lib, self.d.check
        st = torch.cuda.current_stream().cuda_stream
        P = 1 << self.part_bits
        n_out = n if self.stanford is not None and not self.stanford[2] else 2 * n
        rk, ra = d.empty(n_out, torch.int64), d.empty(2 * n_out, torch.int64)
        rws = d.empty(lib.glove_cooc_route_workspace_bytes(n, self.part_bits), torch.uint8)
        counts = np.zeros(P, np.int64)
        if self.stanford is None:
            check(lib.glove_cooc_route(keys.data_ptr(), agg.data_ptr(), n, self.V, self.order_key, self.part_bits,
                                       rws.data_ptr(), rws.numel(), rk.data_ptr(), ra.data_ptr(), n_out, counts.ctypes.data, st),
                  "glove_cooc_route")
        else:
            check(lib.glove_cooc_route_stanford(keys.data_ptr(), agg.data_ptr(), n, self.V, self.order_key, self.part_bits,
                                                int(self.stanford[2]), rws.data_ptr(), rws.numel(), rk.data_ptr(), ra.data_ptr(),
                                                n_out, counts.ctypes.data, st), "glove_cooc_route_stanford")
        del rws
        got = ctypes.c_int64()
        o = 0
        for p in range(P):
            c = int(counts[p])
            if c == 0:
                continue
            m = self.n[p] + c
            if m >= 1 << 31:
                raise MemoryError("co-occurrence partition %d would hold %d entries (limit 2^31)" % (p, m))
            self.require(_PAIR_BYTES * m, m)
            ws = self._workspace(m)
            ok_, oa = d.empty(m, torch.int64), d.empty(2 * m, torch.int64)
            if self.acc[p] is None:
                ak, aa = rk, ra        # merging with an empty table: sorts and reduces the routed entries
            else:
                ak, aa = self.acc[p]
            check(lib.glove_cooc_merge(ak.data_ptr(), aa.data_ptr(), self.n[p], rk[o:].data_ptr(), ra[2 * o:].data_ptr(), c,
                                       self.V, ws.data_ptr(), ws.numel(), ok_.data_ptr(), oa.data_ptr(), m,
                                       ctypes.byref(got), st), "glove_cooc_merge")
            self.n[p] = got.value
            self.acc[p] = (ok_[:got.value].clone(), oa[:2 * got.value].clone())
            del ok_, oa
            o += c

    def finish(self, p, vocab_count, total, context_size):
        """Records of partition p in the keyed-hash order (device columns), and frees the partition."""
        d, torch, lib, check = self.d, self.d.torch, self.d.lib, self.d.check
        st = torch.cuda.current_stream().cuda_stream
        n = self.n[p]
        keys, agg = self.acc[p]
        self.require(48 * n, n)                      # the columns (48 bytes a record) and the finish workspace
        ws = self._workspace(n)
        dts = (torch.int32, torch.int32, torch.int64, torch.float64, torch.float64, torch.float64, torch.float64)
        out = [d.empty(n, dt) for dt in dts]
        got = ctypes.c_int64()
        if self.stanford is None:
            check(lib.glove_cooc_finish_sorted(keys.data_ptr(), agg.data_ptr(), n, self.V, context_size, 10,
                                               vocab_count.data_ptr(), total, self.order_key, ws.data_ptr(), ws.numel(),
                                               *[t.data_ptr() for t in out], n, ctypes.byref(got), st), "glove_cooc_finish_sorted")
        else:
            check(lib.glove_cooc_finish_stanford(keys.data_ptr(), agg.data_ptr(), n, self.V, context_size,
                                                 int(self.stanford[1]), vocab_count.data_ptr(), total, self.order_key,
                                                 ws.data_ptr(), ws.numel(), *[t.data_ptr() for t in out], n, ctypes.byref(got),
                                                 st), "glove_cooc_finish_stanford")
        self.acc[p], self.n[p] = None, 0
        return [t[:got.value] for t in out]


class _PinnedWriter:
    """Writes device bytes to a file: each block is copied to one of two pinned buffers and written by a thread while
    the device prepares the next one."""

    def __init__(self, d, f):
        self.d, self.f = d, f
        self.pinned, self.pending, self.k = [None, None], [None, None], 0
        self.pool = ThreadPoolExecutor(max_workers=1)
        self.bytes = 0

    def _write(self, buf, nbytes, ev):
        ev.synchronize()
        self.f.write(buf.numpy()[:nbytes].data)

    def put(self, data, nbytes):
        """Queues data[:nbytes] (a device tensor of uint8, ready once the current stream reaches this point)."""
        torch = self.d.torch
        s = self.k % 2
        self.k += 1
        if self.pending[s] is not None:
            self.pending[s].result()           # the writer is done with this pinned buffer
        if self.pinned[s] is None or self.pinned[s].numel() < nbytes:
            self.pinned[s] = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
        self.pinned[s][:nbytes].copy_(data[:nbytes], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        self.pending[s] = self.pool.submit(self._write, self.pinned[s], nbytes, ev)
        self.bytes += nbytes

    def close(self):
        try:
            for p in self.pending:
                if p is not None:
                    p.result()
        finally:
            self.pool.shutdown(wait=True)


class _CsvWriter(_PinnedWriter):
    """interaction.csv: header, then blocks of records formatted on the device."""

    def __init__(self, d, f, vocab_tokens):
        super().__init__(d, f)
        torch = d.torch
        quoted = [csv_quote(t).encode("utf8") for t in vocab_tokens]
        off = np.zeros(len(quoted) + 1, np.int64)
        np.cumsum([len(q) for q in quoted], out=off[1:])
        self.tok = torch.frombuffer(bytearray(b"".join(quoted)), dtype=torch.uint8).to(d.dev)
        self.tok_off = torch.from_numpy(off).to(d.dev)
        self.text = d.empty(0, torch.uint8)
        f.write((",".join(COLUMNS) + "\n").encode())

    def write(self, cols, records_per_block):
        d, torch, lib, check = self.d, self.d.torch, self.d.lib, self.d.check
        st = torch.cuda.current_stream().cuda_stream
        n_all = len(cols[0])
        for r0 in range(0, n_all, records_per_block):
            n = min(records_per_block, n_all - r0)
            ptrs = [t[r0:].data_ptr() for t in cols]
            ws = d.empty(lib.glove_cooc_csv_workspace_bytes(n), torch.uint8)
            nbytes = ctypes.c_int64()
            check(lib.glove_cooc_csv_size(*ptrs, n, self.tok_off.data_ptr(), ws.data_ptr(), ws.numel(), ctypes.byref(nbytes),
                                          st), "glove_cooc_csv_size")
            nbytes = nbytes.value
            if self.text.numel() < nbytes:
                self.text = None
                self.text = d.empty(nbytes, torch.uint8)
            check(lib.glove_cooc_csv_format(*ptrs, n, self.tok.data_ptr(), self.tok_off.data_ptr(), ws.data_ptr(), ws.numel(),
                                            self.text.data_ptr(), self.text.numel(), st), "glove_cooc_csv_format")
            self.put(self.text, nbytes)


class _BinWriter(_PinnedWriter):
    """cooccurrence.shuf.bin: Stanford GloVe's 16-byte records (ids + 1, float64 value), formatted on the device in
    blocks of records (glove_cooc_bin_format)."""

    def __init__(self, d, f):
        super().__init__(d, f)
        self.recs = d.empty(0, d.torch.uint8)

    def write(self, cols, records_per_block):
        d, torch, lib, check = self.d, self.d.torch, self.d.lib, self.d.check
        st = torch.cuda.current_stream().cuda_stream
        row, col, value = cols[0], cols[1], cols[3]
        n_all = len(row)
        for r0 in range(0, n_all, records_per_block):
            n = min(records_per_block, n_all - r0)
            if self.recs.numel() < 16 * n:
                self.recs = None
                self.recs = d.empty(16 * n, torch.uint8)
            check(lib.glove_cooc_bin_format(row[r0:].data_ptr(), col[r0:].data_ptr(), value[r0:].data_ptr(), n,
                                            self.recs.data_ptr(), st), "glove_cooc_bin_format")
            self.put(self.recs, 16 * n)


def _newline_after_last_token(text, newline_before):
    """Whether a '\\n' follows the last token of ``text`` (a chunk's own bytes); for a chunk without tokens, whether one
    lies in it or before it."""
    i, window = len(text), 4096
    while i > 0:
        j = max(0, i - window)
        hit = np.flatnonzero(~_SPACE[text[j:i]])
        if len(hit):
            return bool((text[j + int(hit[-1]) + 1:] == 0x0A).any())
        i, window = j, window * 16
    return newline_before or bool((text == 0x0A).any())


class _StanfordStream:
    """Pass 2 of the Stanford scheme: the in-vocabulary tokens of each chunk, in text order, as (line segment << 32) |
    id (glove_tokens_stream); the segment and the '\\n' after the last token carry over to the next chunk."""

    def __init__(self, d, vocab):
        self.d, self.vocab = d, vocab
        self.end, self.newline, self.segment = 0, False, 0

    def ids(self, text, fill, host_text, origin, starts, lens, n):
        d, torch = self.d, self.d.torch
        begin = self.end - origin                     # the chunk's own bytes start here (the rest is padding)
        self.end = origin + fill
        if n == 0:
            self.newline = _newline_after_last_token(host_text[begin:], self.newline)
            return torch.empty(0, dtype=torch.int64, device=d.dev)
        table, slots, vb, voff = self.vocab
        ws = d.empty(d.lib.glove_tokens_stream_workspace_bytes(n), torch.uint8)
        out = d.empty(n, torch.int64)
        got, last = ctypes.c_int64(), ctypes.c_uint32()
        d.check(d.lib.glove_tokens_stream(text.data_ptr(), begin, starts.data_ptr(), lens.data_ptr(), n, int(self.newline),
                                          self.segment, table.data_ptr(), slots, vb.data_ptr(), voff.data_ptr(), ws.data_ptr(),
                                          ws.numel(), out.data_ptr(), n, ctypes.byref(got), ctypes.byref(last),
                                          torch.cuda.current_stream().cuda_stream), "glove_tokens_stream")
        self.segment = last.value
        self.newline = _newline_after_last_token(host_text[begin:], False)
        return out[:got.value]


def _stanford_numerator_bound(n_tokens, window, distance_weighting, symmetric):
    """The largest numerator a pair can reach: every position adds at most sum_k w_k per orientation."""
    unit = math.lcm(*range(1, window + 1))
    per_position = sum(unit // k for k in range(1, window + 1)) if distance_weighting else window
    return int(n_tokens) * per_position * (2 if symmetric else 1)


def preprocess(corpus, dest, vocab_size=VOCAB_SIZE, coverage=COVERAGE, context_size=CONTEXT_SIZE, device="cuda:0",
               chunk_bytes=256 << 20, chunk_positions=16 << 20, partition_entries=1 << 27, records_per_block=1 << 22,
               order_key=0, device_bytes=None, stats=None, format="csv", scheme="reference", window_size=15, min_count=1,
               max_vocab=0, symmetric=True, distance_weighting=True):
    """Writes ``<dest>/vocab.csv``, ``vocab.txt`` and ``interaction.csv`` for the corpus file ``corpus``, byte for byte as
    ``text8.save_data(text8.process_data(text))`` does.  Returns ``(vocabulary frame, number of interaction records)``.

    ``format``: ``"csv"`` (the above), ``"stanford"`` or ``"both"``.  The last two also write the table as Stanford
    GloVe's ``cooccurrence.shuf.bin`` (16-byte records ``int32 word1, int32 word2, float64 value``, ids 1-based lines of
    vocab.txt, in interaction.csv's record order) and ``vocab.stanford.txt`` (``token count`` lines in vocab.txt order);
    ``"stanford"`` writes no interaction.csv.

    ``scheme="stanford"`` counts as Stanford GloVe's ``vocab_count -min-count min_count -max-vocab max_vocab`` and
    ``cooccur -window-size window_size -symmetric symmetric -distance-weighting distance_weighting`` do and writes
    ``<dest>/vocab.txt`` (``word count`` lines) and ``<dest>/cooccurrence.shuf.bin`` only; ``vocab_size``, ``coverage``,
    ``context_size`` and ``format`` are then unused.  Returns the vocabulary (columns token, count) and the record
    count.  The rules are those of DESIGN.md §3, "Stanford GloVe preprocessing".

    ``chunk_bytes``: text read per chunk (< 1 GiB); ``chunk_positions``: token positions per pair-counting block;
    ``partition_entries``: target directed pairs per partition of the table (the partition count follows from it and the
    corpus; small values exercise the partitioning); ``device_bytes``: device memory the pair table may use (default:
    what is free).  ``stats``: a dict that receives pass timings and sizes."""
    import time
    import pandas as pd
    from .text8 import _frame_from_counts
    if scheme not in SCHEMES:
        raise ValueError("scheme must be one of %s, got %r" % (", ".join(SCHEMES), scheme))
    stanford = scheme == "stanford"
    if stanford:
        if not 1 <= int(window_size) <= STANFORD_MAX_WINDOW:
            raise ValueError("window_size must be 1..%d" % STANFORD_MAX_WINDOW)
        if int(min_count) < 1 or int(max_vocab) < 0:
            raise ValueError("min_count must be >= 1 and max_vocab >= 0")
    elif not 1 <= int(context_size) <= 8:
        raise ValueError("context_size must be 1..8")
    if format not in FORMATS:
        raise ValueError("format must be one of %s, got %r" % (", ".join(FORMATS), format))
    if os.path.getsize(corpus) == 0:
        raise ValueError("%s: empty corpus" % corpus)
    d = _Device(device, device_bytes)
    torch, lib, check = d.torch, d.lib, d.check
    stats = {} if stats is None else stats
    with torch.cuda.device(d.dev):
        st = torch.cuda.current_stream().cuda_stream
        t0 = time.perf_counter()
        with torch.profiler.record_function("corpus.pass1"):
            tokens, counts, *first = count_tokens(d, corpus, chunk_bytes, stanford)
        n_tokens = int(counts.sum())
        if n_tokens < 2:
            raise ValueError("%s: need at least two tokens, the corpus holds %d" % (corpus, n_tokens))
        os.makedirs(dest, exist_ok=True)
        if stanford:
            if "<unk>" in tokens:
                raise ValueError("%s: byte %d: the token <unk>, which Stanford GloVe reserves"
                                 % (corpus, int(first[0][tokens.index("<unk>")])))
            ctx = int(window_size)
            if _stanford_numerator_bound(n_tokens, ctx, distance_weighting, symmetric) >= 1 << 63:
                raise ValueError("%s: %d tokens: a pair's exact weight sum could overflow 64 bits" % (corpus, n_tokens))
            vocab_tokens, vocab_counts = stanford_vocab(tokens, counts, int(min_count), int(max_vocab))
            if not vocab_tokens:
                raise ValueError("%s: no token occurs at least %d times" % (corpus, min_count))
            df_vocab = pd.DataFrame({"token": vocab_tokens, "count": vocab_counts})
            with open(os.path.join(dest, "vocab.txt"), "w", encoding="utf8") as f:
                f.writelines("%s %d\n" % (t, c) for t, c in zip(vocab_tokens, vocab_counts.tolist()))
        else:
            ctx = int(context_size)
            df_vocab = _frame_from_counts(tokens, counts, None if vocab_size is None else int(vocab_size), coverage)
            vocab_tokens = df_vocab["token"].tolist()
            df_vocab.to_csv(os.path.join(dest, "vocab.csv"), index=False)
            with open(os.path.join(dest, "vocab.txt"), "w") as f:
                f.write("\n".join(df_vocab["token"]))
            if format != "csv":
                with open(os.path.join(dest, "vocab.stanford.txt"), "w", encoding="utf8") as f:
                    f.writelines("%s %d\n" % (t, c) for t, c in zip(df_vocab["token"], df_vocab["count"].tolist()))
        logger.info("vocab created, size: %s.", df_vocab.shape[0])
        stats.update(pass1_s=time.perf_counter() - t0, distinct_tokens=len(tokens), tokens=n_tokens)

        t1 = time.perf_counter()
        with torch.profiler.record_function("corpus.pass2"):
            V = len(vocab_tokens)
            lines = [t.encode("utf8") for t in vocab_tokens]
            off = np.zeros(V + 1, np.int64)
            np.cumsum([len(t) + 1 for t in lines], out=off[1:])
            vb = torch.frombuffer(bytearray(b"".join(t + b"\n" for t in lines)), dtype=torch.uint8).to(d.dev)
            voff = torch.from_numpy(off).to(d.dev)
            slots = lib.glove_vocab_slots(V)
            table = torch.empty(slots, dtype=torch.int32, device=d.dev)
            check(lib.glove_vocab_build(table.data_ptr(), slots, vb.data_ptr(), voff.data_ptr(), V, st), "glove_vocab_build")
            vocab_count = torch.from_numpy(np.array(df_vocab["count"], np.int64)).to(d.dev)
            total = int(df_vocab["count"].sum())
            block = int(max(1, min(chunk_positions, (1 << 28) // ctx)))
            part_bits = _part_bits(V, n_tokens, ctx, int(partition_entries), diagonal=stanford)
            pairs = _Pairs(d, V, part_bits, order_key,
                           (ctx, bool(distance_weighting), bool(symmetric)) if stanford else None)
            stream = _StanfordStream(d, (table, slots, vb, voff)) if stanford else None
            cws = d.empty(lib.glove_cooc_workspace_bytes(block * ctx), torch.uint8)
            got = ctypes.c_int64()
            # ids (Stanford: (segment << 32) | id) whose right context lies in the next chunk
            tail = torch.empty(0, dtype=torch.int64 if stanford else torch.int32, device=d.dev)
            for text, fill, host_text, origin, final in _chunk_loop(d, corpus, chunk_bytes):
                starts, lens, n = _scan(d, corpus, text, fill, host_text, origin)
                ids = tail
                if stanford:
                    new = stream.ids(text, fill, host_text, origin, starts, lens, n)
                    if new.numel():
                        ids = torch.cat([tail, new])
                elif n:
                    ids = torch.empty(tail.numel() + n, dtype=torch.int32, device=d.dev)
                    ids[:tail.numel()].copy_(tail)
                    check(lib.glove_tokens_lookup(text.data_ptr(), starts.data_ptr(), lens.data_ptr(), n, table.data_ptr(), slots,
                                                  vb.data_ptr(), voff.data_ptr(), ids[tail.numel():].data_ptr(), st),
                          "glove_tokens_lookup")
                T = ids.numel()
                n_pos = T if final else max(T - ctx, 0)   # a position counts in the chunk that holds its whole window
                for p0 in range(0, n_pos, block):
                    n_p = min(block, n_pos - p0)
                    n_t = min(n_p + ctx, T - p0)
                    cap = n_p * ctx
                    k, a = d.empty(cap, torch.int64), d.empty(2 * cap, torch.int64)
                    if stanford:
                        check(lib.glove_cooc_chunk_stanford(ids[p0:].data_ptr(), n_p, n_t, V, ctx, int(distance_weighting),
                                                            cws.data_ptr(), cws.numel(), k.data_ptr(), a.data_ptr(), cap,
                                                            ctypes.byref(got), st), "glove_cooc_chunk_stanford")
                    else:
                        check(lib.glove_cooc_chunk(ids[p0:].data_ptr(), n_p, n_t, V, ctx, cws.data_ptr(), cws.numel(),
                                                   k.data_ptr(), a.data_ptr(), cap, ctypes.byref(got), st), "glove_cooc_chunk")
                    if got.value:
                        pairs.add(k, a, got.value)
                    del k, a
                tail = ids[n_pos:].clone()
            del cws
        stats.update(pass2_s=time.perf_counter() - t1, partitions=1 << part_bits, directed_pairs=int(sum(pairs.n)))

        t2 = time.perf_counter()
        with torch.profiler.record_function("corpus.write"):
            n_records = 0
            with contextlib.ExitStack() as files:
                writers = []
                if format != "stanford" and not stanford:
                    writers.append(_CsvWriter(d, files.enter_context(open(os.path.join(dest, "interaction.csv"), "wb")),
                                              vocab_tokens))
                    files.callback(writers[-1].close)
                if format != "csv" or stanford:
                    writers.append(_BinWriter(d, files.enter_context(open(os.path.join(dest, "cooccurrence.shuf.bin"), "wb"))))
                    files.callback(writers[-1].close)
                for p in range(1 << part_bits):
                    if pairs.n[p] == 0:
                        continue
                    cols = pairs.finish(p, vocab_count, total, ctx)
                    n_records += len(cols[0])
                    for w in writers:
                        w.write(cols, int(records_per_block))
                    del cols
        stats.update(write_s=time.perf_counter() - t2, records=n_records,
                     **{"csv_bytes" if isinstance(w, _CsvWriter) else "bin_bytes": w.bytes for w in writers})
    logger.info("interaction records: %d.", n_records)
    return df_vocab, n_records


def main(argv=None):
    logging.basicConfig(level=logging.INFO, format="%(asctime)s - %(levelname)s - %(name)s - %(message)s")
    ap = ArgumentParser(description="Prepare vocab.csv, vocab.txt and interaction.csv from a corpus file of any size.")
    ap.add_argument("--corpus", required=True, help="corpus text file (UTF-8, tokens separated by whitespace)")
    ap.add_argument("--dest", required=True, help="output directory")
    ap.add_argument("--vocab-size", type=int, default=VOCAB_SIZE, help="maximum size of vocab (default: %(default)s)")
    ap.add_argument("--coverage", type=float, default=COVERAGE, help="token coverage to set token count cutoff (default: %(default)s)")
    ap.add_argument("--context-size", type=int, default=CONTEXT_SIZE, help="size of context window (default: %(default)s)")
    ap.add_argument("--format", default="csv", choices=FORMATS,
                    help="csv: interaction.csv; stanford: Stanford GloVe's cooccurrence.shuf.bin and vocab.stanford.txt "
                         "instead; both: all three (default: %(default)s)")
    ap.add_argument("--scheme", default="reference", choices=SCHEMES,
                    help="reference: the counting rules of text8.process_data and the files above; stanford: those of "
                         "Stanford GloVe's vocab_count and cooccur, written as vocab.txt and cooccurrence.shuf.bin "
                         "(default: %(default)s)")
    ap.add_argument("--window-size", type=int, default=15,
                    help="stanford: words of context on each side, 1..%d (default: %%(default)s)" % STANFORD_MAX_WINDOW)
    ap.add_argument("--min-count", type=int, default=1, help="stanford: least count of a vocabulary word (default: %(default)s)")
    ap.add_argument("--max-vocab", type=int, default=0, help="stanford: largest vocabulary, 0 for no limit (default: %(default)s)")
    ap.add_argument("--asymmetric", action="store_true", help="stanford: left context only (cooccur -symmetric 0)")
    ap.add_argument("--no-distance-weighting", action="store_true",
                    help="stanford: every pair counts 1 instead of 1/distance (cooccur -distance-weighting 0)")
    ap.add_argument("--device", default="cuda:0")
    args = ap.parse_args(argv)
    logger.info("call: %s.", " ".join(sys.argv))
    preprocess(args.corpus, args.dest, args.vocab_size, args.coverage, args.context_size, args.device, format=args.format,
               scheme=args.scheme, window_size=args.window_size, min_count=args.min_count, max_vocab=args.max_vocab,
               symmetric=not args.asymmetric, distance_weighting=not args.no_distance_weighting)


if __name__ == "__main__":
    main()
