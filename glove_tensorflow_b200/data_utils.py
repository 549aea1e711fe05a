"""Input side of the drop-in: interaction.csv + vocab.txt -> device-resident COO arrays.

Replaces ``get_csv_input_fn`` (tf.data ``make_csv_dataset`` with select_columns, ref src/models/data_utils.py:4-26) and
the per-step ``StaticHashTable`` string->id lookup (ref src/models/model_utils.py:121-127, src/models/estimator.py:26-28):
the csv bytes are streamed to the GPU in chunks and parsed ONCE by the CUDA ingest kernels (csrc/glove_ingest.cu: record
index, field split, token -> vocab line number with default 0, decimal text -> float32), and the result is the
device-resident COO triple buffer the trainer shuffles and batches from.  A binary sidecar (<csv>.coo.npz) caches the
parse.  The host only reads the header record and moves bytes."""
import ctypes
import os
import re

import numpy as np


def read_vocab(vocab_txt):
    """One token per line, line number = id, no trailing newline (ref src/data/text8.py:149-150)."""
    with open(vocab_txt, encoding="utf8") as f:
        lines = f.read().split("\n")
    if lines and lines[-1] == "":     # a file that ends with a newline has V lines, not V + 1 (TextLineDataset / file_lines)
        lines.pop()
    return lines


def file_lines(fname):
    """ref src/models/utils.py:4-9 (counts iterated lines; a missing trailing newline still counts the last line)."""
    i = -1
    with open(fname, encoding="utf8") as f:
        for i, _ in enumerate(f):
            pass
    return i + 1


def vocab_blob(vocab_txt):
    """vocab.txt as the ingest kernels want it: every line followed by one '\\n', plus the n+1 line offsets."""
    with open(vocab_txt, "rb") as f:
        lines = f.read().split(b"\n")
    if lines and lines[-1] == b"":    # trailing newline: not an (empty) extra token -- n_vocab must equal file_lines()
        lines.pop()
    blob = b"".join(t + b"\n" for t in lines)
    off = np.zeros(len(lines) + 1, np.int64)
    np.cumsum([len(t) + 1 for t in lines], out=off[1:])
    return blob, off


def read_header(train_csv, limit=1 << 20):
    """Column names of the header record and the byte offset of the first data record."""
    import csv
    import io
    with open(train_csv, "rb") as f:
        head = f.read(limit)
    quoted, end = False, None
    for i, b in enumerate(head):
        if b == 0x22:
            quoted = not quoted
        elif b == 0x0A and not quoted:
            end = i
            break
    if end is None:
        if len(head) == limit:
            raise ValueError("%s: no header record in the first %d bytes" % (train_csv, limit))
        end = len(head)
    line = head[:end].rstrip(b"\r").decode("utf8")
    names = next(csv.reader(io.StringIO(line, newline="")))
    return names, min(end + 1, len(head))


def read_sample_records(train_csv, offset, n=100, limit=1 << 20):
    """The first ``n`` data records (lists of fields) after byte ``offset`` -- what make_csv_dataset's
    num_rows_for_inference=100 looks at to decide a column's dtype [ref src/models/data_utils.py:19]."""
    import csv
    import io
    with open(train_csv, "rb") as f:
        f.seek(offset)
        text = f.read(limit).decode("utf8", errors="replace")
    out = []
    try:
        for rec in csv.reader(io.StringIO(text, newline="")):
            if rec:
                out.append(rec)
            if len(out) > n:
                break
    except csv.Error:
        pass
    return out[:n] if len(out) > n or len(text) < limit else out[:-1]   # a record cut by the read limit is dropped


def _int_like(field):
    import re
    return re.fullmatch(r"[+-]?[0-9]+", field.strip()) is not None


def make_schema(names, row_name, col_name, value_names, sample=None):
    """Column positions and kinds.  A key column (row / col) is a TOKEN column -- resolved through vocab.txt like the
    reference's string_id_table.lookup [ref src/models/estimator.py:27-28] -- unless its values are integers, in which case
    they are taken as ids directly.  Like make_csv_dataset the kind is inferred from the data (``sample`` = the first
    records, see read_sample_records): a string column called 'user_id' is still a token column.  Without a sample the
    name decides ('*_id' = integer ids)."""
    from . import _lib
    sc = _lib.CsvSchema()
    sc.n_cols = len(names)
    for c, name in enumerate((row_name, col_name) + tuple(value_names)):
        if name not in names:
            raise ValueError("column %r not in the csv header %r" % (name, names))
        sc.column[c] = names.index(name)
        if c >= 2:
            sc.kind[c] = _lib.CSV_FLOAT
        elif sample:
            col = sc.column[c]
            sc.kind[c] = _lib.CSV_INT if all(len(r) > col and _int_like(r[col]) for r in sample) else _lib.CSV_TOKEN
        else:
            sc.kind[c] = _lib.CSV_INT if name.endswith("_id") else _lib.CSV_TOKEN
    return sc


_HEAD = 1 << 20   # room in front of every chunk for the unterminated tail of the previous one


class _ChunkReader:
    """Fills pinned host buffers from the file with a few threads (os.preadv releases the GIL), one chunk ahead of the
    GPU.  Chunk k lands at buf[k % 2][_HEAD : _HEAD + n]."""

    def __init__(self, path, offset, size, chunk, bufs, threads=8, piece=8 << 20):
        from concurrent.futures import ThreadPoolExecutor
        self.fd = os.open(path, os.O_RDONLY)
        self.offset, self.size, self.chunk, self.bufs, self.piece = offset, size, chunk, bufs, piece
        self.pool = ThreadPoolExecutor(max_workers=threads)
        self.pending = {}

    def n_chunks(self):
        return (self.size + self.chunk - 1) // self.chunk

    def _read(self, view, pos):
        done = 0
        while done < len(view):
            got = os.preadv(self.fd, [view[done:]], pos + done)
            if got <= 0:
                raise IOError("short read at byte %d" % (pos + done))
            done += got

    def start(self, k):
        if k >= self.n_chunks():
            return
        lo = k * self.chunk
        n = min(self.chunk, self.size - lo)
        view = memoryview(self.bufs[k % 2])[_HEAD:_HEAD + n]
        self.pending[k] = (n, [self.pool.submit(self._read, view[o:min(o + self.piece, n)], self.offset + lo + o)
                               for o in range(0, n, self.piece)])

    def wait(self, k):
        n, futs = self.pending.pop(k)
        for f in futs:
            f.result()
        return n

    def close(self):
        self.pool.shutdown(wait=True)
        os.close(self.fd)


def ingest_csv(train_csv, vocab_txt, row_name="row_token", col_name="col_token",
               value_names=("glove_value", "glove_weight"), device="cuda:0", chunk_bytes=64 << 20):
    """Streams the file through the CUDA ingest kernels.  Returns device tensors
    {'row': i32[n], 'col': i32[n], <value_name>: f32[n] ...} in file order.

    Host side: reader threads fill pinned chunk k+1 while the GPU indexes and parses chunk k; the unterminated tail of a
    chunk is copied in front of the next one (padded to 16-byte alignment with '\n', which the indexer skips as blank
    lines)."""
    import torch
    from . import _lib
    lib, check = _lib.lib, _lib.check
    if len(value_names) != 2:
        raise ValueError("exactly two value columns are read (target, weight) / (pos, neg)")
    dev = torch.device(device)
    names, data_off = read_header(train_csv)
    schema = make_schema(names, row_name, col_name, value_names, sample=read_sample_records(train_csv, data_off))
    size = os.path.getsize(train_csv) - data_off
    parts = {k: [] for k in ("row", "col", "a", "b")}
    with torch.cuda.device(dev):
        st = torch.cuda.current_stream().cuda_stream
        blob, off = vocab_blob(vocab_txt)
        n_vocab = len(off) - 1
        vb = torch.frombuffer(bytearray(blob), dtype=torch.uint8).to(dev)
        voff = torch.from_numpy(off).to(dev)
        slots = lib.glove_vocab_slots(n_vocab)
        table = torch.empty(slots, dtype=torch.int32, device=dev)
        check(lib.glove_vocab_build(table.data_ptr(), slots, vb.data_ptr(), voff.data_ptr(), n_vocab, st), "glove_vocab_build")
        chunk = int(max(1 << 16, min(chunk_bytes, size))) // 16 * 16
        pinned = [torch.empty(_HEAD + chunk, dtype=torch.uint8, pin_memory=True) for _ in range(2 if size > chunk else 1)]
        host = [t.numpy() for t in pinned]
        text = torch.empty(_HEAD + chunk, dtype=torch.uint8, device=dev)
        ws = torch.empty(lib.glove_csv_workspace_bytes(_HEAD + chunk), dtype=torch.uint8, device=dev)
        reader = _ChunkReader(train_csv, data_off, max(size, 0), chunk, host * (2 // len(host)))
        try:
            n_chunks, carry, n_total = reader.n_chunks(), 0, 0
            reader.start(0)
            for k in range(n_chunks):
                n_new = reader.wait(k)
                reader.start(k + 1)
                final = k == n_chunks - 1
                begin = (_HEAD - carry) // 16 * 16
                host[k % 2][begin:_HEAD - carry] = 0x0A
                fill = _HEAD + n_new - begin
                text[:fill].copy_(pinned[k % 2][begin:_HEAD + n_new], non_blocking=True)
                n_rec = ctypes.c_int64()
                check(lib.glove_csv_index(text.data_ptr(), fill, ws.data_ptr(), ws.numel(), ctypes.byref(n_rec), st), "glove_csv_index")
                cap = n_rec.value + 1
                ends = torch.empty(cap, dtype=torch.int64, device=dev)
                row = torch.empty(cap, dtype=torch.int32, device=dev)
                col = torch.empty(cap, dtype=torch.int32, device=dev)
                a = torch.empty(cap, dtype=torch.float32, device=dev)
                b = torch.empty(cap, dtype=torch.float32, device=dev)
                n_rows, consumed = ctypes.c_int64(), ctypes.c_int64()
                check(lib.glove_csv_parse(text.data_ptr(), fill, int(final), ws.data_ptr(), ws.numel(), ctypes.byref(schema),
                                          table.data_ptr(), slots, vb.data_ptr(), voff.data_ptr(), n_vocab, ends.data_ptr(),
                                          row.data_ptr(), col.data_ptr(), a.data_ptr(), b.data_ptr(), cap, n_total,
                                          ctypes.byref(n_rows), ctypes.byref(consumed), st), "glove_csv_parse")
                n = n_rows.value
                for key, t in (("row", row), ("col", col), ("a", a), ("b", b)):
                    parts[key].append(t[:n])
                n_total += n
                carry = fill - consumed.value
                if carry > _HEAD - 16:
                    raise ValueError("%s: a record is longer than %d bytes" % (train_csv, _HEAD - 16))
                if carry:   # the tail goes in front of the next chunk (which is being read into the other buffer)
                    host[(k + 1) % 2][_HEAD - carry:_HEAD] = host[k % 2][begin + consumed.value:begin + fill]
        finally:
            reader.close()
        empty = {"row": torch.int32, "col": torch.int32, "a": torch.float32, "b": torch.float32}
        cat = {k: (torch.cat(v) if len(v) > 1 else v[0]) if v else torch.empty(0, dtype=empty[k], device=dev)
               for k, v in parts.items()}
    return {"row": cat["row"], "col": cat["col"], value_names[0]: cat["a"], value_names[1]: cat["b"]}


def load_interaction_csv(train_csv, vocab_txt, row_name="row_token", col_name="col_token",
                         value_names=("glove_value", "glove_weight"), cache=True, device="cuda:0"):
    """Returns {'row': i32[n], 'col': i32[n], <value_name>: f32[n] ...} in file order (numpy, from the sidecar cache when
    it is current, else parsed on the GPU by ``ingest_csv``).

    ``row_name`` / ``col_name`` may name string columns (resolved through vocab.txt, missing -> 0) or integer id columns
    (``row_token_id``: equal by construction, SURVEY A2).  Tokens like 'na' / 'null' / 'nan' are ordinary vocabulary
    words (ref README.md:54)."""
    # the cached ids were resolved through THIS vocab.txt: its size and mtime are part of the key (an edited or different
    # vocabulary with the same csv must not reuse them)
    vst = os.stat(vocab_txt)
    n_vocab = file_lines(vocab_txt)
    key = "|".join([row_name, col_name] + list(value_names) + ["vocab:%d:%d:%d" % (n_vocab, vst.st_size, vst.st_mtime_ns)])
    side = train_csv + ".coo.npz"
    out = None
    if cache and os.path.exists(side) and os.path.getmtime(side) >= os.path.getmtime(train_csv):
        try:
            z = np.load(side, allow_pickle=False)
            if str(z["key"]) == key:
                out = {k: z[k] for k in z.files if k != "key"}
        except Exception:   # unreadable sidecar: re-ingest
            out = None
    if out is None:
        out = {k: v.cpu().numpy() for k, v in ingest_csv(train_csv, vocab_txt, row_name, col_name, value_names, device).items()}
        if cache:
            try:
                tmp = side + ".tmp.npz"
                np.savez(tmp, key=np.array(key), **out)
                os.replace(tmp, side)
            except OSError:
                pass
    check_ids(out["row"], out["col"], n_vocab, train_csv)
    return out


COOC_RECORD = 16    # Stanford GloVe co-occurrence record: int32 word1, int32 word2, float64 val (little-endian, packed)
_STANFORD_LINE = re.compile(r"(\S+) ([0-9]+)")


def read_stanford_vocab(vocab_txt):
    """(tokens, counts) of a vocabulary file.  A file whose first line is ``word count`` (Stanford GloVe's vocab.txt, as
    vocab_count writes it) must have that form on every line; ``counts`` is then an int64 array.  Any other file is one
    token per line (``read_vocab``) and ``counts`` is None."""
    lines = read_vocab(vocab_txt)
    if not lines or _STANFORD_LINE.fullmatch(lines[0]) is None:
        return lines, None
    tokens, counts = [], []
    for i, line in enumerate(lines):
        m = _STANFORD_LINE.fullmatch(line)
        if m is None:
            raise ValueError("%s: line %d is not 'word count' like line 1: %r" % (vocab_txt, i + 1, line[:80]))
        tokens.append(m.group(1))
        counts.append(int(m.group(2)))
    return tokens, np.array(counts, np.int64)


def _bad_record(path, host_rec, g, kind, V):
    from . import _lib
    rec = np.frombuffer(host_rec, np.dtype([("w1", "<i4"), ("w2", "<i4"), ("val", "<f8")]))[0]
    what = {_lib.CREC_BAD_WORD1: "word1 id %d outside 1..%d" % (rec["w1"], V),
            _lib.CREC_BAD_WORD2: "word2 id %d outside 1..%d" % (rec["w2"], V),
            _lib.CREC_BAD_VALUE: "val %r is not a finite value > 0" % float(rec["val"])}[kind]
    return ValueError("%s: record %d (byte %d): %s" % (path, g + 1, g * COOC_RECORD, what))


def load_cooc_bin(path, vocab_size, x_max=100.0, alpha=0.75, device="cuda:0", chunk_bytes=64 << 20):
    """A Stanford GloVe co-occurrence file (cooccurrence.bin or cooccurrence.shuf.bin) as device tensors
    {'row': i32[n], 'col': i32[n], 'glove_value': f32[n], 'glove_weight': f32[n]} in file order: ids - 1,
    log(val) and the weight of Stanford's glove.c, ``val >= x_max ? 1 : (val / x_max) ** alpha``, both computed in
    float64 and rounded once to float32 (csrc/glove_crec.cu).

    The COO is allocated once (the record count follows from the file size) and the chunks, whole records each, are
    parsed straight into it while reader threads fill the other pinned buffer.  An id outside 1..vocab_size, a val that
    is not finite and > 0, or a file cut inside a record fails, naming the lowest offending 1-based record and its byte
    offset."""
    import torch
    from . import _lib
    V = _check_vocab_size(vocab_size)
    n = os.path.getsize(path) // COOC_RECORD
    dev = torch.device(device)
    with torch.cuda.device(dev):
        out = {"row": torch.empty(n, dtype=torch.int32, device=dev), "col": torch.empty(n, dtype=torch.int32, device=dev),
               "glove_value": torch.empty(n, dtype=torch.float32, device=dev),
               "glove_weight": torch.empty(n, dtype=torch.float32, device=dev)}

    def parse(raw, m, first, err, st):
        _lib.check(_lib.lib.glove_cooc_bin_parse(raw, m, first, V, float(x_max), float(alpha),
                                                 *[out[c][first:].data_ptr() for c in ("row", "col", "glove_value",
                                                                                       "glove_weight")],
                                                 err, st), "glove_cooc_bin_parse")

    stream_cooc_bin(path, V, parse, dev, chunk_bytes)
    return out


def _check_vocab_size(vocab_size):
    V = int(vocab_size)
    if not 1 <= V < (1 << 31):
        raise ValueError("vocab_size must be 1 .. 2^31-1, got %d" % V)
    return V


def stream_cooc_bin(path, V, parse, dev, chunk_bytes=64 << 20):
    """Streams the whole records of a Stanford co-occurrence file to the device in chunks and calls
    ``parse(raw_ptr, m, first, error_ptr, stream)`` on each (m records, the first with the 0-based index ``first``), which
    launches a parser that lowers the error word as glove_cooc_bin_parse does.  Raises on the lowest bad record and on a
    file cut inside a record."""
    import torch
    size = os.path.getsize(path)
    n = size // COOC_RECORD
    with torch.cuda.device(dev):
        if n:
            st = torch.cuda.current_stream().cuda_stream
            whole = n * COOC_RECORD
            chunk = int(max(COOC_RECORD, min(chunk_bytes, whole))) // COOC_RECORD * COOC_RECORD
            pinned = [torch.empty(_HEAD + chunk, dtype=torch.uint8, pin_memory=True) for _ in range(2 if whole > chunk else 1)]
            host = [t.numpy() for t in pinned]
            raw = torch.empty(chunk, dtype=torch.uint8, device=dev)
            err = torch.full((1,), -1, dtype=torch.int64, device=dev)      # all ones: no bad record
            reader = _ChunkReader(path, 0, whole, chunk, host * (2 // len(host)))
            try:
                reader.start(0)
                for k in range(reader.n_chunks()):
                    nb = reader.wait(k)
                    reader.start(k + 1)
                    m, first = nb // COOC_RECORD, k * (chunk // COOC_RECORD)
                    raw[:nb].copy_(pinned[k % len(pinned)][_HEAD:_HEAD + nb], non_blocking=True)
                    parse(raw.data_ptr(), m, first, err.data_ptr(), st)
                    code = int(err.item()) & 0xFFFFFFFFFFFFFFFF       # synchronises: pinned[k % 2] may be refilled after this
                    if code != 0xFFFFFFFFFFFFFFFF:
                        g = code >> 2
                        o = _HEAD + (g - first) * COOC_RECORD
                        raise _bad_record(path, host[k % len(host)][o:o + COOC_RECORD].tobytes(), g, code & 3, V)
            finally:
                reader.close()
    if size % COOC_RECORD:
        raise ValueError("%s: record %d (byte %d): the file ends %d bytes into a %d-byte record (truncated file)"
                         % (path, n + 1, n * COOC_RECORD, size % COOC_RECORD, COOC_RECORD))


def check_ids(row, col, n_vocab, what="COO"):
    """0 <= id < V for every triple: nothing downstream bounds-checks ids (they index the packed tables and are packed
    into vbits-wide sort keys), so a violation is refused here, once."""
    for name, a in (("row", row), ("col", col)):
        if len(a) == 0:
            continue
        lo, hi = int(a.min()), int(a.max())
        if lo < 0 or hi >= n_vocab:
            raise ValueError("%s: %s id out of range [0, %d): min %d, max %d" % (what, name, n_vocab, lo, hi))
