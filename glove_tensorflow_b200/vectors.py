"""Word vectors in the GloVe text format, read and written on the GPU.

The format (``word v_1 ... v_d`` per line, optionally after a word2vec header ``V d``) is what Stanford's GloVe trainer
writes, what the published vectors (glove.6B, glove.840B, ...) are distributed in and what gensim's
``save_word2vec_format`` writes.  Parsing and printing the text runs in the CUDA kernels of csrc/glove_vectors.cu; the
host reads the first line (header and d), moves bytes and slices the words.

Reading: fields are separated by runs of ASCII space or tab, trailing blanks and a ``\\r`` before the ``\\n`` are ignored,
blank lines are skipped.  The LAST d fields are the numbers and the word is everything before them (``rsplit``: words may
contain spaces, like glove.840B's, or look like numbers, like ``nan``).  Numbers are rounded once to float32; nan / inf
are refused.  Errors name the lowest offending 1-based line of the file.  Words come back as str decoded from UTF-8 with
``errors="surrogateescape"``, so their bytes survive a round trip; duplicate words keep their own rows.

Writing: every value is printed as the shortest decimal that parses back to the same float32, so export -> import is
bit-exact."""
import ctypes
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from .data_utils import _HEAD, _ChunkReader

MAX_DIM = 510   # the engine's limit (glove_table_stride(d) / 4 <= 128)


def _content(line: bytes) -> bytes:
    if line.endswith(b"\r"):
        line = line[:-1]
    return line.rstrip(b" \t")


def _fields(s: bytes):
    return s.replace(b"\t", b" ").split()


def read_header(path, dim=None, limit=_HEAD):
    """(V or None, d, byte offset of the line after the header, 1-based number of that line).  A first line of exactly
    two unsigned decimal integers is a word2vec header ``V d``; otherwise d = fields of the first vector line - 1, unless
    ``dim`` is given."""
    with open(path, "rb") as f:
        head = f.read(limit)
    nl = head.find(b"\n")
    first = head if nl < 0 else head[:nl]
    f0 = _fields(_content(first))
    V, offset, line0, where = None, 0, 1, 1
    if len(f0) == 2 and all(x.isdigit() for x in f0):
        V, d_h = int(f0[0]), int(f0[1])
        if dim is not None and int(dim) != d_h:
            raise ValueError("%s: line 1: the header declares d = %d, not %d" % (path, d_h, dim))
        dim, offset, line0 = d_h, (len(head) if nl < 0 else nl + 1), 2
    elif dim is None:
        lines = head.split(b"\n")
        if len(head) == limit:
            lines.pop()                       # may be cut by the read limit
        for no, line in enumerate(lines, 1):
            s = _content(line)
            if s:
                dim, where = len(_fields(s)) - 1, no
                break
        else:
            raise ValueError("%s: no vector line in the first %d bytes" % (path, len(head)))
    dim = int(dim)
    if not 2 <= dim <= MAX_DIM:
        raise ValueError("%s: line %d: d = %d is outside [2, %d]" % (path, where, dim, MAX_DIM))
    return V, dim, offset, line0


def read_vectors(path, dim=None, device="cuda:0", out=None, chunk_bytes=64 << 20):
    """Parses a GloVe / word2vec text file on the GPU.  Returns ``(words, rows)``: a list of str in file order and a
    device float32 tensor [V, d].  ``out``: a 2-D float32 device tensor of at least V rows and d columns with unit column
    stride (a packed one-plane table, rows of glove_table_stride(d) floats, is filled in place); ``rows`` is then
    ``out[:V]``.  Raises ValueError naming the lowest offending line of a malformed file."""
    import torch
    from . import _lib
    lib = _lib.lib
    V, d, data_off, line_no = read_header(path, dim)
    size = os.path.getsize(path) - data_off
    dev = torch.device(device) if out is None else out.device
    if out is not None:
        if out.dim() != 2 or out.dtype != torch.float32 or out.stride(1) != 1 or out.shape[1] < d or not out.is_cuda:
            raise ValueError("read_vectors: out must be a 2-D float32 device tensor with >= %d unit-stride columns" % d)
        if V is not None and out.shape[0] < V:
            raise ValueError("read_vectors: out holds %d rows, the header declares %d" % (out.shape[0], V))
    elif V is not None:
        out = torch.empty(V, d, dtype=torch.float32, device=dev)
    capacity = (V if V is not None else out.shape[0]) if out is not None else None
    words, parts, n_rows = [], [], 0
    with torch.cuda.device(dev):
        st = torch.cuda.current_stream().cuda_stream
        chunk = int(max(64, min(chunk_bytes, max(size, 1)))) // 16 * 16
        pinned = [torch.empty(_HEAD + chunk, dtype=torch.uint8, pin_memory=True) for _ in range(2 if size > chunk else 1)]
        host = [t.numpy() for t in pinned]
        text = torch.empty(_HEAD + chunk, dtype=torch.uint8, device=dev)
        ws = torch.empty(0, dtype=torch.uint8, device=dev)
        reader = _ChunkReader(path, data_off, max(size, 0), chunk, host * (2 // len(host)))
        try:
            n_chunks, carry = reader.n_chunks(), 0
            reader.start(0)
            for k in range(n_chunks):
                n_new = reader.wait(k)
                reader.start(k + 1)
                final = k == n_chunks - 1
                # the carried tail sits right before the new bytes; the 16-byte aligned start is padded with '\n' (blank lines)
                begin = (_HEAD - carry) // 16 * 16
                pad = _HEAD - carry - begin
                host[k % 2][begin:_HEAD - carry] = 0x0A
                fill = _HEAD + n_new - begin
                text[:fill].copy_(pinned[k % 2][begin:_HEAD + n_new], non_blocking=True)
                need = lib.glove_vectors_workspace_bytes(fill, 0)
                if ws.numel() < need:
                    ws = torch.empty(need, dtype=torch.uint8, device=dev)
                n_nl = ctypes.c_int64()
                _check(lib.glove_vectors_index(text.data_ptr(), fill, ws.data_ptr(), ws.numel(), ctypes.byref(n_nl), st), path)
                n_lines = n_nl.value
                need = lib.glove_vectors_workspace_bytes(fill, n_lines + 1)
                if ws.numel() < need:   # a larger workspace keeps the index pass's prefix: copy it over
                    bigger = torch.empty(need, dtype=torch.uint8, device=dev)
                    bigger[:ws.numel()].copy_(ws)
                    ws = bigger
                if out is not None:
                    dst, ld, cap = out.data_ptr() + 4 * n_rows * out.stride(0), out.stride(0), capacity - n_rows
                else:
                    part = torch.empty(n_lines + 1, d, dtype=torch.float32, device=dev)
                    dst, ld, cap = part.data_ptr(), d, n_lines + 1
                wstart = torch.empty(n_lines + 1, dtype=torch.int64, device=dev)
                wlen = torch.empty(n_lines + 1, dtype=torch.int32, device=dev)
                n, consumed = ctypes.c_int64(), ctypes.c_int64()
                _check(lib.glove_vectors_parse(text.data_ptr(), fill, int(final), d, n_lines, ws.data_ptr(), ws.numel(), dst, ld,
                                               cap, wstart.data_ptr(), wlen.data_ptr(), line_no - pad, ctypes.byref(n),
                                               ctypes.byref(consumed), st), path)
                n = n.value
                if out is None:
                    parts.append(part[:n])
                if n:
                    blob = host[k % 2][begin:begin + consumed.value].tobytes()
                    for s, m in zip(wstart[:n].cpu().numpy().tolist(), wlen[:n].cpu().numpy().tolist()):
                        words.append(blob[s:s + m].decode("utf8", "surrogateescape"))
                n_rows += n
                line_no += n_lines - pad
                carry = fill - consumed.value
                if carry > _HEAD - 16:
                    raise ValueError("%s: line %d is longer than %d bytes" % (path, line_no, _HEAD - 16))
                if carry:   # the tail goes in front of the next chunk (which is being read into the other buffer)
                    host[(k + 1) % 2][_HEAD - carry:_HEAD] = host[k % 2][begin + consumed.value:begin + fill]
        finally:
            reader.close()
        if size > 0:
            with open(path, "rb") as f:
                f.seek(-1, os.SEEK_END)
                if f.read(1) != b"\n":
                    line_no += 1            # the unterminated last line
        if V is not None and n_rows != V:
            raise ValueError("%s: line %d: the header declares %d vectors, the file holds %d" % (path, line_no, V, n_rows))
        if out is not None:
            rows = out[:n_rows]
        elif parts:
            rows = torch.cat(parts) if len(parts) > 1 else parts[0]
        else:
            rows = torch.empty(0, d, dtype=torch.float32, device=dev)
    return words, rows


def _check(rc, path):
    from . import _lib
    if rc != _lib.OK:
        msg = _lib.lib.glove_last_error()
        msg = msg.decode() if msg else "error %d" % rc
        if rc == _lib.EINVAL and msg.startswith("vectors file: "):
            raise ValueError("%s: %s" % (path, msg[len("vectors file: "):]))
        raise _lib.GloveError("%s: %s" % (path, msg))


def word_bytes(word) -> bytes:
    """The bytes a word is written as (str: UTF-8 with surrogateescape, the inverse of the reader's decoding)."""
    return word if isinstance(word, bytes) else word.encode("utf8", "surrogateescape")


def write_vectors(path, words, rows, header=False, rows_per_chunk=1 << 16):
    """Writes ``rows`` (float32 [V, d], a device tensor with unit column stride, or anything numpy can convert) with their
    ``words`` as a GloVe text file, one ``word v_1 ... v_d`` line per row in order; ``header`` adds the word2vec first line
    ``V d``.  The text is formatted on the GPU, ``rows_per_chunk`` rows at a time, copied back to pinned memory and
    written by a thread while the next block is formatted."""
    import torch
    from . import _lib
    lib = _lib.lib
    if not isinstance(rows, torch.Tensor) or not rows.is_cuda:
        rows = torch.as_tensor(np.ascontiguousarray(rows, np.float32)).to("cuda")
    if rows.dim() != 2 or rows.dtype != torch.float32 or rows.stride(1) != 1:
        raise ValueError("write_vectors: rows must be a 2-D float32 tensor with unit column stride")
    V, d = rows.shape
    if not 2 <= d <= MAX_DIM:
        raise ValueError("write_vectors: d = %d is outside [2, %d]" % (d, MAX_DIM))
    enc = [word_bytes(w) for w in words]
    if len(enc) != V:
        raise ValueError("write_vectors: %d words for %d rows" % (len(enc), V))
    for i, w in enumerate(enc):   # a word the reader would not give back
        if not w or b"\n" in w or w[-1:] in (b" ", b"\t"):
            raise ValueError("write_vectors: word %d (%r) is empty, holds a newline or ends with a blank" % (i, w))
    dev = rows.device
    with torch.cuda.device(dev), open(path, "wb") as f:
        if header:
            f.write(b"%d %d\n" % (V, d))
        if V == 0:
            return path
        st = torch.cuda.current_stream().cuda_stream
        off = np.zeros(V + 1, np.int64)
        np.cumsum([len(w) for w in enc], out=off[1:])
        blob = torch.frombuffer(bytearray(b"".join(enc) or b"\0"), dtype=torch.uint8).to(dev)
        woff = torch.from_numpy(off).to(dev)
        step = min(int(rows_per_chunk), V)
        ws = torch.empty(lib.glove_vectors_workspace_bytes(0, step), dtype=torch.uint8, device=dev)
        text = torch.empty(0, dtype=torch.uint8, device=dev)
        pinned, pending = [None, None], [None, None]
        pool = ThreadPoolExecutor(max_workers=1)
        ld = rows.stride(0)

        def write(buf, nbytes, ev):
            ev.synchronize()
            f.write(buf.numpy()[:nbytes].data)

        try:
            for k, r0 in enumerate(range(0, V, step)):
                n = min(step, V - r0)
                rp, op = rows.data_ptr() + 4 * r0 * ld, woff.data_ptr() + 8 * r0
                nbytes = ctypes.c_int64()
                _check(lib.glove_vectors_format_size(rp, ld, d, n, op, ws.data_ptr(), ws.numel(), ctypes.byref(nbytes), st),
                       path)
                nbytes = nbytes.value
                if text.numel() < nbytes:
                    text = torch.empty(nbytes, dtype=torch.uint8, device=dev)
                _check(lib.glove_vectors_format(rp, ld, d, n, blob.data_ptr(), op, ws.data_ptr(), ws.numel(), text.data_ptr(),
                                                text.numel(), st), path)
                s = k % 2
                if pending[s] is not None:
                    pending[s].result()           # the writer is done with this pinned buffer
                if pinned[s] is None or pinned[s].numel() < nbytes:
                    pinned[s] = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
                pinned[s][:nbytes].copy_(text[:nbytes], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record()
                pending[s] = pool.submit(write, pinned[s], nbytes, ev)
            for p in pending:
                if p is not None:
                    p.result()
        finally:
            pool.shutdown(wait=True)
    return path


def vectors_engine(path, dim=None, device="cuda:0", chunk_bytes=64 << 20):
    """An evaluation-only GloveEngine (one-plane SGD tables) whose row table holds the vectors of a text file, parsed
    on the device straight into the table (a file with a word2vec header) or into a [V, d] tensor that is then copied
    into it (without one, V is known only at the end).  Returns ``(engine, words)``."""
    from .engine import GloveEngine
    V, d, _, _ = read_header(path, dim)

    def engine(n):
        if n < 1:
            raise ValueError("%s holds no vectors" % path)
        return GloveEngine(n, d, optimizer="SGD", batch_size=64, plan_steps=1, max_steps=4, device=device)

    if V is not None:
        eng = engine(V)
        words, _ = read_vectors(path, d, out=eng.row_plane(), chunk_bytes=chunk_bytes)
    else:
        words, rows = read_vectors(path, d, device=device, chunk_bytes=chunk_bytes)
        eng = engine(len(words))
        eng.row_plane()[:, :d].copy_(rows)
    return eng, words
