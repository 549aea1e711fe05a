"""TEST INFRASTRUCTURE ONLY -- plain-Python restatement of the GloVe text format of word vectors, the checker for the CUDA
import / export kernels (glove_tensorflow_b200/csrc/glove_vectors.cu, glove_ftoa.cuh).  Nothing in the product path may
import this file.

Reading (``read_vectors``):
  * one vector per line, ``word v_1 ... v_d``; fields are separated by runs of ASCII space or tab; a ``\\r`` before the
    ``\\n`` and trailing blanks are ignored; blank lines are skipped; the last line may lack its ``\\n``;
  * the last d fields are the numbers, the word is everything before them with the separating blanks trimmed (the
    ``rsplit`` rule: words may contain spaces or look like numbers);
  * a first line of exactly two unsigned decimal integers is a word2vec header ``V d``, and exactly V vector lines must
    follow; otherwise d = fields of the first vector line - 1 (unless given); 2 <= d <= 510;
  * numbers are rounded once, decimal -> float32 (csv_oracle.f32_exact); nan / inf are refused;
  * errors name the lowest offending 1-based line of the file (blank lines and the header count).
Writing (``format_f32``, ``format_vectors``): shortest round-trip digits (numpy's Dragon4 "unique" mode), positional for
decimal exponents -5 .. 8, ``d[.ddd]e+XX`` otherwise."""
import re

import numpy as np

from .csv_oracle import f32_exact

MAX_DIM = 510


class VectorsFormatError(ValueError):
    def __init__(self, line, what):
        super().__init__("line %d: %s" % (line, what))
        self.line = line


def _content(line: bytes) -> bytes:
    """The line without its \\r\\n / \\n and trailing blanks."""
    if line.endswith(b"\r"):
        line = line[:-1]
    return line.rstrip(b" \t")


def _fields(s: bytes):
    return s.replace(b"\t", b" ").split()


def number(t: bytes) -> np.float32:
    """f32_exact, with the parser's limit: more than 19 significant digits are refused unless dropping the tail provably
    does not change the rounding (glove_strtof.cuh)."""
    v = f32_exact(t)
    m = re.match(rb"^[+-]?(\d*)(?:\.(\d*))?(?:[eE]([+-]?\d+))?$", t)
    if m and np.isfinite(v):
        ip, fp, ex = m.group(1) or b"", m.group(2) or b"", int(m.group(3) or 0)
        digits = (ip + fp).lstrip(b"0")
        if len(digits) > 19 and digits[19:].strip(b"0"):
            lead = (ip + fp).lstrip(b"0")
            scale = ex - len(fp) + (len(lead) - 19)
            w = int(lead[:19])
            if f32_exact(b"%de%d" % (w, scale)) != f32_exact(b"%de%d" % (w + 1, scale)):
                raise ValueError("more than 19 significant digits and the tail decides the rounding: %r" % t)
    return v


def is_header(line: bytes) -> bool:
    f = _fields(_content(line))
    return len(f) == 2 and all(x.isdigit() for x in f)


def read_vectors(data: bytes, dim=None):
    """bytes of a whole file -> (words: list of bytes, rows: float32 [V, d]); VectorsFormatError on a malformed file."""
    lines = data.split(b"\n")
    if lines and lines[-1] == b"":
        lines.pop()
    first, V, first_vector_line = 0, None, 1
    if lines and is_header(lines[0]):
        V, d_h = (int(x) for x in _fields(_content(lines[0])))
        if dim is not None and dim != d_h:
            raise VectorsFormatError(1, "the header declares d = %d, the caller %d" % (d_h, dim))
        dim, first = d_h, 1
    if dim is None:
        for no in range(len(lines)):
            s = _content(lines[no])
            if s:
                dim, first_vector_line = len(_fields(s)) - 1, no + 1
                break
        else:
            dim = 2                                       # an empty file holds no vectors whatever d is
    if not 2 <= dim <= MAX_DIM:
        raise VectorsFormatError(first_vector_line, "d = %d is outside [2, %d]" % (dim, MAX_DIM))
    words, rows = [], []
    for no in range(first, len(lines)):
        s = _content(lines[no])
        if not s:
            continue
        if V is not None and len(rows) == V:
            raise VectorsFormatError(no + 1, "more vectors than the header's %d" % V)
        # the last d fields, from the right
        end, vals = len(s), []
        for _ in range(dim):
            while end > 0 and s[end - 1] in b" \t":
                end -= 1
            start = end
            while start > 0 and s[start - 1] not in b" \t":
                start -= 1
            if start == end:
                break
            vals.append(s[start:end])
            end = start
        word = s[:end].rstrip(b" \t")
        if len(vals) < dim or not word:
            raise VectorsFormatError(no + 1, "fewer than d + 1 = %d fields" % (dim + 1))
        row = []
        for t in reversed(vals):
            try:
                v = number(t)
            except ValueError:
                raise VectorsFormatError(no + 1, "not a number: %r" % t) from None
            if not np.isfinite(v):
                raise VectorsFormatError(no + 1, "not a finite number: %r" % t)
            row.append(v)
        words.append(word)
        rows.append(row)
    if V is not None and len(rows) != V:
        raise VectorsFormatError(len(lines) + 1, "the header declares %d vectors, the file holds %d" % (V, len(rows)))
    return words, np.asarray(rows, np.float32).reshape(len(rows), dim)


def format_f32(x) -> str:
    """The text the exporter writes for one float32."""
    x = np.float32(x)
    if np.isnan(x):
        return "nan"
    if np.isinf(x):
        return "inf" if x > 0 else "-inf"
    if x == 0:
        return "-0" if np.signbit(x) else "0"
    mant, ex = np.format_float_scientific(x, unique=True, trim="-").split("e")
    E, sign, dg = int(ex), "-" if mant.startswith("-") else "", mant.lstrip("-").replace(".", "")
    if 0 <= E <= 8:
        body = dg[:E + 1].ljust(E + 1, "0") + ("." + dg[E + 1:] if len(dg) > E + 1 else "")
    elif -5 <= E < 0:
        body = "0." + "0" * (-E - 1) + dg
    else:
        body = dg[0] + ("." + dg[1:] if len(dg) > 1 else "") + "e%s%02d" % ("-" if E < 0 else "+", abs(E))
    return sign + body


def format_vectors(words, rows, header=False) -> bytes:
    """words (bytes) and float32 [V, d] -> the exported file."""
    rows = np.asarray(rows, np.float32)
    out = [b"%d %d\n" % rows.shape] if header else []
    for w, r in zip(words, rows):
        out.append(w + b"".join(b" " + format_f32(v).encode() for v in r) + b"\n")
    return b"".join(out)


def handmade_files():
    """name -> bytes: the layouts the format allows (see the module docstring)."""
    return {
        "header": b"3 2\nthe 0.1 -0.2\nnan 1e-3 +4\n1 -0 0\n",
        "header_crlf_blank_lines": b"2 3\r\n\r\nx 1 2 3\r\n   \n\ty 4 5 6  \r\n",
        "no_header_mixed": (b"a\t0.5  1.5 \r\n\n   \n-0 2 3\r\ninf\t-1E+2\t.5\nword with  spaces 1 2\n"
                            b"\xc3\xa9t\xc3\xa9 3 4\n\"quoted\" 7 8\n  lead 9 10\na 5 6"),
        "number_forms": (b"x 1.00000000000000000000001 -2.5e-3 +7\ny 1E38 3.4028234663852886e38 -0.0\n"
                         b"z 1.401298464324817e-45 0.000001401298464324817 123456789012345678901234\n"
                         b"w 1. .5 -00012.50e+001\n"),
    }


def malformed_files():
    """(name, bytes, dim, lowest bad line)."""
    return [
        ("too_few_fields", b"a 1 2\nb 3\n", None, 2),
        ("bad_number", b"a 1 2\n\nb 3 x\n", None, 3),
        ("nan", b"a 1 2\nb nan 1\n", None, 2),
        ("inf", b"a 1 2\nb 1 -inf\n", None, 2),
        ("overflow", b"a 1 2\nb 1 1e39\n", None, 2),
        ("lowest_of_two", b"a 1 2\nb x 2\nc 1\n", None, 2),
        ("header_more", b"1 2\na 1 2\nb 3 4\n", None, 3),
        ("header_fewer", b"3 2\na 1 2\nb 3 4\n", None, 4),
        ("header_fewer_unterminated", b"3 2\na 1 2\n\nb 3 4", None, 5),
        ("header_dim", b"2 3\na 1 2 3\nb 1 2\n", None, 3),
        ("dim_given", b"a 1 2 3\nb 1 2 3\n", 4, 1),
        ("empty_word", b"a 1 2\n 1 2\n", None, 2),
        ("too_long", b"a 1 2\n\r\nb 1.000000059604644775390625000001 2\n", None, 3),
        ("d1_header", b"2 1\na 1\n", None, 1),
        ("d1", b"\n a 1\n", None, 2),
        ("d_too_big", b"2 511\n", None, 1),
    ]
