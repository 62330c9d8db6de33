"""The device reader of saved trajectory text (csrc/vap_parse.cuh: k_line_starts / k_body_starts / k_line_offsets /
k_path_lines, k_line_kinds, k_parse_lines, k_compare_bodies, behind export.parse_text_batch / compare_text_batch) against
a plain Python reader of the same grammar, and the formatter / number parser of vap_format.cuh / vap_parse.cuh built
for the host and compared with repr() / float() on every exponent band.

The reader (ref_lines, ref_line, ref_parse, ref_compare) is the specification:
- lines: a body is split after every '\\n'; a non-empty tail without '\\n' is a line too; an empty body has no lines;
- the first token is the bytes up to the first ' ' or '\\n' ('\\r', '\\t' are token bytes): empty -> LINE_ERR_BLANK,
  "0" a trajectory row, "1" an action row, anything else LINE_ERR_KIND;
- trajectory rows: tokens are separated by runs of ' '; a token must match TOKEN (its value is float(token)), a bad one
  is NaN and the first bad one sets 4 + column; a token count other than 7 sets LINE_ERR_TOKENS instead, missing columns
  are NaN; an erroneous row is still a row;
- comparison: the first differing byte (min(len) when one body is a prefix of the other, -1 when equal) and its line
  old[:diff].count('\\n') + 1; action rows compared by their line bytes, k-th saved against k-th fresh, plus the
  unpaired ones; max |old - new| of columns 1..6 over the common rows (equal or both NaN: 0; a NaN difference: inf);
  the t of the last row of each side (NaN without rows)."""
import ctypes as C
import dataclasses
import os
import re
import subprocess
from decimal import Decimal, getcontext

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "vexautonomousplanner_b200", "csrc")
NAN = float("nan")
TOKEN = re.compile(rb"-?(?:\d+(?:\.\d+)?(?:[eE][+-]?\d+)?|inf|nan)")
FIRST = re.compile(rb"[^ \n]*")
# a body exactly as the writer lays it out: "0 " + six good tokens, each followed by " ", then "\n"; "1 ...\n"
WRITER_BODY = re.compile(rb"(?:0(?: " + TOKEN.pattern + rb"){6} \n|1 [^\n]*\n)*+")
ACTION = re.compile(rb"^1(?: [^\n]*)?(?:\n|\Z)", re.M)             # a line whose first token is "1"
LINE_TRAJ, LINE_ACTION, LINE_OTHER = 0, 1, 2
ERR_BLANK, ERR_KIND, ERR_TOKENS, ERR_TOKEN = 1, 2, 3, 4


# ---------------------------------------------------------------------------------------------------------- reader
def ref_lines(body: bytes):
    """(start, end) of every line of one body."""
    out, s = [], 0
    while s < len(body):
        e = body.find(b"\n", s)
        e = len(body) if e < 0 else e + 1
        out.append((s, e))
        s = e
    return out


def ref_kind(line: bytes):
    """(kind, error code) of one line from its first token."""
    first = FIRST.match(line).group()
    if not first:
        return LINE_OTHER, ERR_BLANK
    if first in (b"0", b"1"):
        return (LINE_TRAJ, 0) if first == b"0" else (LINE_ACTION, 0)
    return LINE_OTHER, ERR_KIND


def ref_line(line: bytes):
    """(kind, error code, row) of one line; row is [0.0, six values] for a trajectory row, else None."""
    kind, err = ref_kind(line)
    if kind != LINE_TRAJ:
        return kind, err, None
    toks = [t for t in line.rstrip(b"\n").split(b" ") if t]
    row = [0.0]
    for c, t in enumerate(toks[1:7], start=1):
        ok = TOKEN.fullmatch(t) is not None
        row.append(float(t) if ok else NAN)
        if not ok and err == 0:
            err = ERR_TOKEN + c
    row += [NAN] * (7 - len(row))
    return LINE_TRAJ, (ERR_TOKENS if len(toks) != 7 else err), row


@dataclasses.dataclass
class RefParsed:
    line_offsets: list
    path_line_offsets: list
    kinds: list
    errors: list
    rows: list
    row_offsets: list
    act_lines: list
    act_offsets: list


def ref_parse(bodies):
    """parse_text_batch of the concatenated bodies, restated."""
    r = RefParsed([], [0], [], [], [], [0], [], [0])
    base = 0
    for body in bodies:
        for s, e in ref_lines(body):
            kind, err, row = ref_line(body[s:e])
            if kind == LINE_ACTION:
                r.act_lines.append(len(r.kinds))
            if row is not None:
                r.rows.append(row)
            r.line_offsets.append(base + s)
            r.kinds.append(kind)
            r.errors.append(err)
        base += len(body)
        r.path_line_offsets.append(len(r.kinds))
        r.row_offsets.append(len(r.rows))
        r.act_offsets.append(len(r.act_lines))
    r.line_offsets.append(base)
    return r


def first_diff(a: bytes, b: bytes) -> int:
    m = min(len(a), len(b))
    ne = np.flatnonzero(np.frombuffer(a[:m], dtype=np.uint8) != np.frombuffer(b[:m], dtype=np.uint8))
    if ne.size:
        return int(ne[0])
    return m if len(a) != len(b) else -1


def ref_body(body: bytes):
    """(rows [R, 7], action row lines, first error line from 1 or 0, its code) of one body: line by line, with every
    run of lines in the writer's layout read in bulk (no error there; the same values, sooner)."""
    rows, acts, err_line, err_code, n_lines, pos = [], [], 0, 0, 0, 0
    while pos < len(body):
        end = WRITER_BODY.match(body, pos).end()
        if end > pos:
            vals = b" ".join(re.findall(rb"^0 (.*) $", body[pos:end], re.M)).decode()
            rows += [[0.0] + r for r in np.array(list(map(float, vals.split(" "))) if vals else []).reshape(-1, 6).tolist()]
            acts += ACTION.findall(body, pos, end)
            n_lines += body.count(b"\n", pos, end)
            pos = end
            continue
        end = body.find(b"\n", pos) + 1 or len(body)
        kind, err, row = ref_line(body[pos:end])
        n_lines += 1
        if err and not err_line:
            err_line, err_code = n_lines, err
        if row is not None:
            rows.append(row)
        if kind == LINE_ACTION:
            acts.append(body[pos:end])
        pos = end
    return np.array(rows, dtype=np.float64).reshape(-1, 7), acts, err_line, err_code


def ref_compare(old: bytes, new: bytes, new_rows):
    """(ints named by export.CMP_I, floats named by export.CMP_F) of one saved body against the fresh body and its
    numeric rows new_rows [R, 7]."""
    diff = first_diff(old, new)
    a, old_acts, err_line, err_code = ref_body(old)
    new_acts = ACTION.findall(new)
    act = sum(x != y for x, y in zip(old_acts, new_acts)) + abs(len(old_acts) - len(new_acts))
    c = np.asarray(new_rows, dtype=np.float64).reshape(-1, 7)
    n = min(len(a), len(c))
    x, y = a[:n, 1:], c[:n, 1:]
    with np.errstate(invalid="ignore", over="ignore"):
        d = np.where((x == y) | (np.isnan(x) & np.isnan(y)), 0.0, np.abs(x - y))
    d[np.isnan(d)] = np.inf
    ints = [diff, old[:diff].count(b"\n") + 1 if diff >= 0 else 0, len(a), len(c), act, err_line, err_code]
    floats = [a[-1, 1] if len(a) else NAN, c[-1, 1] if len(c) else NAN, *d.max(axis=0, initial=0.0)]
    return np.array(ints, dtype=np.int64), np.array(floats, dtype=np.float64)


def _same_f(got, want) -> np.ndarray:
    """Bit-equal, NaN by class."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    return (got.view(np.int64) == want.view(np.int64)) | (np.isnan(got) & np.isnan(want))


# ---------------------------------------------------------------------------------------------------------- corpus
def _row(*vals) -> bytes:
    return ("".join(f"{v} " for v in (0, *vals)) + "\n").encode()


def _base(n_rows: int, seed: int, crlf: bool = False) -> bytes:
    """A body of action and trajectory rows as the writer lays it out."""
    rng = np.random.default_rng(seed)
    lines = [b"1 0 0 \n"]
    for k in range(n_rows):
        lines.append(_row(*[float(v) for v in np.round(rng.normal(0, 30, 6), int(rng.integers(0, 17)))]))
        if k % 9 == 4:
            lines.append(f"1 {k} True \n".encode())
    lines.append(b"1 \n")
    body = b"".join(lines)
    return body.replace(b"\n", b"\r\n") if crlf else body


# decimals on or just off the midpoint of two neighbouring doubles, more than 19 significant digits: float() decides
# them, the device leaves them for the host (the host-built parser below checks that it does)
HOST_TIE = b"1.00000000000000011102230246251565404236316680908203125"
HOST_UP = b"1.00000000000000011102230246251565404236316680908203126"
HOST_TOKENS = (HOST_TIE, HOST_UP, b"-9007199254740993.0000000000000000000001",
               b"0.100000000000000012490009027033011079765856266021728515625")
MALFORMED = [b"-", b"1.", b".5", b"1e", b"1e+", b"--1", b"1.2.3", b"abc", b"0x10", b"1e5x", b"+1", b"in", b"infinity",
             b"nan0", b"1_000", b"0,5", b"1e-", b"-.5", b"e5", b"1.0e5.0", b"1\t", b"\r", b"Inf", b"NaN", b"1e5\r"]


def _flip(body: bytes, i: int) -> bytes:
    return body[:i] + bytes([body[i] ^ 1]) + body[i + 1:]


def corpus_pairs():
    """(saved, fresh) body pairs at the edges of the line split, the classifier, the row parser and the comparison."""
    base, long_, crlf = _base(16, 1), _base(70, 2), _base(16, 1, crlf=True)
    assert len(base) > 1000 and len(long_) > 5000
    pairs = [(b"", b""), (b"", base), (base, b""), (base, base), (long_, long_)]
    pairs += [(base[:-1], base), (base, base[:-1]), (base[:-1], base[:-1])]          # no final '\n'
    cut = base.index(b"\n", 600) + 1
    pairs += [(base[:cut], base), (base, base[:cut]), (base[:cut + 5], base), (base, base[:cut + 5])]   # prefixes
    for i in (0, 31, 32, 511, 512, 513, len(base) - 1):                                # the 32-lane x 16 byte strides
        pairs += [(_flip(base, i), base), (base, _flip(base, i))]
    for i in (1023, 1024, 1535, 4000, len(long_) - 2):
        pairs.append((_flip(long_, i), long_))
    pairs += [(crlf, base), (base, crlf), (crlf, crlf)]                                 # '\r\n' line ends
    body_rows = base.split(b"\n")
    pairs.append((b"\n".join(body_rows[:3] + [b""] + body_rows[3:]), base))             # a blank line
    pairs.append((b"\n".join(body_rows[:3] + [b"   "] + body_rows[3:]), base))          # spaces only
    pairs.append((b"\n".join(body_rows[:5] + [b" " + body_rows[5]] + body_rows[5:]), base))   # a leading space
    pairs += [(b"\n", b"\n"), (b"\n\n\n", base), (b"0", b"0 "), (b"0\n", _row(1, 2, 3, 4, 5, 6)),
              (b"0\n0 \n0", b"0 1 \n"), (b"1", b"1 "), (b"1\n", b"1\n"), (b" ", b"")]
    pairs += [(_row(1, 2, 3, 4, 5), _row(1, 2, 3, 4, 5, 6)), (_row(1, 2, 3, 4, 5, 6, 7), _row(1, 2, 3, 4, 5, 6)),
              (_row(1, 2, 3, 4, 5, 6) + _row(*range(8, 16)), _row(1, 2, 3, 4, 5, 6)),
              (b"0 1 2 3 4 5 6", b"0 1 2 3 4 5 6 \n"), (b"0   1 2  3 4 5 6   \n", b"0 1 2 3 4 5 6 \n")]
    for first in (b"01", b"00", b"0.0", b"-0", b"1.0", b"2", b"0\t", b"0\r", b"\t0", b"#"):
        pairs.append((_row(1, 2, 3, 4, 5, 6) + first + b" 1 2 3 4 5 6 \n", _row(1, 2, 3, 4, 5, 6) * 2))
    special = [("nan", "nan"), ("inf", 1.0), ("nan", 1.0), ("-0.0", "0.0"), ("inf", "inf"), ("inf", "-inf"),
               ("-nan", "nan"), ("1e308", "-1e308"), ("0", "-0.0"), ("-inf", "-inf")]
    for j, (u, v) in enumerate(special):
        cols_u, cols_v = [1.5, 2, 3, 4, 5, 6], [1.5, 2, 3, 4, 5, 6]
        cols_u[j % 6], cols_v[j % 6] = u, v
        pairs.append((base + _row(*cols_u) + _row(9, 9, 9, 9, 9, 9), base + _row(*cols_v)))
    for j, tok in enumerate(MALFORMED):
        cols = ["1", "2", "3", "4", "5", "6"]
        cols[j % 6] = tok.decode()
        pairs.append((base + ("0 " + " ".join(cols) + " \n").encode() + _row(1, 2, 3, 4, 5, 6), base + _row(1, 2, 3, 4, 5, 6)))
    pairs.append((long_ + b"x\n" + _row(1, 2, 3, 4, 5, 6, 7), long_ + _row(1, 2)))      # first error past 32 lines
    for j, tok in enumerate(HOST_TOKENS):                                                # tokens left for the host
        cols = [b"1", b"2", b"3", b"4", b"5", b"6"]
        cols[(2 * j + 1) % 6] = tok
        pairs.append((base + b"0 " + b" ".join(cols) + b" \n", base + _row(1, 2, 3, 4, 5, 6)))
    # a host token behind a token holding '\t' or '\r': the host must count the columns as the device does
    pairs.append((b"0 1\t2 " + HOST_UP + b" 3 4 5 6 \n", _row(1, 2, 3, 4, 5, 6)))
    pairs.append((b"0 a\rb " + HOST_UP + b" 3 4 5 " + HOST_TIE + b" \n" + _row(1, 2, 3, 4, 5, 6), _row(1, 2, 3, 4, 5, 6)))
    acts = [b"1 0 0 \n", b"1 5 True \n", b"1 [1, 2] \n"]
    pairs += [(base.replace(b"1 13 True", b"1 13 False"), base), (base + acts[1], base), (base, base + acts[1]),
              (acts[0] * 40, acts[0] * 39 + acts[2]), (acts[0] * 40 + acts[1], acts[0] * 41),
              (base.replace(b"1 4 True \n", b""), base), (acts[2] + _row(1, 2, 3, 4, 5, 6), acts[2][:-1] + _row(1, 2, 3, 4, 5, 6))]
    return pairs


def corpus_bodies():
    seen, out = set(), []
    for pair in corpus_pairs():
        for body in pair:
            if body not in seen:
                seen.add(body)
                out.append(body)
    return out


def _chunks(items, B):
    """Consecutive chunks of B items that cover every item (the last one wraps around)."""
    n = len(items)
    return [[items[(k + j) % n] for j in range(B)] for k in range(0, n, B)]


# ------------------------------------------------------------------------------------------------------------- CPU
def test_reference_reader_cpu():
    """The reader itself on cases worked out by hand, so that a slip in it cannot hide a kernel bug."""
    assert ref_lines(b"") == [] and ref_lines(b"a") == [(0, 1)] and ref_lines(b"a\n\nb") == [(0, 2), (2, 3), (3, 4)]
    assert ref_line(b"\n")[:2] == (LINE_OTHER, ERR_BLANK) and ref_line(b" 0 1\n")[:2] == (LINE_OTHER, ERR_BLANK)
    assert ref_line(b"0\r\n")[:2] == (LINE_OTHER, ERR_KIND) and ref_line(b"1")[:2] == (LINE_ACTION, 0)
    assert ref_line(b"0 1 2 3 4 5 6 \r\n")[1] == ERR_TOKENS
    kind, err, row = ref_line(b"0 1 2 3 4 5 6\r\n")
    assert kind == LINE_TRAJ and err == ERR_TOKEN + 6 and row[1:6] == [1, 2, 3, 4, 5] and row[6] != row[6]
    kind, err, row = ref_line(b"0 x 2 +3 4")
    assert err == ERR_TOKENS and row[2] == 2.0 and row[4] == 4.0 and all(v != v for v in (row[1], row[3], row[5], row[6]))
    assert ref_line(b"0 1 2 3 4 5 6 7 \n")[1] == ERR_TOKENS and ref_line(b"0 -0.0 nan -inf 1e5 2E-3 7")[1] == 0
    r = ref_parse([b"0 1 2 3 4 5 6 \n1 a \n", b"", b"\n1 \n0 9"])
    assert r.line_offsets == [0, 15, 20, 21, 24, 27] and r.path_line_offsets == [0, 2, 2, 5]
    assert r.kinds == [0, 1, 2, 1, 0] and r.errors == [0, 0, ERR_BLANK, 0, ERR_TOKENS]
    assert r.row_offsets == [0, 1, 1, 2] and r.act_lines == [1, 3] and r.act_offsets == [0, 1, 1, 2]
    i, f = ref_compare(b"0 1 2 3 4 5 6 \n1 a \n", b"0 1 2 3 4 5 6 \n1 a \n", [[0, 1, 2, 3, 4, 5, 6]])
    assert i.tolist() == [-1, 0, 1, 1, 0, 0, 0] and f.tolist() == [1, 1, 0, 0, 0, 0, 0, 0]
    i, f = ref_compare(b"0 1 2 3 4 5 6 \n", b"0 1 2 3 4 5 6 \n1 a \n0 2 2 3 4 5 nan \n",
                       [[0, 1, 2, 3, 4, 5, 6], [0, 2, 2, 3, 4, 5, NAN]])
    assert i.tolist() == [15, 2, 1, 2, 1, 0, 0] and f[0] == 1 and f[1] == 2
    i, f = ref_compare(b"0 1 2 3 4 5 nan \n0 3 inf 3 4 5 6\n1 b \n1 c \n", b"0 1 2 3 4 5 6 \n1 a \n",
                       [[0, 1.5, 2, 3, 4, 5, 6], [0, 3, 2, 3, 4, 5, 6]])
    assert i.tolist() == [12, 1, 2, 2, 2, 0, 0] and f[0] == 3 and f[1] == 3
    assert f[2:].tolist() == [0.5, np.inf, 0, 0, 0, np.inf]
    i, f = ref_compare(b"ab", b"a", np.zeros((0, 7)))
    assert i.tolist() == [1, 1, 0, 0, 0, 1, ERR_KIND] and np.isnan(f[:2]).all()
    assert ref_compare(b"a\n", b"a\nb", np.zeros((0, 7)))[0][:2].tolist() == [2, 2]
    assert ref_compare(b"", b"x", np.zeros((0, 7)))[0][:2].tolist() == [0, 1]
    n_bulk = 0
    for body in corpus_bodies() + [b"1", b"1 2", b"1\n1", b"0 1 2 3 4 5 6 \n1 x\n"]:
        lines = [body[s:e] for s, e in ref_lines(body)]
        assert ACTION.findall(body) == [l for l in lines if ref_kind(l)[0] == LINE_ACTION], body
        rows, acts, err_line, err_code = ref_body(body)
        want = [ref_line(l) for l in lines]
        first_err = next(((k + 1, w[1]) for k, w in enumerate(want) if w[1]), (0, 0))
        assert (err_line, err_code) == first_err and acts == [l for l, w in zip(lines, want) if w[0] == LINE_ACTION]
        assert _same_f(rows, np.array([w[2] for w in want if w[2] is not None]).reshape(-1, 7)).all(), body
        n_bulk += WRITER_BODY.match(body).end() > 0
    assert n_bulk >= 50


def test_byte_groups_cpu():
    """The groups check_batch compares in: consecutive, covering every route once, at most the limit unless one route
    alone exceeds it."""
    from vexautonomousplanner_b200.save_routes import byte_groups
    assert byte_groups([], 10) == []
    assert byte_groups([5, 5, 5], 10) == [(0, 2), (2, 3)]
    assert byte_groups([0, 0, 11, 0, 3, 10, 10], 10) == [(0, 2), (2, 3), (3, 5), (5, 6), (6, 7)]
    rng = np.random.default_rng(1)
    for _ in range(200):
        sizes = rng.integers(0, 50, int(rng.integers(1, 40))).tolist()
        limit = int(rng.integers(1, 120))
        g = byte_groups(sizes, limit)
        assert [a for a, _ in g] == [0] + [z for _, z in g[:-1]] and g[-1][1] == len(sizes) and all(a < z for a, z in g)
        assert all(sum(sizes[a:z]) <= limit or z == a + 1 for a, z in g)
        assert all(sum(sizes[a:z + 1]) > limit for (a, _), (z, _) in zip(g, g[1:]))      # greedy: none could grow


_SHIM = r"""
#include <cstdint>
#include <cstring>
#define __device__
#define __forceinline__ inline
#define __global__
static inline uint64_t __ldg(const uint64_t* p) { return *p; }
static inline long long __double_as_longlong(double x) { long long b; memcpy(&b, &x, 8); return b; }
#define VAP_FORMAT_HOST_TEST
#define VAP_PARSE_HOST_TEST
#define VAP_POW5_128_SPACE
#include "vap_format.cuh"
#include "vap_parse.cuh"
extern "C" void h_repr(long long n, const double* x, char* out, int* len) { for (long long i = 0; i < n; i++) len[i] = format_repr(x[i], out + 32 * i); }
extern "C" void h_parse(long long n, const char* s, const long long* off, double* out, signed char* flag)
{ for (long long i = 0; i < n; i++) flag[i] = (signed char)parse_token(s + off[i], off[i + 1] - off[i], out[i]); }
"""


@pytest.fixture(scope="module")
def host_lib(tmp_path_factory):
    """format_repr and parse_token of the device headers, compiled for the host with g++."""
    d = tmp_path_factory.mktemp("vap_host")
    src, so = d / "shim.cpp", d / "libvap_host.so"
    src.write_text(_SHIM)
    subprocess.run(["g++", "-O2", "-fPIC", "-shared", "-I", CSRC, "-o", str(so), str(src)], check=True)
    L = C.CDLL(str(so))
    L.h_repr.argtypes = [C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p]
    L.h_parse.argtypes = [C.c_longlong, C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p]

    def repr_all(xs):
        x = np.ascontiguousarray(xs, dtype=np.float64)
        out = np.zeros((x.size, 32), dtype=np.uint8)
        lens = np.zeros(x.size, dtype=np.int32)
        L.h_repr(x.size, x.ctypes.data, out.ctypes.data, lens.ctypes.data)
        return [bytes(out[i, :lens[i]]).decode() for i in range(x.size)]

    def parse_all(toks):
        enc = [t.encode() if isinstance(t, str) else t for t in toks]
        off = np.zeros(len(enc) + 1, dtype=np.int64)
        np.cumsum([len(t) for t in enc], out=off[1:])
        out = np.zeros(len(enc), dtype=np.float64)
        flags = np.zeros(len(enc), dtype=np.int8)
        L.h_parse(len(enc), b"".join(enc), off.ctypes.data, out.ctypes.data, flags.ctypes.data)
        return out, flags

    return repr_all, parse_all


def _edge_values(seed: int, n_random: int):
    """Every exponent x 8 mantissa edges, the neighbours of 1ek, 5ek and 9.999999999999999ek for k in [-330, 310],
    random bit patterns; finite values only."""
    rng = np.random.default_rng(seed)
    e = np.repeat(np.arange(2047, dtype=np.uint64), 8)
    m = np.tile(np.array([0, 1, 2, (1 << 52) - 1, (1 << 52) - 2, 1 << 51, 0, 0], dtype=np.uint64), 2047)
    m[6::8] = rng.integers(0, 1 << 52, 2047, dtype=np.uint64)
    m[7::8] = rng.integers(0, 1 << 52, 2047, dtype=np.uint64)
    xs = ((e << np.uint64(52)) | m).view(np.float64)
    dec = np.array([float(f"{s}e{k}") for k in range(-330, 311) for s in ("1", "5", "9.999999999999999")])
    near = np.concatenate([dec, np.nextafter(dec, np.inf), np.nextafter(dec, 0)])
    rnd = rng.integers(0, 2 ** 63, n_random, dtype=np.int64).view(np.float64)
    allx = np.concatenate([xs, near, rnd, -xs[:2047 * 8:5]])
    return allx[np.isfinite(allx)]


def test_host_format_repr_every_exponent_cpu(host_lib):
    """format_repr == repr() on every exponent band (mantissa edges), around every power of ten and on random bits."""
    repr_all, _ = host_lib
    xs = _edge_values(1, 200_000)
    got = repr_all(xs)
    bad = [(x, g) for x, g in zip(xs.tolist(), got) if g != repr(x)]
    assert not bad, bad[:5]
    assert len(xs) > 210_000


def test_host_parse_token_every_exponent_cpu(host_lib):
    """parse_token == float() bit for bit on the same values in repr, %.17g, %.16e and %.20e forms, the midpoint and
    1e-30-off tokens of test_trajectory_check._tokens and the malformed ones; a token it leaves for the host is one
    that needs more than 19 significant digits."""
    from test_trajectory_check import MALFORMED as MAL, _tokens
    _, parse_all = host_lib
    xs = _edge_values(2, 30_000).tolist()
    toks = [f % x for x in xs for f in ("%r", "%.17g", "%.16e", "%.20e")]
    more, _ = _tokens(40_000, seed=4)
    toks += more + [t.decode() for t in HOST_TOKENS] + ["-0", "-0.0", "0e999", "1e400", "-1e400", "1e-400", "-inf", "-nan"]
    got, flags = parse_all(toks)
    assert (flags != 2).all(), [toks[i] for i in np.flatnonzero(flags == 2)[:5]]
    want = np.array([float(t) for t in toks])
    dev = flags == 0
    bad = np.flatnonzero(dev & ~_same_f(got, want))
    assert bad.size == 0, [(toks[i], got[i], want[i]) for i in bad[:5]]
    host = {toks[i] for i in np.flatnonzero(flags == 1)}
    assert {t.decode() for t in HOST_TOKENS} <= host
    assert dev.sum() > 300_000 and (flags[: 4 * len(xs): 4] == 0).all()              # repr never needs the host
    _, mflags = parse_all(MAL + [t for t in MALFORMED])
    assert (mflags == 2).all(), [t for t, f in zip(MAL + MALFORMED, mflags) if f != 2]


# ------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def eng():
    from vexautonomousplanner_b200.engine import Engine
    return Engine("cuda:0")


def _check_parsed(p, r, tag):
    got = {"line_offsets": p.line_offsets, "path_line_offsets": p.path_line_offsets, "kinds": p.line_kinds,
           "errors": p.line_errors, "row_offsets": p.row_offsets, "act_lines": p.act_lines, "act_offsets": p.act_offsets}
    for name, t in got.items():
        assert t.cpu().tolist() == getattr(r, name), (tag, name)
    rows = p.rows.cpu().numpy()
    want = np.array(r.rows, dtype=np.float64).reshape(-1, 7)
    assert rows.shape == want.shape, tag
    same = _same_f(rows, want)
    assert same.all(), (tag, [(tuple(ix), rows[tuple(ix)], want[tuple(ix)]) for ix in np.argwhere(~same)[:5]])


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 3, 4, 5, 129])
def test_parse_corpus_vs_reader(eng, B):
    """parse_text_batch on the hand-made corpus, B bodies per call: line offsets, kinds, errors, rows (bit for bit, NaN
    by class, host-finished tokens included), row / action / line offsets per body."""
    from vexautonomousplanner_b200 import export as ex
    n_host = 0
    for k, bodies in enumerate(_chunks(corpus_bodies(), B)):
        offs = np.cumsum([0] + [len(b) for b in bodies])
        p = ex.parse_text_batch(eng, b"".join(bodies), offs)
        _check_parsed(p, ref_parse(bodies), (B, k))
        n_host += p.n_host
    assert n_host >= 7


def _compare_chunk(eng, pairs, pinned: bool):
    import torch
    from vexautonomousplanner_b200 import export as ex
    old, new = [a for a, _ in pairs], [b for _, b in pairs]
    oo, no = np.cumsum([0] + [len(b) for b in old]), np.cumsum([0] + [len(b) for b in new])
    r = ref_parse(new)
    new_rows = torch.tensor(np.array(r.rows, dtype=np.float64).reshape(-1, 7), device=eng.device)
    new_ro = torch.tensor(r.row_offsets, dtype=torch.int64, device=eng.device)
    old_text, new_text = b"".join(old), b"".join(new)
    if pinned:                                          # room for the fresh text behind the saved one, and then some
        buf = torch.full((len(old_text) + len(new_text) + 7,), 0x7f, dtype=torch.uint8, pin_memory=True)
        buf[:len(old_text)].numpy()[:] = np.frombuffer(old_text, dtype=np.uint8)
        ints, floats, _ = ex.compare_text_batch(eng, buf, oo, new_text, no, new_rows, new_ro)
        assert bytes(buf[len(old_text):len(old_text) + len(new_text)].numpy()) == new_text   # the fresh text went there
    else:
        ints, floats, _ = ex.compare_text_batch(eng, old_text, oo, new_text, no, new_rows, new_ro)
    return ints, floats, r


def _check_compare(pairs, ints, floats, new_rows_of, tag):
    from vexautonomousplanner_b200.export import CMP_F, CMP_I
    assert ints.shape == (len(pairs), len(CMP_I)) and floats.shape == (len(pairs), len(CMP_F))
    for b, (old, new) in enumerate(pairs):
        wi, wf = ref_compare(old, new, new_rows_of(b))
        assert ints[b].tolist() == wi.tolist(), (tag, b, dict(zip(CMP_I, ints[b])), dict(zip(CMP_I, wi)), old[:80], new[:80])
        ok = _same_f(floats[b], wf)
        assert ok.all(), (tag, b, dict(zip(CMP_F, floats[b])), dict(zip(CMP_F, wf)))


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 3, 4, 5, 129])
def test_compare_corpus_vs_reader(eng, B):
    """compare_text_batch on the hand-made (saved, fresh) pairs, B pairs per call, with a fresh buffer and with a pinned
    saved text that has room for the fresh one: every CMP_I exactly, every CMP_F bit for bit (NaN by class)."""
    pairs = corpus_pairs()
    for k, chunk in enumerate(_chunks(pairs, B)):
        for pinned in (False, True):
            ints, floats, r = _compare_chunk(eng, chunk, pinned)
            rows = np.array(r.rows, dtype=np.float64).reshape(-1, 7)
            _check_compare(chunk, ints, floats, lambda b: rows[r.row_offsets[b]:r.row_offsets[b + 1]], (B, k, pinned))


def _mutate(body: bytes, kind: int, rng) -> bytes:
    """One seeded change of a saved body (kinds 0..7; any other kind leaves it as it is)."""
    if not body:
        return body
    lines = body.splitlines(keepends=True)
    traj = [i for i, l in enumerate(lines) if l.startswith(b"0 ")]
    acts = [i for i, l in enumerate(lines) if l.startswith(b"1 ")]
    if kind == 0:                                        # a flipped byte at a stride edge
        pos = [p for p in (0, 31, 32, 511, 512, 513, len(body) - 1) if p < len(body)]
        return _flip(body, pos[int(rng.integers(len(pos)))])
    if kind == 1 and traj:                               # a row deleted
        del lines[traj[int(rng.integers(len(traj)))]]
    elif kind == 2 and traj:                             # a row duplicated
        i = traj[int(rng.integers(len(traj)))]
        lines.insert(i, lines[i])
    elif kind == 3 and acts:                             # an action row changed
        i = acts[int(rng.integers(len(acts)))]
        lines[i] = lines[i][:-1] + b"7 \n"
    elif kind == 4:                                      # an action row added
        lines.insert(int(rng.integers(len(lines) + 1)), b"1 3 False \n")
    elif kind == 5 and acts:                             # an action row removed
        del lines[acts[int(rng.integers(len(acts)))]]
    elif kind == 6 and traj:                             # a token float() reads that the device leaves for the host
        i = traj[int(rng.integers(len(traj)))]
        tok = lines[i].split(b" ")
        c = int(rng.integers(1, 7))
        x = abs(float(tok[c]))
        if x == 0 or not np.isfinite(x):
            x = 1.0
        getcontext().prec = 800
        mid = (Decimal(x) + Decimal(float(np.nextafter(x, np.inf)))) / 2
        tok[c] = format(mid, "f").encode()
        lines[i] = b" ".join(tok)
    elif kind == 7:                                      # truncated mid-line
        i = int(rng.integers(len(lines)))
        return b"".join(lines[:i]) + lines[i][:max(1, len(lines[i]) // 2)]
    return b"".join(lines)


@pytest.mark.gpu
def test_compare_real_bodies_vs_reader(eng):
    """2048 mixed paths saved at the factory constraints, then changed (flipped bytes at the stride edges, rows
    deleted / duplicated, action rows changed / added / removed, host-only tokens, mid-line truncation), compared with
    the fresh bodies of a second constraint set and other action values: every path's CMP_I / CMP_F against the reader."""
    from test_trajectory_check import _mixed_batch
    from vexautonomousplanner_b200 import export as ex
    from vexautonomousplanner_b200.synth import FACTORY
    packed, na, aa = _mixed_batch(2048, 3)
    B = packed.B

    def save(cons, node_actions):
        db = eng.upload(dataclasses.replace(packed, cons=np.tile(np.array(cons, dtype=np.float64), (B, 1))))
        res = eng.profile(db)
        text, offs, _ = ex.save_text_batch(eng, res, db, node_actions, aa)
        return [text[offs[b]:offs[b + 1]].tobytes() for b in range(B)], res

    saved, _ = save(FACTORY, na)
    fresh, res = save((3.25, 6.5, 6.5, 0.8, 16.0, 11.0 / 12),
                      [[[9, 9] if (b % 5 == 0 and i == 0) else v for i, v in enumerate(n)] for b, n in enumerate(na)])
    rows, row_off = ex.export_rows(eng, res)
    rng = np.random.default_rng(11)
    old = [fresh[b] if b % 97 == 0 else _mutate(body, b % 10, rng) for b, body in enumerate(saved)]   # kinds 8, 9: as saved
    oo, no = np.cumsum([0] + [len(o) for o in old]), np.cumsum([0] + [len(f) for f in fresh])
    ints, floats, n_host = ex.compare_text_batch(eng, b"".join(old), oo, b"".join(fresh), no, rows, row_off)
    R = rows.cpu().numpy()
    ro = row_off.cpu().numpy()
    _check_compare(list(zip(old, fresh)), ints, floats, lambda b: R[ro[b]:ro[b + 1]], "real")
    assert n_host > 0
    diff = ints[:, 0]
    assert (diff == -1).sum() >= B // 97 and (ints[:, 4] > 0).sum() > B // 10 and (ints[:, 5] > 0).sum() > 0
    assert (ints[:, 2] != ints[:, 3]).sum() > B // 2 and (floats[:, 0] != floats[:, 1]).sum() > B // 2


@pytest.mark.gpu
def test_check_splits_reads_at_the_byte_limit(eng, tmp_path, monkeypatch):
    """check_routes with export.MAX_READ_BYTES lowered to the largest saved + fresh pair of one route: every read stays
    within it, one tile takes several reads, and the report is the one of the run that reads the tile at once."""
    from test_trajectory_check import _route_folder
    from vexautonomousplanner_b200 import export as ex, save_routes as sr
    from vexautonomousplanner_b200.synth import FACTORY
    half = (FACTORY[0] / 2,) + tuple(FACTORY[1:])
    rdir, odir, hdir = tmp_path / "routes", tmp_path / "out", tmp_path / "half"
    names = sorted(_route_folder(eng, rdir, half))
    routes, _ = sr.read_routes(str(rdir))
    for d, cons in ((odir, FACTORY), (hdir, half)):
        d.mkdir()
        assert sr.save_routes(routes, str(d), cons) == []
    (odir / names[1]).unlink()
    (odir / names[2]).write_bytes((odir / names[2]).read_bytes() + b"x\n")
    (odir / names[3]).write_bytes((hdir / names[3]).read_bytes())
    pair = max((odir / n).stat().st_size + (hdir / n).stat().st_size if (odir / n).exists() else 0 for n in names)
    reads, read = [], ex._read_bodies
    monkeypatch.setattr(ex, "_read_bodies", lambda e, text, offs, pp: reads.append(int(offs[-1])) or read(e, text, offs, pp))
    whole = sr.check_routes(routes, str(odir), half)
    assert len(reads) == 1
    reads.clear()
    monkeypatch.setattr(ex, "MAX_READ_BYTES", pair)
    split = sr.check_routes(routes, str(odir), half)
    assert split == whole and 1 < len(reads) <= len(names) and max(reads) <= pair, reads
    assert [s for _, s, _ in whole].count("stale") == len(names) - 3
    assert {s for _, s, _ in whole} == {"stale", "missing", "unreadable", "up to date"}
