"""Minimal reader for R `save()` files (gzip + "RDX3" XDR serialisation, version 2/3).

TEST INFRASTRUCTURE ONLY (part of the parity oracle; never imported by the product path).

Purpose: load the reference's bundled fixture `inst/extdata/pbmc3k-50cells.rda`
(a `dgCMatrix` X with slots i, p, Dim, Dimnames, x + a character vector `celltype`;
built by reference `dev/extdata.R:1-15`) without an R installation, so that the
oracle and the CUDA path can be exercised on the reference's own real input.

Only the SEXP types that occur in such files are supported: NILVALUE, LISTSXP,
SYMSXP, REFSXP, CHARSXP, LGLSXP, INTSXP, REALSXP, STRSXP, VECSXP, S4SXP and the
ALTREP wrappers R emits for plain vectors (compact_intseq / compact_realseq /
wrap_*).  S4 objects are returned as dicts {"__class__": ..., slot: value}.
"""
from __future__ import annotations

import gzip
import bz2
import lzma
import struct
import numpy as np

_NILVALUE, _GLOBALENV, _EMPTYENV, _BASEENV = 254, 253, 242, 241
_REFSXP, _ALTREP, _NAMESPACESXP, _PACKAGESXP, _PERSISTSXP = 255, 238, 249, 250, 247
_MISSINGARG, _UNBOUND, _BASENAMESPACE = 251, 252, 247 + 0
_ATTRLANG, _ATTRLIST = 240, 239

NA_INTEGER = -2147483648


class _Reader:
    def __init__(self, buf: bytes):
        self.b = buf
        self.o = 0
        self.refs: list = []

    def _int(self) -> int:
        v = struct.unpack_from(">i", self.b, self.o)[0]
        self.o += 4
        return v

    def _bytes(self, n: int) -> bytes:
        v = self.b[self.o:self.o + n]
        self.o += n
        return v

    def _len(self) -> int:
        n = self._int()
        if n == -1:  # long vector: two ints (upper, lower)
            hi, lo = self._int(), self._int()
            n = (hi << 32) + (lo & 0xFFFFFFFF)
        return n

    def item(self):
        flags = self._int()
        typ = flags & 0xFF
        has_attr = bool(flags & 0x200)
        has_tag = bool(flags & 0x400)
        is_obj = bool(flags & 0x100)

        if typ == _NILVALUE:
            return None
        if typ in (_GLOBALENV, _EMPTYENV, _BASEENV, _MISSINGARG, _UNBOUND):
            return None
        if typ == _REFSXP:
            idx = flags >> 8
            if idx == 0:
                idx = self._int()
            return self.refs[idx - 1]
        if typ == 1:  # SYMSXP
            name = self.item()
            self.refs.append(name)
            return name
        if typ in (_NAMESPACESXP, _PACKAGESXP, _PERSISTSXP):
            self._int()  # always 0
            n = self._int()
            val = [self.item() for _ in range(n)]
            self.refs.append(val)
            return val
        if typ in (2, 6, _ATTRLANG, _ATTRLIST):  # LISTSXP / LANGSXP: walk iteratively
            out = []
            attrs = None
            while True:
                if typ in (_ATTRLANG, _ATTRLIST):
                    has_attr = True
                if has_attr:
                    attrs = self.item()
                tag = self.item() if has_tag else None
                car = self.item()
                out.append((tag, car))
                flags = self._int()
                typ = flags & 0xFF
                has_attr = bool(flags & 0x200)
                has_tag = bool(flags & 0x400)
                if typ == _NILVALUE:
                    break
                if typ not in (2, 6, _ATTRLANG, _ATTRLIST):
                    raise ValueError(f"unexpected cdr type {typ}")
            return out
        if typ == 9:  # CHARSXP
            n = self._int()
            if n == -1:
                return None
            return self._bytes(n).decode("utf-8", errors="replace")
        if typ == _ALTREP:
            info = self.item()
            state = self.item()
            attr = self.item()
            cls = info[0][1] if info else None
            val = self._altrep(cls, state)
            return self._with_attr(val, attr, False)
        if typ == 25:  # S4SXP: body is only its attributes (slots)
            attr = self.item() if has_attr else []
            obj = {}
            for tag, v in attr or []:
                if tag == "class":
                    obj["__class__"] = v[0] if isinstance(v, list) else v
                else:
                    obj[tag] = v
            return obj

        if typ == 10 or typ == 13:  # LGLSXP / INTSXP
            n = self._len()
            val = np.frombuffer(self.b, dtype=">i4", count=n, offset=self.o).astype(np.int32)
            self.o += 4 * n
        elif typ == 14:  # REALSXP
            n = self._len()
            val = np.frombuffer(self.b, dtype=">f8", count=n, offset=self.o).astype(np.float64)
            self.o += 8 * n
        elif typ == 16:  # STRSXP
            n = self._len()
            val = [self.item() for _ in range(n)]
        elif typ in (19, 20):  # VECSXP / EXPRSXP
            n = self._len()
            val = [self.item() for _ in range(n)]
        elif typ == 24:  # RAWSXP
            n = self._len()
            val = self._bytes(n)
        else:
            raise NotImplementedError(f"SEXP type {typ} at offset {self.o}")
        attr = self.item() if has_attr else None
        return self._with_attr(val, attr, is_obj)

    @staticmethod
    def _altrep(cls, state):
        if cls == "compact_intseq":
            n, start, inc = (int(v) for v in state[:3])
            return (start + inc * np.arange(n)).astype(np.int32)
        if cls == "compact_realseq":
            n, start, inc = state[:3]
            return start + inc * np.arange(int(n), dtype=np.float64)
        if cls and cls.startswith("wrap_"):
            return state[0][1] if isinstance(state, list) and isinstance(state[0], tuple) else state[0]
        if cls == "deferred_string":
            arg = state[0][1] if isinstance(state[0], tuple) else state[0]
            return [str(v) for v in np.asarray(arg).tolist()]
        raise NotImplementedError(f"ALTREP class {cls}")

    @staticmethod
    def _with_attr(val, attr, is_obj):
        if not attr:
            return val
        d = {tag: v for tag, v in attr}
        if isinstance(val, list) and "names" in d and len(d) == 1:
            return dict(zip(d["names"], val)) if len(set(d["names"])) == len(val) else val
        if len(d) == 0:
            return val
        return {"__value__": val, "__attr__": d}


def _decompress(raw: bytes) -> bytes:
    if raw[:2] == b"\x1f\x8b":
        return gzip.decompress(raw)
    if raw[:3] == b"BZh":
        return bz2.decompress(raw)
    if raw[:6] == b"\xfd7zXZ\x00":
        return lzma.decompress(raw)
    return raw


def read_rda(path: str) -> dict:
    """Return {object name: value} for an R `save()` file."""
    with open(path, "rb") as fh:
        buf = _decompress(fh.read())
    if buf[:5] not in (b"RDX3\n", b"RDX2\n"):
        raise ValueError("not an RDX2/RDX3 file")
    if buf[5:7] != b"X\n":
        raise ValueError("only XDR serialisation is supported")
    r = _Reader(buf)
    r.o = 7
    version = r._int()
    r._int()  # writer R version
    r._int()  # min reader version
    if version == 3:
        n = r._int()
        r._bytes(n)  # native encoding
    top = r.item()
    return {tag: val for tag, val in top}


def dgc_to_scipy(obj: dict):
    """dgCMatrix dict (slots i, p, Dim, Dimnames, x) → (scipy.sparse.csc_matrix, rownames, colnames)."""
    import scipy.sparse as sp

    dim = np.asarray(obj["Dim"]).astype(np.int64)
    m = sp.csc_matrix(
        (np.asarray(obj["x"], dtype=np.float64), np.asarray(obj["i"], dtype=np.int32),
         np.asarray(obj["p"], dtype=np.int32)), shape=(int(dim[0]), int(dim[1])))
    dn = obj.get("Dimnames") or [None, None]
    return m, dn[0], dn[1]


# ---------------------------------------------------------------------------------------
# writer (tests only): serialise a dgCMatrix the way R's save() / saveRDS() do, so that the product's
# C++ reader (plaid_b200/csrc/matio.cu) can be exercised on generated files
# ---------------------------------------------------------------------------------------
def _w_int(out, v):
    out.append(struct.pack(">i", v))


def _w_sym(out, name, symtab):
    if name in symtab:  # REFSXP, index packed in the flags
        _w_int(out, (symtab[name] << 8) | _REFSXP)
        return
    symtab[name] = len(symtab) + 1
    _w_int(out, 1)  # SYMSXP
    _w_chr(out, name)


def _w_chr(out, s):
    b = s.encode("utf-8")
    _w_int(out, 9 | (1 << 15))  # CHARSXP, UTF-8 gp bit (0x8000 >> ... R packs levels in bits 12+; value irrelevant to readers)
    _w_int(out, len(b))
    out.append(b)


def _w_strsxp(out, strings):
    _w_int(out, 16)
    _w_int(out, len(strings))
    for s in strings:
        _w_chr(out, s)


def _w_dgc(out, m, rownames, colnames, symtab):
    """S4SXP with attribute pairlist i, p, Dim, Dimnames, x, factors, class (slot order of Matrix)"""
    _w_int(out, 25 | 0x100 | 0x200 | (1 << 16))  # S4SXP, object bit, attributes, S4 gp bit (bit 4 of gp << 12)

    def slot(name, writer):
        _w_int(out, 2 | 0x400)  # LISTSXP with tag
        _w_sym(out, name, symtab)
        writer()

    def ints(v):
        _w_int(out, 13)
        _w_int(out, len(v))
        out.append(np.asarray(v, dtype=">i4").tobytes())

    def reals(v):
        _w_int(out, 14)
        _w_int(out, len(v))
        out.append(np.asarray(v, dtype=">f8").tobytes())

    def dimnames():
        _w_int(out, 19)
        _w_int(out, 2)
        for nm in (rownames, colnames):
            if nm is None:
                _w_int(out, _NILVALUE)
            else:
                _w_strsxp(out, list(nm))

    def klass():
        _w_int(out, 16 | 0x200)  # STRSXP with attribute package = "Matrix"
        _w_int(out, 1)
        _w_chr(out, "dgCMatrix")
        _w_int(out, 2 | 0x400)
        _w_sym(out, "package", symtab)
        _w_strsxp(out, ["Matrix"])
        _w_int(out, _NILVALUE)

    slot("i", lambda: ints(m.indices))
    slot("p", lambda: ints(m.indptr))
    slot("Dim", lambda: ints(m.shape))
    slot("Dimnames", dimnames)
    slot("x", lambda: reals(m.data))
    slot("factors", lambda: (_w_int(out, 19), _w_int(out, 0)))
    slot("class", klass)
    _w_int(out, _NILVALUE)


def write_rda(path: str, objects: dict, version: int = 3, compress: bool = True, rds: bool = False):
    """objects: {name: (scipy csc_matrix, rownames | None, colnames | None) or a list of str (a character
    vector)}.  `rds=True` writes the first object, a matrix, the way saveRDS() does (no RDX header, no name)."""
    out: list = []
    if not rds:
        out.append(b"RDX3\n" if version == 3 else b"RDX2\n")
    out.append(b"X\n")
    _w_int(out, version)
    _w_int(out, 0x040303)  # R 4.3.3
    _w_int(out, 0x030500 if version == 3 else 0x020300)
    if version == 3:
        _w_int(out, 5)
        out.append(b"UTF-8")
    symtab: dict = {}
    if rds:
        m, rn, cn = next(iter(objects.values()))
        m = m.tocsc()
        m.sort_indices()
        _w_dgc(out, m, rn, cn, symtab)
    else:
        for name, obj in objects.items():
            _w_int(out, 2 | 0x400)
            _w_sym(out, name, symtab)
            if isinstance(obj, list):
                _w_strsxp(out, obj)
                continue
            m, rn, cn = obj
            m = m.tocsc()
            m.sort_indices()
            _w_dgc(out, m, rn, cn, symtab)
        _w_int(out, _NILVALUE)
    raw = b"".join(out)
    with open(path, "wb") as fh:
        fh.write(gzip.compress(raw) if compress else raw)
