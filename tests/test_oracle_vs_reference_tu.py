"""The oracle's delimiter FSM restatement checked against the REFERENCE's own translation unit
(core/parser/DelimiterModeFsmParser.cpp).  What that translation unit returns for every input below is stored in
tests/golden/ref_delim_fsm.npz (recorded by tests/golden/extract_delim_fsm_vectors.py from oracle/_ref/, which
oracle/build_ref.sh compiles in place from a reference checkout), so the comparison runs without one."""
import ctypes as C
import hashlib
import os
import random

import numpy as np

from oracle import oracle as orc

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_delim_fsm.npz")
N_RANDOM = 80000


def fsm_cases():
    """(line, sep, quote) in a fixed order: N_RANDOM seeded random lines over small alphabets dense in separators and
    quotes, then the reference's own TestProcessDoubleQuote inputs (ProcessorParseDelimiterNativeUnittest.cpp:1841-1904)."""
    rng = random.Random(20260922)
    for sep, quote in ((44, 39), (44, 34), (124, 39), (9, 34)):
        alpha = "ab1 " + chr(sep) * 3 + chr(quote) * 3 + "x,"
        for _ in range(N_RANDOM // 4):
            yield "".join(rng.choice(alpha) for _ in range(rng.randint(1, 24))).encode(), sep, quote
    for url in ("''PutData?Category=YunOsAccountOpLog", "PutData?Category=YunOs''AccountOpLog",
                "PutData?Category=YunOsAccountOpLog''", "''PutData?Category=YunOsAccountOpLog'",
                "'PutData?Category=Yun'Os'AccountOpLog'", "'PutData?Category=YunOs''AccountOpLog'",
                "'PutData?Category=YunOsAccountOpLog''", "'''PutData?Category=YunOs''AccountOpLog'''"):
        yield ("2013-10-31 21:03:49,POST," + url + ",0.024").encode(), 44, 39


def cases_digest(cases):
    h = hashlib.sha256()
    for line, sep, quote in cases:
        h.update(len(line).to_bytes(4, "little") + line + bytes([sep, quote]))
    return h.hexdigest()


def encode_results(results):
    """Column lists (None = the FSM rejects the line) -> the arrays stored in ref_delim_fsm.npz."""
    ncols = np.array([-1 if r is None else len(r) for r in results], np.int16)
    col_len = np.array([len(c) for r in results if r for c in r], np.uint32)
    col_bytes = np.frombuffer(b"".join(c for r in results if r for c in r), np.uint8)
    return {"ncols": ncols, "col_len": col_len, "col_bytes": col_bytes}


def decode_results(ncols, col_len, col_bytes):
    raw = col_bytes.tobytes()
    out, j, at = [], 0, 0
    for k in ncols.tolist():
        if k < 0:
            out.append(None)
            continue
        cols = []
        for l in col_len[j:j + k].tolist():
            cols.append(raw[at:at + l])
            at += l
        out.append(cols)
        j += k
    assert j == col_len.size and at == len(raw)
    return out


def oracle_fsm(line: bytes, sep: int, quote: int):
    L = orc.lib()
    a = np.frombuffer(line, np.uint8) if line else np.zeros(0, np.uint8)
    cap = len(line) + 2
    fo, fl, fd = (np.zeros(cap, np.uint32) for _ in range(3))
    k = int(L.orc_delim_fsm(a.ctypes.data_as(C.c_void_p) if a.size else None, 0, len(line), sep, quote,
                            fo.ctypes.data_as(C.c_void_p), fl.ctypes.data_as(C.c_void_p),
                            fd.ctypes.data_as(C.c_void_p), cap))
    if k < 0:
        return None
    cols = []
    for j in range(k):
        if fd[j]:
            dst = np.zeros(int(fl[j]) + 1, np.uint8)
            w = L.orc_delim_unquote(a.ctypes.data_as(C.c_void_p), int(fo[j]), int(fl[j]), quote,
                                    dst.ctypes.data_as(C.c_void_p))
            cols.append(bytes(dst[:w]))
        else:
            cols.append(line[int(fo[j]):int(fo[j]) + int(fl[j])])
    return cols


def test_fsm_restatement_equals_reference_translation_unit():
    cases = list(fsm_cases())
    with np.load(GOLDEN) as g:
        assert str(g["cases_sha256"]) == cases_digest(cases), "inputs differ from those the vectors were recorded on"
        want = decode_results(g["ncols"], g["col_len"], g["col_bytes"])
    assert len(want) == len(cases) == N_RANDOM + 8
    fails = 0
    for n, ((line, sep, quote), r) in enumerate(zip(cases, want)):
        o = oracle_fsm(line, sep, quote)
        assert r == o, (line, sep, quote, r, o)
        fails += n < N_RANDOM and r is None
    assert 1000 < fails < N_RANDOM - 1000  # both outcomes exercised
