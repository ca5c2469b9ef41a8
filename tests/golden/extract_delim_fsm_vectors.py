#!/usr/bin/env python3
"""Records what the reference's delimiter FSM translation unit (core/parser/DelimiterModeFsmParser.cpp) returns for
every input of tests/test_oracle_vs_reference_tu.py into tests/golden/ref_delim_fsm.npz.

Needs oracle/_ref/libref_delim.so, which oracle/build_ref.sh compiles in place from a reference checkout
(LC_REFERENCE).  Only the results are stored: the test regenerates its seeded inputs and checks them against the
stored digest."""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tests.test_oracle_vs_reference_tu import GOLDEN, cases_digest, encode_results, fsm_cases  # noqa: E402

SO = os.path.join(ROOT, "oracle", "_ref", "libref_delim.so")


def ref_fsm(lib, line: bytes, sep: int, quote: int):
    out = np.zeros(len(line) * 5 + 64, np.uint8)
    used = C.c_uint64(0)
    k = lib.ref_delim_fsm(line, 0, len(line), C.c_char(bytes([sep])), C.c_char(bytes([quote])),
                          out.ctypes.data_as(C.c_void_p), out.size, C.byref(used))
    if k < 0:
        return None
    cols, at = [], 0
    raw = out.tobytes()
    for _ in range(k):
        l = int.from_bytes(raw[at:at + 4], "little")
        cols.append(raw[at + 4:at + 4 + l])
        at += 4 + l
    return cols


def main():
    lib = C.CDLL(SO)
    lib.ref_delim_fsm.restype = C.c_int64
    lib.ref_delim_fsm.argtypes = [C.c_char_p, C.c_int32, C.c_int32, C.c_char, C.c_char, C.c_void_p, C.c_uint64,
                                  C.POINTER(C.c_uint64)]
    cases = list(fsm_cases())
    results = [ref_fsm(lib, line, sep, quote) for line, sep, quote in cases]
    np.savez_compressed(GOLDEN, cases_sha256=np.array(cases_digest(cases)), **encode_results(results))
    print("%s: %d cases, %d rejected by the FSM" % (GOLDEN, len(cases), sum(r is None for r in results)))


if __name__ == "__main__":
    main()
