"""ctypes binding of the oracle's cs:Z: restatement (tests/oracle_cs.c: awo_cs_string, awo_alignment_to_paf_cs).

TEST INFRASTRUCTURE: the C file is compiled on first use into a private temporary directory (the repository tree may be
read-only) and linked against oracle/liballwave_oracle.so, whose alignments and PAF writer it extends."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import oracle_lib

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    oracle_lib.lib()  # builds oracle/liballwave_oracle.so when it is missing
    odir = os.path.dirname(oracle_lib._SO)
    tmp = tempfile.mkdtemp(prefix="oracle_cs_")
    atexit.register(shutil.rmtree, tmp, True)
    so = os.path.join(tmp, "liboracle_cs.so")
    subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-Wall", "-Wextra", "-std=c11", "-shared", "-o", so,
                           os.path.join(_HERE, "oracle_cs.c"), "-L" + odir, "-lallwave_oracle", "-Wl,-rpath," + odir])
    L = C.CDLL(so)
    L.awo_cs_string.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_int]
    L.awo_cs_string.restype = C.c_void_p
    L.awo_alignment_to_paf_cs.argtypes = [C.POINTER(oracle_lib.Result), C.c_char_p, C.c_char_p, C.c_size_t, C.c_char_p, C.c_char_p,
                                          C.c_size_t, C.c_int]
    L.awo_alignment_to_paf_cs.restype = C.c_void_p
    _lib = L
    return L


def _take(ptr):
    assert ptr, "the alignment does not consume both sequences"
    s = C.string_at(ptr).decode("latin-1")
    oracle_lib.lib().free(ptr)
    return s


def cs_string(ops: bytes, query: bytes, target: bytes, long_form=False) -> str:
    """awo_cs_string: the tag of the alignment `ops` (WFA2 letters) of the oriented query against the target"""
    return _take(lib().awo_cs_string(ops, len(ops), query, len(query), target, len(target), 1 if long_form else 0))


def align_pair_paf(query: bytes, target: bytes, qi, ti, p, qname, tname, long_form=False, use_mash=True, orientation_params=None):
    """oracle_lib.align_pair's PAF line with the cs column appended (awo_alignment_to_paf_cs)"""
    L0 = oracle_lib.lib()
    op = orientation_params or oracle_lib.Params(0, 1, 1, 1, 0, 0, 0, 0)
    r = oracle_lib.Result()
    L0.awo_align_pair(query, len(query), target, len(target), qi, ti, C.byref(p), C.byref(op), 1 if use_mash else 0, C.byref(r))
    try:
        return _take(lib().awo_alignment_to_paf_cs(C.byref(r), qname.encode(), query, len(query), tname.encode(), target, len(target),
                                                    1 if long_form else 0))
    finally:
        L0.awo_result_free(C.byref(r))
