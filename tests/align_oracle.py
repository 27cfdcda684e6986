"""ctypes binding of tests/align_oracle.c, the CPU restatement of read alignment (U16) the GPU results are checked against.

The library is compiled into the temporary directory, named by a hash of its sources, so the tree stays untouched."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = [os.path.join(HERE, "align_oracle.c"), os.path.join(ROOT, "minorseq_b200", "csrc", "align_rule.h")]
OPS = "MIDNSHP=X"
_COMP = str.maketrans("ACGT", "TGCA")


def revcomp(s: str) -> str:
    return "".join("N" if c not in "ACGT" else c for c in s[::-1]).translate(_COMP)


def cigar_string(ops) -> str:
    return "".join(f"{int(x) >> 4}{OPS[int(x) & 15]}" for x in ops)


def _build():
    h = hashlib.sha256()
    for s in SOURCES:
        with open(s, "rb") as f:
            h.update(f.read())
    lib = os.path.join(tempfile.gettempdir(), f"ms_align_oracle_{os.getuid()}_{h.hexdigest()[:16]}.so")
    if not os.path.exists(lib):
        tmp = f"{lib}.{os.getpid()}"
        subprocess.check_call(["gcc", "-O2", "-Wall", "-shared", "-fPIC", "-o", tmp, SOURCES[0]])
        os.replace(tmp, lib)
    return lib


class AlignOracle:
    def __init__(self):
        self.lib = C.CDLL(_build())
        self.lib.mso_align_index_new.restype = C.c_void_p
        self.lib.mso_align_index_new.argtypes = [C.c_char_p, C.c_int32]
        self.lib.mso_align_index_free.argtypes = [C.c_void_p]
        self.lib.mso_align_read.restype = C.c_int
        self.lib.mso_align_read.argtypes = [C.c_void_p, C.c_char_p, C.c_int32, C.c_int32] + [C.POINTER(C.c_int32)] * 3 + \
            [C.POINTER(C.c_uint32), C.c_int32, C.POINTER(C.c_int32)]
        self.lib.mso_overlap_score.restype = C.c_int32
        self.lib.mso_overlap_score.argtypes = [C.c_char_p, C.c_int32, C.c_char_p, C.c_int32]
        self.ix = None

    def set_reference(self, ref: str):
        if self.ix:
            self.lib.mso_align_index_free(self.ix)
        self._ref = ref.encode()          # the index points into it
        self.ix = self.lib.mso_align_index_new(self._ref, len(self._ref))

    def align(self, reads, min_seeds=10):
        """Same tuples as minorseq_b200.Aligner.align: (mapped, strand, pos, score, cigar string)."""
        out = []
        for r in reads:
            b = r.encode()
            st, pos, sc, n = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
            cap = 2 * len(b) + 1
            cig = (C.c_uint32 * cap)()
            rc = self.lib.mso_align_read(self.ix, b, len(b), min_seeds, C.byref(st), C.byref(pos), C.byref(sc), cig, cap, C.byref(n))
            assert rc >= 0
            out.append((bool(rc), st.value, pos.value, sc.value, cigar_string(cig[:n.value]) if rc else ""))
        return out

    def overlap_score(self, a: str, ref: str) -> int:
        return int(self.lib.mso_overlap_score(a.encode(), len(a), ref.encode(), len(ref)))
