"""Host replica of the insertion table's slot placement in csrc/fuse.cu (ins_tally_kernel), for tests that must know where
an insertion key lands: its 64-bit hash (mix64f over the column, the length and the bytes), the table size ms_fuse and
ms_group_consensus choose, and whether linear probing is forced past the table's last slot.

The replica is only as good as its agreement with the source, so `source_mismatches()` reads fuse.cu back and names every
constant or step of the hash that is no longer written there."""
import os
import re

import numpy as np

FUSE_CU = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "minorseq_b200", "csrc", "fuse.cu")
M64 = (1 << 64) - 1
SEED = 0x66757365
MIX = ((30, 0xbf58476d1ce4e5b9), (27, 0x94d049bb133111eb), (31, None))


def mix64f(x):
    """mix64f over a numpy uint64 array (wrapping arithmetic)"""
    x = np.asarray(x, dtype=np.uint64)
    with np.errstate(over="ignore"):
        for shift, mul in MIX:
            x = x ^ (x >> np.uint64(shift))
            if mul is not None:
                x = x * np.uint64(mul)
    return x


def key_hash(col, strings):
    """hash of the keys (col[i], strings[i]); strings: equal-length bytes objects"""
    strings = list(strings)
    n = len(strings[0]) if strings else 0
    assert all(len(s) == n for s in strings)
    col = np.broadcast_to(np.asarray(col, dtype=np.int64), (len(strings),))
    h = mix64f(np.uint64(SEED) ^ ((col.astype(np.uint32).astype(np.uint64)) << np.uint64(32)) ^ np.uint64(n))
    b = np.frombuffer(b"".join(strings), dtype=np.uint8).reshape(len(strings), n) if n else np.zeros((len(strings), 0), np.uint8)
    for k in range(n):
        h = mix64f(h ^ b[:, k].astype(np.uint64))
    return np.where(h == 0, np.uint64(1), h)


def table_size(nins):
    """slots of the table for nins events: the smallest power of two >= max(1024, 2 * nins)"""
    ts = 1024
    while ts < 2 * nins:
        ts <<= 1
    return ts


def forced_wrap(homes, ts):
    """True when linear probing must carry some key past slot ts - 1, whatever the order of insertion: for some a, more
    distinct keys have their home slot in [a, ts) than there are slots there."""
    h = np.sort(np.asarray(homes, dtype=np.int64))[::-1]
    return bool(np.any(np.arange(1, len(h) + 1) > ts - h))


def source_mismatches():
    """the parts of the replica that fuse.cu no longer says (empty: the replica matches the source)"""
    src = open(FUSE_CU).read()
    m = re.search(r"uint64_t mix64f\(uint64_t x\) \{(.*?)return x;", src, re.S)
    if not m:
        return ["mix64f not found in fuse.cu"]
    steps = re.findall(r"x \^= x >> (\d+);(?:\s*x \*= (0x[0-9a-fA-F]+)ULL;)?", m.group(1))
    want = [(str(s), "" if k is None else hex(k)) for s, k in MIX]
    bad = [] if [(s, k.lower()) for s, k in steps] == want else [f"mix64f steps {steps} != {want}"]
    m = re.search(r"__global__ void ins_tally_kernel\(.*?\n\}", src, re.S)
    body = m.group(0) if m else ""
    for needle in (f"mix64f(0x{SEED:x}ULL ^ (static_cast<uint64_t>(static_cast<uint32_t>(col[i])) << 32) ^ static_cast<uint32_t>(len[i]))",
                   "hsh = mix64f(hsh ^ static_cast<uint8_t>(s[k]))", "if (!hsh) hsh = 1;", "idx = static_cast<int64_t>(hsh) & mask;",
                   "idx = (idx + 1) & mask;"):
        if needle not in body:
            bad.append(f"ins_tally_kernel no longer has: {needle}")
    if "int64_t ts = 1024;\n        while (ts < 2 * nins) ts <<= 1;" not in src:
        bad.append("ms_fuse's table size rule changed")
    return bad
