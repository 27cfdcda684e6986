"""Host-side mirror of the juliet / fuse process interface over the C ABI.

The reference exposes only two executables (`juliet [options] in.bam out.{json,html}`,
/root/reference/doc/JULIET.md:61-66; `fuse in.bam out.fasta`, /root/reference/doc/FUSE.md:26-32).
`Juliet` and `Fuse` below keep their option names (config genes, region, mode_phasing,
min_perc, max_perc) and drive the CUDA kernels through libminorseq_b200.so.  PyTorch is
used only for device memory, streams and torch.distributed; with more than one rank the
reads are sharded and the count tensor is summed by ONE NCCL all-reduce.
"""
import ctypes as C
from dataclasses import dataclass, field

import numpy as np

from . import _lib
from ._lib import (AbundanceCounters, AbundanceParams, AbundanceRow, AlignParams, CallParams, FuseParams, Gene, Indel, IndelParams, LinkagePair, LinkageParams, PhaseCounters, ReadAlignment, SynthParams, Variant,
                   check)
from .synth import start_mask_words, tile_rows, untile_rows

CODONS = [a + b + c for a in "ACGT" for b in "ACGT" for c in "ACGT"]
# standard genetic code (NCBI table 1, TCAG order), re-indexed to 16*b0+4*b1+b2 with A<C<G<T.
# Stop codons are reported as amino acid "X" (screenshot juliet_hiv-hiv.png: CGA->TGA, R8X).
_NCBI = "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG"
_AA = "".join(_NCBI[16 * "TCAG".index(a) + 4 * "TCAG".index(b) + "TCAG".index(c)].replace("*", "X")
              for a in "ACGT" for b in "ACGT" for c in "ACGT")


def translate(codon_index: int) -> str:
    return _AA[codon_index]


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(C.c_void_p)
    return C.c_void_p(int(a))


@dataclass
class Haplotypes:
    patterns: np.ndarray            # [H, ceil(V/32)] uint32, juliet order
    counts: np.ndarray              # [H] uint64
    nreported: int
    names: list
    counters: dict
    hap_id: np.ndarray = None       # per local read, -1 = damaged
    ndistinct: int = -1             # distinct patterns in total (patterns/counts may hold only the first ones of the order)


@dataclass
class Linkage:
    """Pairwise linkage of the phasing keys (Juliet.linkage).  The significant pairs, ordered by v then w, as parallel arrays;
    and, for every pair, the counts behind the tests as dense [V, V] int64 matrices: n[v, w] informative reads (both codons
    clean), a[v, w] reads carrying both, b[v, w] v but not w, c[v, w] w but not v (over the informative reads)."""
    v: np.ndarray
    w: np.ndarray
    both: np.ndarray
    v_only: np.ndarray
    w_only: np.ndarray
    neither: np.ndarray
    d_prime: np.ndarray
    r2: np.ndarray
    pvalue: np.ndarray
    relation: np.ndarray            # 1 linked, 2 exclusive
    ntested: int                    # Bonferroni m
    keys: list
    n: np.ndarray
    a: np.ndarray
    b: np.ndarray
    c: np.ndarray


@dataclass
class Abundance:
    """Haplotype abundance (Juliet.haplotype_abundance, restatement choice U18): per pattern, in the order given, the reads
    compatible with it alone and with it at all, and the EM's frequency over the unique and ambiguous reads."""
    unique_reads: np.ndarray        # [H] uint64
    compatible_reads: np.ndarray    # [H] uint64
    em_frequency: np.ndarray        # [H] float64
    counters: dict                  # unique, ambiguous, uninformative, incompatible
    reads_used: int                 # unique + ambiguous: the EM's reads
    iterations: int
    converged: bool
    log_likelihood: float
    tolerance: float
    max_iterations: int

    @property
    def em_reads(self):
        return self.em_frequency * self.reads_used


@dataclass
class Indels:
    """In-frame codon deletions and insertions (Juliet.indels, restatement choice U19).  The calls, sorted by (gene, codon,
    deletion before insertion, string), as parallel arrays; inserted[i] is the upper-cased inserted string ('' for a
    deletion) and label[i] the amino-acid label (D67del, T69_S70insSS).  The counts behind them: cnt[L, 2] = k_del (reads
    with '-' at s, s+1, s+2) and n_ins (reads clean at c and c+1) of every column, tally[sid] the reads of each inserted
    string strings[sid] at column string_col[sid]."""
    gene: np.ndarray
    codon_index: np.ndarray
    col: np.ndarray
    kind: np.ndarray                # 0 deletion, 1 insertion
    sid: np.ndarray
    ref_codon: np.ndarray
    next_codon: np.ndarray
    count: np.ndarray
    coverage: np.ndarray
    expected: np.ndarray
    ntests: np.ndarray
    pvalue: np.ndarray
    inserted: list
    label: list
    cnt: np.ndarray
    tally: np.ndarray
    strings: list
    string_col: np.ndarray


def translate_dna(x: str) -> str:
    """Amino acids of an in-frame string, '*' for a stop (the indel labels)."""
    return "".join(_AA[CODONS.index(x[i:i + 3])].replace("X", "*") for i in range(0, len(x) - 2, 3))


def indel_label(kind, ref_codon, next_codon, aa_pos, inserted):
    """D67del; T69_S70insSS (flanking reference amino acids, then the inserted ones).  A codon without a clean read is '?'."""
    aa = lambda c: translate(int(c)) if c >= 0 else "?"
    if kind == 0:
        return f"{aa(ref_codon)}{aa_pos}del"
    return f"{aa(ref_codon)}{aa_pos}_{aa(next_codon)}{aa_pos + 1}ins{translate_dna(inserted)}"


@dataclass
class JulietResult:
    variants: list = field(default_factory=list)     # list of ms_variant records
    keys: list = field(default_factory=list)         # pooled (start column, codon) list the haplotype bit-vectors refer to
    haplotypes: Haplotypes = None
    col_counts: np.ndarray = None
    codon_counts: np.ndarray = None


class Handle:
    """Thin RAII wrapper of ms_handle (one per GPU / rank)."""

    def __init__(self, device: int = 0):
        self.lib = _lib.load()
        h = C.c_void_p()
        rc = self.lib.ms_create(device, C.byref(h))
        if rc != 0:
            raise _lib.MsError(f"ms_create failed ({rc}): {self.lib.ms_last_error(None).decode()}")
        self.h = h
        self.device = device
        self.native_comm = False

    def close(self):
        if getattr(self, "h", None):
            self.lib.ms_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def attach_comm(self):
        """Give the handle its own NCCL communicator over the ranks of the initialised torch.distributed
        group (torch only carries the 128-byte unique id).  After this the count all-reduce and the
        haplotype-list all-gather run inside the library on the handle's stream."""
        import torch
        import torch.distributed as dist
        self.native_comm = False
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1 or dist.get_backend() != "nccl":
            return False
        ident = C.create_string_buffer(128)
        if dist.get_rank() == 0:
            rc = self.lib.ms_comm_unique_id(ident)
            if rc != 0:
                raise _lib.MsError(f"ms_comm_unique_id failed ({rc})")
        t = torch.frombuffer(bytearray(ident.raw), dtype=torch.uint8).to(f"cuda:{self.device}")
        dist.broadcast(t, src=0)
        ident = C.create_string_buffer(bytes(t.cpu().numpy().tobytes()), 128)
        check(self.lib.ms_comm_init(self.h, ident, dist.get_rank(), dist.get_world_size()), self.h)
        self.native_comm = True
        return True

    def use_torch_stream(self):
        import torch
        check(self.lib.ms_set_stream(self.h, C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)), self.h)

    @property
    def launches(self):
        return int(self.lib.ms_launch_count(self.h))


class Juliet:
    """juliet's pileup -> codon test -> phasing pass for one rank's shard of the reads."""

    def __init__(self, L, genes, refseq=None, device=0, region=None, mode_phasing=False, min_perc=None,
                 max_perc=None, substitution_rate=5e-4, deletion_rate=3e-3, alpha=0.01, min_hap_reads=10,
                 handle=None):
        self.hd = handle or Handle(device)
        self.lib = self.hd.lib
        self.L = int(L)
        self.genes = [(int(b), int(e)) for (b, e) in genes]
        self.refseq = refseq
        self.region = region
        self.mode_phasing = mode_phasing
        self.min_hap_reads = min_hap_reads
        p = CallParams()
        self.lib.ms_call_params_default(C.byref(p))
        p.substitution_rate, p.deletion_rate, p.alpha = substitution_rate, deletion_rate, alpha
        p.min_perc = -1.0 if min_perc is None else float(min_perc)
        p.max_perc = -1.0 if max_perc is None else float(max_perc)
        if region:
            p.region_begin, p.region_end = int(region[0]), int(region[1])
        self.params = p
        self.start_mask = start_mask_words(self.L, self.genes, region)
        check(self.lib.ms_set_layout(self.hd.h, self.L, _ptr(self.start_mask)), self.hd.h)

    @property
    def row_words(self):
        return int(self.lib.ms_row_words(self.L))

    def reset(self):
        check(self.lib.ms_reset_counts(self.hd.h), self.hd.h)

    def set_count_insertions(self, on: bool):
        """juliet ignores insertions (doc/JULIET.md:26-27); turn the tally on to get col[:, 6] as well."""
        check(self.lib.ms_set_count_insertions(self.hd.h, 1 if on else 0), self.hd.h)

    # -- K1
    def pileup_device(self, d_packed_ptr: int, nreads: int):
        check(self.lib.ms_pileup_dev(self.hd.h, C.c_void_p(d_packed_ptr), nreads), self.hd.h)

    def pileup_host(self, packed: np.ndarray) -> int:
        """packed: [R, row_words] uint32 host array (pinned recommended). Returns device ptr of the upload."""
        keep = C.c_void_p()
        check(self.lib.ms_pileup_host(self.hd.h, _ptr(packed), packed.shape[0], C.byref(keep)), self.hd.h)
        return keep.value

    def counts_tensor(self):
        """torch view of the device count tensor [L*72] (int32 reinterpretation for NCCL)."""
        import torch
        p, n = C.c_void_p(), C.c_int64()
        check(self.lib.ms_counts_device(self.hd.h, C.byref(p), C.byref(n)), self.hd.h)
        return _as_tensor(p.value, (n.value,), torch.int32, self.hd.device)

    def allreduce_counts(self):
        """The path's one data-path collective: integer sum of the count tensor over the ranks.
        The handle works on its own non-blocking stream, NCCL on torch's: the hand-over is two host
        synchronisations (tens of microseconds), which keeps the legacy default stream and NCCL's
        internal streams out of each other's way."""
        import torch
        import torch.distributed as dist
        if getattr(self.hd, "native_comm", False):
            check(self.lib.ms_allreduce_counts(self.hd.h), self.hd.h)   # ncclAllReduce on the handle's stream
            return
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            check(self.lib.ms_synchronize(self.hd.h), self.hd.h)
            dist.all_reduce(self.counts_tensor(), op=dist.ReduceOp.SUM)
            if dist.get_backend() == "nccl":
                torch.cuda.current_stream(self.hd.device).synchronize()

    def get_counts(self):
        col = np.empty((self.L, 8), dtype=np.uint32)
        codon = np.empty((self.L, 64), dtype=np.uint32)
        check(self.lib.ms_get_counts(self.hd.h, _ptr(col), _ptr(codon)), self.hd.h)
        return col, codon

    def context(self, col_counts: np.ndarray, col: int):
        """The 9-row MSA context juliet shows under a variant (rows -3..+5 around the codon's first
        column; doc/JULIET.md:99-100, screenshot juliet_hiv-context.png): list of (rel, A, C, G, T, -, N)."""
        rows = []
        for rel in range(-3, 6):
            j = col + rel
            if 0 <= j < self.L:
                rows.append((rel,) + tuple(int(x) for x in col_counts[j, :6]))
        return rows

    # -- K2
    def call(self, cap=1024):
        if getattr(self, "_call_cap", 0) < cap:          # ctypes buffers are reused from pass to pass
            self._call_cap = cap
            self._call_out = (Variant * cap)()
            self._call_genes = (Gene * len(self.genes))(*[Gene(b, e) for (b, e) in self.genes])
        cap, out = self._call_cap, self._call_out
        n = C.c_int64()
        ref = self.refseq.encode() if self.refseq else None
        check(self.lib.ms_call(self.hd.h, self._call_genes, len(self.genes), ref, C.byref(self.params), out, cap, C.byref(n)), self.hd.h)
        if n.value > cap:
            return self.call(cap=int(n.value))
        return [Variant.from_buffer_copy(out[i]) for i in range(n.value)]

    # -- K3
    def phase_device(self, variants, d_packed_ptr: int, nreads: int, want_hap_id=True, host_merge=False, cap=4096,
                     linkage=False, abundance=False) -> Haplotypes:
        """linkage / abundance: also record which reads are clean at each key, for Juliet.linkage / Juliet.haplotype_abundance
        afterwards"""
        import torch.distributed as dist
        keys = sorted({(v.col, v.codon) for v in variants})
        V = len(keys)
        vc = np.array([k[0] for k in keys], dtype=np.int32)
        vd = np.array([k[1] for k in keys], dtype=np.int32)
        nw = max(1, (V + 31) // 32)
        self._V = V
        self._keys = keys
        self._nreported = None             # set when the device path below leaves per-read ranks on the device
        self._reported = None
        check(self.lib.ms_set_linkage(self.hd.h, 1 if linkage else 0), self.hd.h)
        check(self.lib.ms_set_abundance(self.hd.h, 1 if abundance else 0), self.hd.h)
        check(self.lib.ms_phase_begin(self.hd.h, _ptr(vc), _ptr(vd), V, nreads), self.hd.h)
        check(self.lib.ms_phase_dev(self.hd.h, C.c_void_p(d_packed_ptr), nreads), self.hd.h)
        if not host_merge and (getattr(self.hd, "native_comm", False) or _torch_world() == 1):
            hap = self._haplotypes_device(V, nw, nreads, want_hap_id, cap)
            self._reported = hap.patterns[:hap.nreported].copy()
            return hap, keys
        # torch.distributed exchange (e.g. gloo in the CPU tests): the three-call protocol with a host merge
        while True:
            if getattr(self, "_grp_shape", None) != (cap, nw):   # reused from pass to pass
                self._grp_shape = (cap, nw)
                self._grp_pat = np.zeros((cap, nw), dtype=np.uint32)
                self._grp_cnt = np.zeros(cap, dtype=np.uint64)
            pat, cnt = self._grp_pat, self._grp_cnt
            H, ctr = C.c_int64(), PhaseCounters()
            check(self.lib.ms_phase_groups(self.hd.h, _ptr(pat), _ptr(cnt), cap, C.byref(H), C.byref(ctr)), self.hd.h)
            if H.value <= cap:
                break
            cap = int(H.value)
        pat, cnt = pat[:H.value].copy(), cnt[:H.value].copy()
        marg = np.array([ctr.damaged, ctr.gaps, ctr.heteroduplex, ctr.partial], dtype=np.int64)
        if not getattr(self.hd, "native_comm", False) and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            pat, cnt, marg = _gather_groups(pat, cnt, marg, self.hd.device)   # torch.distributed fallback (e.g. gloo)
        pat = np.ascontiguousarray(pat)
        cnt = np.ascontiguousarray(cnt)
        Hm, nrep, c2 = C.c_int64(), C.c_int64(), PhaseCounters()
        check(self.lib.ms_haplotype_order(_ptr(pat), _ptr(cnt), len(cnt), V, self.min_hap_reads, C.byref(Hm),
                                          C.byref(nrep), C.byref(c2)))
        pat, cnt = pat[:Hm.value], cnt[:Hm.value]
        names = []
        buf = C.create_string_buffer(3)
        for i in range(nrep.value):
            self.lib.ms_haplotype_name(i, buf)
            names.append(buf.value.decode())
        counters = dict(reported=int(c2.reported), insufficient=int(c2.insufficient), damaged=int(marg[0]),
                        gaps=int(marg[1]), heteroduplex=int(marg[2]), partial=int(marg[3]))
        hap = None
        if want_hap_id:
            hap = np.empty(nreads, dtype=np.int32)
            check(self.lib.ms_phase_assign(self.hd.h, _ptr(pat), len(cnt), _ptr(hap)), self.hd.h)
        self._reported = pat[:nrep.value].copy()
        return Haplotypes(patterns=pat, counts=cnt, nreported=int(nrep.value), names=names, counters=counters, hap_id=hap), keys

    def _haplotypes_device(self, V, nw, nreads, want_hap_id, cap=4096) -> Haplotypes:
        """grouping + merge over ranks + order + per-read ids in one C-ABI call (ms_phase_haplotypes)"""
        while True:
            if getattr(self, "_grp_shape", None) != (cap, nw):   # reused from pass to pass
                self._grp_shape = (cap, nw)
                self._grp_pat = np.zeros((cap, nw), dtype=np.uint32)
                self._grp_cnt = np.zeros(cap, dtype=np.uint64)
            pat, cnt = self._grp_pat, self._grp_cnt
            H, nrep, ctr = C.c_int64(), C.c_int64(), PhaseCounters()
            hap = np.empty(nreads, dtype=np.int32) if want_hap_id else None
            check(self.lib.ms_phase_haplotypes(self.hd.h, self.min_hap_reads, _ptr(pat), _ptr(cnt), cap, C.byref(H), C.byref(nrep), C.byref(ctr),
                                               _ptr(hap) if want_hap_id else None), self.hd.h)
            if nrep.value <= cap:
                break
            cap = int(nrep.value)
        k = min(cap, int(H.value))
        self._nreported = int(nrep.value)
        names = []
        buf = C.create_string_buffer(3)
        for i in range(nrep.value):
            self.lib.ms_haplotype_name(i, buf)
            names.append(buf.value.decode())
        counters = dict(reported=int(ctr.reported), insufficient=int(ctr.insufficient), damaged=int(ctr.damaged), gaps=int(ctr.gaps),
                        heteroduplex=int(ctr.heteroduplex), partial=int(ctr.partial))
        return Haplotypes(patterns=pat[:k].copy(), counts=cnt[:k].copy(), nreported=int(nrep.value), names=names, counters=counters, hap_id=hap,
                          ndistinct=int(H.value))

    def cooccurrence(self):
        """[V, V] int32 torch tensor (device memory owned by the handle), summed over ranks."""
        import torch
        import torch.distributed as dist
        p = C.c_void_p()
        check(self.lib.ms_cooccurrence(self.hd.h, C.byref(p)), self.hd.h)
        t = _as_tensor(p.value, (max(1, self._V * self._V),), torch.int32, self.hd.device)
        check(self.lib.ms_synchronize(self.hd.h), self.hd.h)
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            torch.cuda.current_stream(self.hd.device).synchronize()
        return t[: self._V * self._V].view(self._V, self._V)

    def linkage(self, alpha=None, min_reads=10, cap=1024) -> Linkage:
        """Pairwise linkage of the keys of the last phase_device(..., linkage=True) (ms_linkage): the pairs that are
        significantly "linked" (relation 1) or "exclusive" (relation 2) after Bonferroni over the tested pairs, and the dense
        counts.  alpha None = the codon test's alpha.  With several ranks the handle needs its own communicator
        (Handle.attach_comm): the counts are summed inside the library."""
        import torch
        if not getattr(self.hd, "native_comm", False) and _torch_world() > 1:
            raise _lib.MsError("linkage over several ranks needs the handle's own communicator (Handle.attach_comm)")
        p = LinkageParams()
        self.lib.ms_linkage_params_default(C.byref(p))
        p.alpha = self.params.alpha if alpha is None else float(alpha)
        p.min_reads = int(min_reads)
        n, m = C.c_int64(), C.c_int64()
        while True:
            out = (LinkagePair * max(1, cap))()
            check(self.lib.ms_linkage(self.hd.h, C.byref(p), out, cap, C.byref(n), C.byref(m)), self.hd.h)
            if n.value <= cap:
                break
            cap = int(n.value)             # the counts are cached: only the statistics run again
        rec = np.ctypeslib.as_array(out)[: n.value].copy()
        g, dim = C.c_void_p(), C.c_int32()
        check(self.lib.ms_linkage_device(self.hd.h, C.byref(g), C.byref(dim)), self.hd.h)
        check(self.lib.ms_synchronize(self.hd.h), self.hd.h)
        G = _as_tensor(g.value, (dim.value, dim.value), torch.int32, self.hd.device).cpu().numpy().astype(np.int64)
        V, h = self._V, dim.value // 2
        a = G[:V, :V]
        return Linkage(v=rec["v"], w=rec["w"], both=rec["both"], v_only=rec["v_only"], w_only=rec["w_only"], neither=rec["neither"],
                       d_prime=rec["d_prime"], r2=rec["r2"], pvalue=rec["pvalue"], relation=rec["relation"], ntested=int(m.value),
                       keys=list(self._keys), n=G[h:h + V, h:h + V].copy(), a=a.copy(), b=G[:V, h:h + V] - a, c=G[h:h + V, :V] - a)

    def haplotype_abundance(self, patterns=None, tol=1e-10, max_iter=10000) -> Abundance:
        """Haplotype abundance over every phased read of the last phase_device(..., abundance=True) (ms_haplotype_abundance,
        restatement choice U18).  patterns: [H, ceil(V/32)] uint32 phasing patterns, distinct; None = the reported haplotypes
        of that phasing, in report order.  With several ranks the handle needs its own communicator (Handle.attach_comm) and
        every rank passes the same patterns."""
        if not getattr(self.hd, "native_comm", False) and _torch_world() > 1:
            raise _lib.MsError("haplotype abundance over several ranks needs the handle's own communicator (Handle.attach_comm)")
        if patterns is None:
            patterns = getattr(self, "_reported", None)
            if patterns is None:
                raise _lib.MsError("haplotype_abundance needs the haplotypes of a phase_device call on this handle")
        nw = max(1, (getattr(self, "_V", 0) + 31) // 32)
        pat = np.ascontiguousarray(np.asarray(patterns, dtype=np.uint32).reshape(-1, nw))
        H = pat.shape[0]
        p = AbundanceParams()
        self.lib.ms_abundance_params_default(C.byref(p))
        p.tolerance, p.max_iterations = float(tol), int(max_iter)
        rows = (AbundanceRow * max(1, H))()
        ctr = AbundanceCounters()
        it, conv, ll = C.c_int32(), C.c_int32(), C.c_double()
        check(self.lib.ms_haplotype_abundance(self.hd.h, C.byref(p), _ptr(pat) if H else None, H, rows, H, C.byref(ctr), C.byref(it),
                                              C.byref(conv), C.byref(ll)), self.hd.h)
        rec = np.ctypeslib.as_array(rows)[:H]
        counters = dict(unique=int(ctr.unique), ambiguous=int(ctr.ambiguous), uninformative=int(ctr.uninformative),
                        incompatible=int(ctr.incompatible))
        return Abundance(unique_reads=rec["unique_reads"].copy(), compatible_reads=rec["compatible_reads"].copy(),
                         em_frequency=rec["em_frequency"].copy(), counters=counters, reads_used=counters["unique"] + counters["ambiguous"],
                         iterations=int(it.value), converged=bool(conv.value), log_likelihood=float(ll.value), tolerance=float(tol),
                         max_iterations=int(max_iter))

    # -- in-frame indels (restatement choice U19)
    def indels(self, d_packed_ptr: int, nreads: int, insertions=None, read0=0, deletion_rate=None, insertion_rate=3e-3,
               alpha=None, min_perc=None, max_perc=None, cap=256) -> Indels:
        """In-frame codon deletions and insertions of the reads that were piled up (ms_indel_count_dev + ms_indel_call): needs
        the all-reduced K1 counts of the same reads.  d_packed_ptr / nreads: this rank's reads (device tiles), reads
        [read0, read0 + nreads) of the run.  insertions: (read, col, off, len, pool) insertion events of ALL the run's reads
        (read in the run's numbering, pool = bytes), in ms_expand_cigar's order.  The rates, alpha and the percentage filters
        default to the codon test's.  With several ranks the handle needs its own communicator (Handle.attach_comm)."""
        if not getattr(self.hd, "native_comm", False) and _torch_world() > 1:
            raise _lib.MsError("indels over several ranks need the handle's own communicator (Handle.attach_comm)")
        nins, ir, ic, io, il, pl, pool = 0, None, None, None, None, None, b""
        if insertions is not None and len(insertions[0]):
            read, col, off, ln, pool = insertions
            ir = np.ascontiguousarray(read, dtype=np.int64)
            ic = np.ascontiguousarray(col, dtype=np.int32)
            io = np.ascontiguousarray(off, dtype=np.int64)
            il = np.ascontiguousarray(ln, dtype=np.int32)
            pl = np.frombuffer(pool, dtype=np.uint8)
            nins = len(ir)
        check(self.lib.ms_indel_count_dev(self.hd.h, C.c_void_p(d_packed_ptr), int(nreads), int(read0), _ptr(ir), _ptr(ic), _ptr(io), _ptr(il),
                                          nins, _ptr(pl), len(pool)), self.hd.h)
        p = IndelParams()
        self.lib.ms_indel_params_default(C.byref(p))
        p.deletion_rate = self.params.deletion_rate if deletion_rate is None else float(deletion_rate)
        p.insertion_rate = float(insertion_rate)
        p.alpha = self.params.alpha if alpha is None else float(alpha)
        p.min_perc = self.params.min_perc if min_perc is None else float(min_perc)
        p.max_perc = self.params.max_perc if max_perc is None else float(max_perc)
        p.region_begin, p.region_end = self.params.region_begin, self.params.region_end
        genes = (Gene * max(1, len(self.genes)))(*[Gene(b, e) for (b, e) in self.genes])
        ref = self.refseq.encode() if self.refseq else None
        n = C.c_int64()
        while True:
            out = (Indel * max(1, cap))()
            rc = self.lib.ms_indel_call(self.hd.h, genes, len(self.genes), ref, C.byref(p), out, cap, C.byref(n))
            if rc == -4:   # MS_ERR_CAPACITY: the counts are kept, only the test runs again
                cap = int(n.value)
                continue
            check(rc, self.hd.h)
            break
        rec = np.ctypeslib.as_array(out)[: n.value].copy()
        cnt = np.empty((self.L, 2), dtype=np.uint32)
        ns = C.c_int64()
        check(self.lib.ms_indel_counts(self.hd.h, _ptr(cnt), None, 0, C.byref(ns)), self.hd.h)
        tally = np.zeros(max(1, ns.value), dtype=np.uint32)
        check(self.lib.ms_indel_counts(self.hd.h, _ptr(cnt), _ptr(tally), ns.value, C.byref(ns)), self.hd.h)
        strings, scol = [], np.zeros(ns.value, dtype=np.int32)
        for sid in range(ns.value):
            c, ln = C.c_int32(), C.c_int64()
            buf = C.create_string_buffer(self.L + 1)
            rc = self.lib.ms_indel_inserted(self.hd.h, sid, C.byref(c), buf, len(buf), C.byref(ln))
            if rc == -4:
                buf = C.create_string_buffer(int(ln.value))
                rc = self.lib.ms_indel_inserted(self.hd.h, sid, C.byref(c), buf, len(buf), C.byref(ln))
            check(rc, self.hd.h)
            strings.append(buf.raw[: ln.value].decode())
            scol[sid] = c.value
        ins = [strings[s] if k == 1 else "" for k, s in zip(rec["kind"], rec["sid"])]
        labels = [indel_label(int(r["kind"]), int(r["ref_codon"]), int(r["next_codon"]), int(r["codon_index"]) + 1, x) for r, x in zip(rec, ins)]
        return Indels(gene=rec["gene"], codon_index=rec["codon_index"], col=rec["col"], kind=rec["kind"], sid=rec["sid"],
                      ref_codon=rec["ref_codon"], next_codon=rec["next_codon"], count=rec["count"], coverage=rec["coverage"],
                      expected=rec["expected"], ntests=rec["ntests"], pvalue=rec["pvalue"], inserted=ins, label=labels, cnt=cnt,
                      tally=tally[: ns.value].copy(), strings=strings, string_col=scol)

    # -- grouped pile-up and per-haplotype consensus (restatement choice U15)
    def group_pileup(self, d_packed_ptr: int, d_group_ptr: int, nreads: int, ngroups: int, accumulate=False):
        """K1's column counts per group of reads (ms_group_pileup_dev): read r of the device tiles is counted into group
        g = label[r] (d_group_ptr: device int32, one per read) when 0 <= g < ngroups and skipped otherwise.  accumulate=False
        starts from zero counts; True adds to the counts of the previous call with the same ngroups."""
        if accumulate and getattr(self, "_ngroups", None) != ngroups:
            raise ValueError("accumulate=True needs a previous group_pileup with the same ngroups")
        if not accumulate:
            check(self.lib.ms_set_groups(self.hd.h, int(ngroups)), self.hd.h)
            self._ngroups = int(ngroups)
        check(self.lib.ms_group_pileup_dev(self.hd.h, C.c_void_p(d_packed_ptr), C.c_void_p(d_group_ptr), int(nreads)), self.hd.h)

    def group_counts(self) -> np.ndarray:
        """[ngroups, L, 8] uint32: A, C, G, T, -, N, insertion flags and coverage of each group's reads (after haplotype_consensus:
        summed over the ranks)."""
        out = np.empty((self._ngroups, self.L, 8), dtype=np.uint32)
        check(self.lib.ms_get_group_counts(self.hd.h, _ptr(out)), self.hd.h)
        return out

    def haplotype_consensus(self, d_packed_ptr: int, nreads: int, insertions=None, min_coverage=10, ins_fraction=0.5,
                            ins_distance=20) -> list:
        """The sequence of every reported haplotype of the last phase_device, in report order (restatement choice U15): fuse's
        consensus over the haplotype's reads, with columns of fewer than min_coverage votes inside the covered span written as
        'N'.  d_packed_ptr / nreads: the reads that were phased.  insertions: (read, col, off, len, pool) insertion events of
        these reads (read = index among them, pool = bytes); each event belongs to its read's haplotype.  With several ranks
        the handle needs its own communicator (Handle.attach_comm), the counts are summed inside the library, and insertion
        events are not supported (their read indices are local to a rank)."""
        import torch
        if not getattr(self.hd, "native_comm", False) and _torch_world() > 1:
            raise _lib.MsError("haplotype consensus over several ranks needs the handle's own communicator (Handle.attach_comm)")
        nrep = getattr(self, "_nreported", None)
        if nrep is None:
            raise _lib.MsError("haplotype_consensus needs the per-read haplotype ranks of a phase_device call on this handle")
        d_hap, R = C.c_void_p(), C.c_int64()
        check(self.lib.ms_phase_hap_device(self.hd.h, C.byref(d_hap), C.byref(R)), self.hd.h)
        if R.value != nreads:
            raise ValueError(f"{nreads} reads given, {R.value} were phased")
        self.group_pileup(d_packed_ptr, d_hap.value or 0, nreads, nrep)
        check(self.lib.ms_allreduce_group_counts(self.hd.h), self.hd.h)
        nins, ig, ic, io, il, pool = 0, None, None, None, None, b""
        if insertions is not None and len(insertions[0]):
            if _torch_world() > 1:
                raise _lib.MsError("haplotype_consensus: insertion events are not supported with several ranks")
            read, col, off, ln, pool = insertions
            read = np.asarray(read, dtype=np.int64)
            if read.min() < 0 or read.max() >= nreads:
                raise ValueError("insertion read index outside the phased reads")
            check(self.lib.ms_synchronize(self.hd.h), self.hd.h)
            hap = _as_tensor(d_hap.value, (max(1, nreads),), torch.int32, self.hd.device).cpu().numpy()[:nreads]
            ig = np.ascontiguousarray(hap[read], dtype=np.int32)
            ic = np.ascontiguousarray(col, dtype=np.int32)
            io = np.ascontiguousarray(off, dtype=np.int64)
            il = np.ascontiguousarray(ln, dtype=np.int32)
            nins = len(ig)
        pl = np.frombuffer(pool, dtype=np.uint8) if nins else None
        prm = FuseParams(int(min_coverage), float(ins_fraction), int(ins_distance))
        seq_off = np.zeros(nrep + 1, dtype=np.int64)
        cap = nrep * (self.L + 16)
        while True:
            seq = np.empty(max(1, cap), dtype=np.uint8)
            rc = self.lib.ms_group_consensus(self.hd.h, C.byref(prm), _ptr(ig), _ptr(ic), _ptr(io), _ptr(il), nins, _ptr(pl), len(pool),
                                             _ptr(seq), cap, _ptr(seq_off))
            if rc == -4:   # MS_ERR_CAPACITY: seq_off holds the size
                cap = int(seq_off[-1])
                continue
            check(rc, self.hd.h)
            break
        return [seq[seq_off[g]: seq_off[g + 1]].tobytes().decode() for g in range(nrep)]

    # -- the whole pass in one C-ABI call (what bench.py times)
    @staticmethod
    def _hap_names(n):
        """[A-Z][a-z]? in rank order (doc/JULIET.md:198; ms_haplotype_name)"""
        return [chr(65 + i) if i < 26 else chr(65 + ((i - 26) // 26) % 26) + chr(97 + (i - 26) % 26) for i in range(n)]

    def _pass(self, ptr, nreads, host, want_hap_id, events=None):
        from ._lib import JulietResult as _JR
        st = getattr(self, "_pass_state", None)
        if st is None:
            st = self._pass_state = dict(vcap=1024, kcap=1024, pcap=4096)
        while True:
            sig = (st["vcap"], st["kcap"], st["pcap"], self.mode_phasing, self.min_hap_reads, self.refseq, tuple(self.genes))
            if st.get("alloc") != sig:          # ctypes buffers and the argument tail are reused from pass to pass
                st["alloc"] = sig
                st["var"] = (Variant * st["vcap"])()
                st["kc"] = np.zeros(st["kcap"], dtype=np.int32)
                st["kk"] = np.zeros(st["kcap"], dtype=np.int32)
                st["pat"] = np.zeros(st["pcap"] * ((st["kcap"] + 31) // 32), dtype=np.uint32)
                st["cnt"] = np.zeros(st["pcap"], dtype=np.uint64)
                st["genes"] = (Gene * len(self.genes))(*[Gene(b, e) for (b, e) in self.genes])
                st["ref"] = self.refseq.encode() if self.refseq else None
                r = st["res"] = _JR()
                r.variants = st["var"]; r.variants_cap = st["vcap"]
                r.key_col = st["kc"].ctypes.data_as(C.POINTER(C.c_int32)); r.key_codon = st["kk"].ctypes.data_as(C.POINTER(C.c_int32)); r.keys_cap = st["kcap"]
                r.patterns = st["pat"].ctypes.data_as(C.POINTER(C.c_uint32)); r.counts = st["cnt"].ctypes.data_as(C.POINTER(C.c_uint64)); r.patterns_cap = st["pcap"]
                st["tail"] = (st["genes"], len(self.genes), st["ref"], C.byref(self.params), 1 if self.mode_phasing else 0, self.min_hap_reads, C.byref(r))
            r = st["res"]
            hap = np.empty(nreads, dtype=np.int32) if (want_hap_id and self.mode_phasing) else None
            r.hap_id = hap.ctypes.data_as(C.POINTER(C.c_int32)) if hap is not None else None
            if events is not None:
                rc = self.lib.ms_juliet_pass_events_host(self.hd.h, ptr, events.ctypes.data, nreads, *st["tail"])
            else:
                fn = self.lib.ms_juliet_pass_host if host else self.lib.ms_juliet_pass_dev
                rc = fn(self.hd.h, ptr, nreads, *st["tail"])
            if rc == -4:   # MS_ERR_CAPACITY: grow what was too small and run the pass again
                st["vcap"] = max(st["vcap"], int(r.nvariants)); st["kcap"] = max(st["kcap"], int(r.nkeys)); st["pcap"] = max(st["pcap"], int(r.nreported))
                continue
            check(rc, self.hd.h)
            break
        nv = int(r.nvariants)
        res = JulietResult(variants=list((Variant * nv).from_buffer_copy(st["var"])) if nv else [])
        V = int(r.nkeys)
        res.keys = list(zip(st["kc"][:V].tolist(), st["kk"][:V].tolist()))
        if self.mode_phasing:
            self._V = V
            nw = max(1, (V + 31) // 32)
            H = min(int(r.npatterns), st["pcap"])
            pat = st["pat"][: H * nw].reshape(H, nw).copy()
            cnt = st["cnt"][:H].copy()
            c = r.counters
            counters = dict(reported=int(c.reported), insufficient=int(c.insufficient), damaged=int(c.damaged), gaps=int(c.gaps),
                            heteroduplex=int(c.heteroduplex), partial=int(c.partial))
            res.haplotypes = Haplotypes(patterns=pat, counts=cnt, nreported=int(r.nreported), names=self._hap_names(int(r.nreported)),
                                        counters=counters, hap_id=hap, ndistinct=int(r.npatterns))
        return res

    def run_device(self, d_packed_ptr: int, nreads: int, want_hap_id=False) -> JulietResult:
        """pileup -> all-reduce -> call -> phase on device-resident packed reads (one C-ABI call)."""
        if not getattr(self.hd, "native_comm", False) and _torch_world() > 1:
            return self._run_staged(d_packed_ptr, nreads, want_hap_id)     # torch.distributed exchange between the stages
        return self._pass(d_packed_ptr, nreads, False, want_hap_id)

    # -- event rows (the compact host->device form, csrc/events.cu)
    def set_base(self, base):
        """base: the sequence the event rows are encoded against -- a string over ACGT or an array of 0..3, L long
        (the configured referenceSequence, or any sequence close to the reads)."""
        self.base = base_array(base, self.L)
        check(self.lib.ms_set_base(self.hd.h, _ptr(self.base)), self.hd.h)

    def run_events_host(self, hdr: np.ndarray, events: np.ndarray, want_hap_id=False) -> JulietResult:
        """Reference-facing call with HOST event rows (encode_rows / encode_states): H2D of the events, expansion on the GPU,
        pileup -> call -> phase, D2H of the results (one C-ABI call, ms_juliet_pass_events_host)."""
        if not getattr(self.hd, "native_comm", False) and _torch_world() > 1:
            self.reset()
            keep = C.c_void_p()
            check(self.lib.ms_pileup_events_host(self.hd.h, _ptr(hdr), _ptr(events), len(hdr) - 1, C.byref(keep)), self.hd.h)
            return self._run_staged(keep.value, len(hdr) - 1, want_hap_id, piled=True)
        return self._pass(hdr.ctypes.data, len(hdr) - 1, True, want_hap_id, events=events)

    def run_host(self, packed: np.ndarray, want_hap_id=False) -> JulietResult:
        """Reference-facing call with HOST buffers: H2D + kernels + D2H of the results (one C-ABI call)."""
        if not getattr(self.hd, "native_comm", False) and _torch_world() > 1:
            self.reset()
            dptr = self.pileup_host(packed)
            return self._run_staged(dptr, packed.shape[0], want_hap_id, piled=True)
        return self._pass(packed.ctypes.data, packed.shape[0], True, want_hap_id)

    def _run_staged(self, d_packed_ptr, nreads, want_hap_id, piled=False) -> JulietResult:
        if not piled:
            self.reset()
            self.pileup_device(d_packed_ptr, nreads)
        self.allreduce_counts()
        res = JulietResult(variants=self.call())
        if self.mode_phasing:
            res.haplotypes, res.keys = self.phase_device(res.variants, d_packed_ptr, nreads, want_hap_id)
        return res

    def variant_dicts(self, variants):
        out = []
        for v in variants:
            out.append(dict(gene=v.gene, aa_pos=v.codon_index + 1, col=v.col, ref_codon=CODONS[v.ref_codon],
                            ref_aa=translate(v.ref_codon), codon=CODONS[v.codon], aa=translate(v.codon),
                            count=int(v.count), coverage=int(v.coverage), frequency=v.count / v.coverage,
                            expected=int(v.expected), ntests=int(v.ntests), pvalue=float(v.pvalue)))
        return out


class Fuse:
    """fuse's consensus for one rank's shard (doc/FUSE.md:17-24)."""

    def __init__(self, L, device=0, min_coverage=50, ins_fraction=0.5, ins_distance=20, handle=None):
        self.hd = handle or Handle(device)
        self.lib = self.hd.lib
        self.L = int(L)
        self.params = FuseParams(min_coverage, ins_fraction, ins_distance)
        check(self.lib.ms_set_layout(self.hd.h, self.L, None), self.hd.h)

    def pileup_device(self, d_packed_ptr: int, nreads: int):
        check(self.lib.ms_pileup_dev(self.hd.h, C.c_void_p(d_packed_ptr), nreads), self.hd.h)

    def pileup_host(self, packed: np.ndarray) -> int:
        keep = C.c_void_p()
        check(self.lib.ms_pileup_host(self.hd.h, _ptr(packed), packed.shape[0], C.byref(keep)), self.hd.h)
        return keep.value

    allreduce_counts = Juliet.allreduce_counts
    counts_tensor = Juliet.counts_tensor
    set_base = Juliet.set_base

    def reset(self):
        check(self.lib.ms_reset_counts(self.hd.h), self.hd.h)

    def consensus(self, ins_col=None, ins_off=None, ins_len=None, ins_pool=b"") -> str:
        nins = 0 if ins_col is None else len(ins_col)
        ic = np.ascontiguousarray(ins_col, dtype=np.int32) if nins else None
        io = np.ascontiguousarray(ins_off, dtype=np.int64) if nins else None
        il = np.ascontiguousarray(ins_len, dtype=np.int32) if nins else None
        pool = np.frombuffer(ins_pool, dtype=np.uint8) if nins else None
        cap = self.L + (int(il.sum()) if nins else 0) + 16
        seq = np.empty(cap, dtype=np.uint8)
        n = C.c_int64()
        check(self.lib.ms_fuse(self.hd.h, C.byref(self.params), _ptr(ic), _ptr(io), _ptr(il), nins, _ptr(pool),
                               len(ins_pool), _ptr(seq), cap, C.byref(n)), self.hd.h)
        return seq[: n.value].tobytes().decode()


def device_rows(packed: np.ndarray, device=0):
    """[R, row_words] plain host rows -> int32 torch tensor on the GPU in the device tile layout (csrc/rows.cuh), i.e. what
    pileup_device / phase_device / run_device take.  ceil(R/8) whole tiles."""
    import torch
    packed = np.ascontiguousarray(packed, dtype=np.uint32)
    if packed.shape[0] == 0:
        return torch.zeros(max(1, packed.shape[1]) * 8, dtype=torch.int32, device=f"cuda:{device}")
    return torch.from_numpy(tile_rows(packed).view(np.int32)).to(f"cuda:{device}")


def host_rows(d_tiled, R: int, L: int) -> np.ndarray:
    """device tile tensor -> [R, row_words] plain uint32 rows on the host (tests, fixtures)"""
    return untile_rows(d_tiled.reshape(-1).cpu().numpy().view(np.uint32), R, L)


def synth_device(hd, tables, read0: int, R: int, device=None):
    """R synthetic reads [read0, read0+R) of `tables` written on the GPU in the device tile layout (ms_synth_dev);
    returns the int32 torch tensor (ceil(R/8) whole tiles)."""
    import torch
    lib = hd.lib
    L = tables.cfg.L
    dev = hd.device if device is None else device
    out = torch.empty(max(8, int(lib.ms_tiled_words(L, max(R, 1)))), dtype=torch.int32, device=f"cuda:{dev}")
    sp = SynthParams(tables.cfg.seed, L, tables.nstrains, tables.thr_N, tables.thr_sub, tables.thr_ins20, tables.thr_trunc16)
    check(lib.ms_synth_dev(hd.h, C.byref(sp), tables.strain_base.ctypes.data_as(C.c_void_p), tables.thr_del.ctypes.data_as(C.c_void_p),
                           tables.strain_cum.ctypes.data_as(C.c_void_p), read0, R, C.c_void_p(out.data_ptr())), hd.h)
    return out


HDR_DTYPE = np.dtype([("ev_off", "<u4"), ("begin", "<u2"), ("end", "<u2")])


def base_array(base, L):
    if isinstance(base, str):
        lut = np.full(256, 0, dtype=np.uint8)
        for i, ch in enumerate("ACGT"):
            lut[ord(ch)] = i
            lut[ord(ch.lower())] = i
        base = lut[np.frombuffer(base.encode(), dtype=np.uint8)]
    base = np.ascontiguousarray(base, dtype=np.uint8)
    if base.shape != (L,):
        raise ValueError(f"base sequence must have {L} entries")
    return base


def _encode(fn_name, src, R, L, base):
    """-> (hdr[R+1] structured array, event bytes: uint8 array, per read [nN u16][N list][12-bit rest list], include/minorseq_b200.h)"""
    lib = _lib.load()
    base = base_array(base, L)
    cap = max(1024, int(R) * 128)
    while True:
        hdr = np.zeros(R + 1, dtype=HDR_DTYPE)
        ev = np.empty(cap, dtype=np.uint8)
        n = C.c_int64()
        rc = getattr(lib, fn_name)(_ptr(src), R, L, _ptr(base), _ptr(hdr), _ptr(ev), cap, C.byref(n))
        if rc == -4:
            cap *= 4
            continue
        check(rc)
        return hdr, ev[: n.value].copy()


def encode_states(states: np.ndarray, base):
    """[R, L] uint8 column states -> event rows against `base` (ms_encode_states)."""
    states = np.ascontiguousarray(states, dtype=np.uint8)
    return _encode("ms_encode_states", states, states.shape[0], states.shape[1], base)


def encode_rows(packed: np.ndarray, L: int, base):
    """[R, row_words] uint32 planar rows -> event rows against `base` (ms_encode_rows)."""
    packed = np.ascontiguousarray(packed, dtype=np.uint32)
    return _encode("ms_encode_rows", packed, packed.shape[0], L, base)


def decode_events(hdr, events, L, base):
    """numpy decoder of the event-row format (tests only; the product expands on the GPU): -> [R, L] uint8 states."""
    base = base_array(base, L)
    R = len(hdr) - 1
    out = np.full((R, L), 7, dtype=np.uint8)
    for r in range(R):
        b, e = int(hdr["begin"][r]), int(hdr["end"][r])
        out[r, b:e] = base[b:e]
        raw = np.asarray(events[int(hdr["ev_off"][r]): int(hdr["ev_off"][r + 1])], dtype=np.uint8).astype(np.int64)
        if len(raw) < 2:
            continue                                              # no bytes: the read is the base on its whole span
        nN = int(raw[0] | (raw[1] << 8))
        d = raw[2: 2 + nN]                                        # N list: one byte per entry, 255 = move on by 255 columns
        out[r, (b + np.cumsum(d))[d != 255]] = 5
        rest = raw[2 + nN:]
        n = (2 * len(rest)) // 3                                  # ceil(1.5 n) bytes hold n 12-bit entries
        k = np.arange(n)
        o = (3 * k) >> 1
        two = rest[o] | (rest[np.minimum(o + 1, len(rest) - 1)] << 8) if n else np.zeros(0, dtype=np.int64)
        ev = np.where(k & 1, two >> 4, two & 0xFFF)
        cols = b + np.cumsum(ev >> 4)
        keep = (ev >> 4) != 255
        out[r, cols[keep]] = (ev[keep] & 15).astype(np.uint8)
    return out


def _torch_world():
    try:
        import torch.distributed as dist
        return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    except Exception:
        return 1


def _as_tensor(ptr, shape, dtype, device):
    """Zero-copy torch tensor over raw device memory owned by the handle."""
    import torch

    class _Holder:
        pass

    itemsize = torch.empty((), dtype=dtype).element_size()
    hold = _Holder()
    hold.__cuda_array_interface__ = {
        "shape": tuple(shape), "typestr": {4: "<i4", 8: "<i8", 1: "|u1"}[itemsize], "data": (int(ptr), False),
        "version": 2, "strides": None,
    }
    return torch.as_tensor(hold, device=f"cuda:{device}")


_GATHER_ROWS = 2048


def _gather_groups(pat, cnt, marg, device):
    """all-gather the ranks' (pattern, count) lists in ONE collective: every rank contributes a fixed
    block of _GATHER_ROWS rows whose row 0 is [n, damaged, gaps, heteroduplex, partial].  A rank with
    more than _GATHER_ROWS distinct patterns (the dense phasing stress case) triggers a second,
    exactly-sized exchange on all ranks.  The marginals are summed on the host."""
    import torch
    import torch.distributed as dist
    ws = dist.get_world_size()
    dev = f"cuda:{device}" if dist.get_backend() == "nccl" else "cpu"
    nw = pat.shape[1]
    cols = max(nw + 1, 5)

    def exchange(rows):
        host = np.zeros((rows + 1, cols), dtype=np.int64)
        host[0, 0] = len(cnt)
        host[0, 1:5] = marg
        k = min(len(cnt), rows)
        if k:
            host[1: 1 + k, :nw] = pat[:k]
            host[1: 1 + k, nw] = cnt[:k].astype(np.int64)
        buf = torch.from_numpy(host).to(dev)
        out = torch.empty((ws,) + tuple(buf.shape), dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(out, buf) if dev != "cpu" else dist.all_gather(list(out.unbind(0)), buf)
        return out.cpu().numpy()

    blocks = exchange(_GATHER_ROWS)
    need = int(blocks[:, 0, 0].max())
    if need > _GATHER_ROWS:
        blocks = exchange(need)
    pats, cnts, m = [], [], np.zeros(4, dtype=np.int64)
    for b in blocks:
        k = int(b[0, 0])
        m += b[0, 1:5]
        pats.append(b[1: 1 + k, :nw].astype(np.uint32))
        cnts.append(b[1: 1 + k, nw].astype(np.uint64))
    return np.concatenate(pats, axis=0), np.concatenate(cnts), m


CIGAR_OPS = "MIDNSHP=X"


class Aligner:
    """Overlap alignment of unaligned reads to one amplicon reference on the GPU (K6, restatement choice U16)."""

    def __init__(self, device=0, min_seeds=10, handle=None):
        self.hd = handle or Handle(device)
        self.lib = self.hd.lib
        self.params = AlignParams(int(min_seeds))

    def set_reference(self, ref: str):
        b = ref.encode()
        check(self.lib.ms_align_set_reference(self.hd.h, b, len(b)), self.hd.h)

    def align_raw(self, reads):
        """reads: list of str (native orientation).  Returns (ms_read_alignment array, u32 BAM-encoded CIGAR ops)."""
        seq = "".join(reads).encode()
        off = np.zeros(len(reads) + 1, dtype=np.int64)
        off[1:] = np.cumsum([len(r) for r in reads])
        out = (ReadAlignment * max(1, len(reads)))()
        cap = int(off[-1] // 8 + 16)
        while True:
            cig = np.zeros(cap, dtype=np.uint32)
            n = C.c_int64()
            rc = self.lib.ms_align_reads(self.hd.h, C.byref(self.params), seq, _ptr(off), len(reads), out, _ptr(cig), cap, C.byref(n))
            if rc == -4:   # MS_ERR_CAPACITY: n holds the number of ops
                cap = n.value
                continue
            check(rc, self.hd.h)
            return out, cig[:n.value]

    def align(self, reads):
        """list of (mapped, strand, pos, score, cigar string) in read order; unmapped reads are (False, 0, -1, 0, "")."""
        out, cig = self.align_raw(reads)
        res = []
        for r in range(len(reads)):
            a = out[r]
            ops = cig[a.cigar_off:a.cigar_off + a.ncigar]
            res.append((bool(a.mapped), int(a.strand), int(a.pos), int(a.score),
                        "".join(f"{int(x) >> 4}{CIGAR_OPS[int(x) & 15]}" for x in ops)))
        return res
