"""ctypes binding of libminorseq_b200.so (the C ABI in include/minorseq_b200.h).

There is no Python or CPU fallback: if the library is missing this module raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libminorseq_b200.so")

MS_OK = 0
FLAG_GAP, FLAG_HET, FLAG_PARTIAL = 1, 2, 4


class Gene(C.Structure):
    _fields_ = [("begin", C.c_int32), ("end", C.c_int32)]


class CallParams(C.Structure):
    _fields_ = [("substitution_rate", C.c_double), ("deletion_rate", C.c_double), ("alpha", C.c_double),
                ("min_perc", C.c_double), ("max_perc", C.c_double),
                ("region_begin", C.c_int32), ("region_end", C.c_int32)]


class Variant(C.Structure):
    _fields_ = [("gene", C.c_int32), ("codon_index", C.c_int32), ("col", C.c_int32), ("ref_codon", C.c_int32),
                ("codon", C.c_int32), ("count", C.c_uint32), ("coverage", C.c_uint32), ("expected", C.c_uint32),
                ("ntests", C.c_uint32), ("pvalue", C.c_double)]


class PhaseCounters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("reported", "insufficient", "damaged", "gaps", "heteroduplex", "partial")]


class FuseParams(C.Structure):
    _fields_ = [("min_coverage", C.c_int32), ("ins_fraction", C.c_double), ("ins_distance", C.c_int32)]


class JulietResult(C.Structure):
    _fields_ = [("variants", C.POINTER(Variant)), ("variants_cap", C.c_int64), ("nvariants", C.c_int64),
                ("key_col", C.POINTER(C.c_int32)), ("key_codon", C.POINTER(C.c_int32)), ("keys_cap", C.c_int32), ("nkeys", C.c_int32),
                ("patterns", C.POINTER(C.c_uint32)), ("counts", C.POINTER(C.c_uint64)), ("patterns_cap", C.c_int64),
                ("npatterns", C.c_int64), ("nreported", C.c_int64), ("counters", PhaseCounters), ("hap_id", C.POINTER(C.c_int32))]


class LinkageParams(C.Structure):
    _fields_ = [("alpha", C.c_double), ("min_reads", C.c_int32)]


class LinkagePair(C.Structure):
    _fields_ = [("v", C.c_int32), ("w", C.c_int32), ("both", C.c_uint32), ("v_only", C.c_uint32), ("w_only", C.c_uint32),
                ("neither", C.c_uint32), ("d_prime", C.c_double), ("r2", C.c_double), ("pvalue", C.c_double), ("relation", C.c_int32)]


class RareParams(C.Structure):
    _fields_ = [("candidate_alpha", C.c_double), ("min_reads", C.c_int32)]


class ControlVariant(C.Structure):
    _fields_ = [("gene", C.c_int32), ("codon_index", C.c_int32), ("col", C.c_int32), ("ref_codon", C.c_int32), ("codon", C.c_int32),
                ("count", C.c_uint32), ("coverage", C.c_uint32), ("control_count", C.c_uint32), ("control_coverage", C.c_uint32),
                ("ntests", C.c_uint32), ("called", C.c_int32), ("listed", C.c_int32), ("pvalue", C.c_double)]


class AbundanceParams(C.Structure):
    _fields_ = [("tolerance", C.c_double), ("max_iterations", C.c_int32)]


class AbundanceRow(C.Structure):
    _fields_ = [("unique_reads", C.c_uint64), ("compatible_reads", C.c_uint64), ("em_frequency", C.c_double)]


class AbundanceCounters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("unique", "ambiguous", "uninformative", "incompatible")]


class IndelParams(C.Structure):
    _fields_ = [("deletion_rate", C.c_double), ("insertion_rate", C.c_double), ("alpha", C.c_double), ("min_perc", C.c_double),
                ("max_perc", C.c_double), ("region_begin", C.c_int32), ("region_end", C.c_int32)]


class Indel(C.Structure):
    _fields_ = [("gene", C.c_int32), ("codon_index", C.c_int32), ("col", C.c_int32), ("kind", C.c_int32), ("sid", C.c_int32),
                ("ref_codon", C.c_int32), ("next_codon", C.c_int32), ("count", C.c_uint32), ("coverage", C.c_uint32),
                ("expected", C.c_uint32), ("ntests", C.c_uint32), ("pvalue", C.c_double)]


class ReadHdr(C.Structure):
    _fields_ = [("ev_off", C.c_uint32), ("begin", C.c_uint16), ("end", C.c_uint16)]


class AlignParams(C.Structure):
    _fields_ = [("min_seeds", C.c_int32)]


class ReadAlignment(C.Structure):
    _fields_ = [("mapped", C.c_int32), ("strand", C.c_int32), ("pos", C.c_int32), ("score", C.c_int32), ("cigar_off", C.c_int64),
                ("ncigar", C.c_int32)]


class SynthParams(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("L", C.c_int32), ("nstrains", C.c_int32), ("thr_N", C.c_uint32),
                ("thr_sub", C.c_uint32), ("thr_ins20", C.c_uint32), ("thr_trunc16", C.c_uint32)]


_P = C.c_void_p
_SIGNATURES = {
    "ms_row_words": (C.c_int32, [C.c_int32]),
    "ms_read_admitted": (C.c_int, [C.c_uint32]),
    "ms_pack_states": (C.c_int, [_P, C.c_int64, C.c_int32, _P]),
    "ms_unpack_states": (C.c_int, [_P, C.c_int64, C.c_int32, _P]),
    "ms_tiled_words": (C.c_int64, [C.c_int32, C.c_int64]),
    "ms_tile_rows": (C.c_int, [_P, C.c_int64, C.c_int32, _P]),
    "ms_untile_rows": (C.c_int, [_P, C.c_int64, C.c_int32, _P]),
    "ms_tile_rows_dev": (C.c_int, [_P, _P, C.c_int64, _P]),
    "ms_expand_cigar": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_char_p, _P, C.c_int32, C.c_int32, _P, _P, _P, _P,
                                  C.c_int64, _P, _P, C.c_int64, _P]),
    "ms_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "ms_destroy": (None, [_P]),
    "ms_last_error": (C.c_char_p, [_P]),
    "ms_set_stream": (C.c_int, [_P, _P]),
    "ms_synchronize": (C.c_int, [_P]),
    "ms_alloc_pinned": (_P, [C.c_size_t]),
    "ms_free_pinned": (None, [_P]),
    "ms_launch_count": (C.c_int64, [_P]),
    "ms_set_timing": (C.c_int, [_P, C.c_int]),
    "ms_timer_start": (C.c_int, [_P]),
    "ms_timer_stop": (C.c_int, [_P, C.POINTER(C.c_double)]),
    "ms_pileup_kernel_ms": (C.c_int, [_P, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "ms_stage_kernel_ms": (C.c_int, [_P, C.c_int, C.POINTER(C.c_double)]),
    "ms_set_layout": (C.c_int, [_P, C.c_int32, _P]),
    "ms_set_count_insertions": (C.c_int, [_P, C.c_int]),
    "ms_reset_counts": (C.c_int, [_P]),
    "ms_pileup_dev": (C.c_int, [_P, _P, C.c_int64]),
    "ms_pileup_host": (C.c_int, [_P, _P, C.c_int64, C.POINTER(_P)]),
    "ms_counts_device": (C.c_int, [_P, C.POINTER(_P), C.POINTER(C.c_int64)]),
    "ms_get_counts": (C.c_int, [_P, _P, _P]),
    "ms_set_pileup_variant": (C.c_int, [_P, C.c_int]),
    "ms_comm_unique_id": (C.c_int, [C.c_char_p]),
    "ms_comm_init": (C.c_int, [_P, C.c_char_p, C.c_int, C.c_int]),
    "ms_comm_size": (C.c_int, [_P]),
    "ms_allreduce_counts": (C.c_int, [_P]),
    "ms_call_params_default": (None, [C.POINTER(CallParams)]),
    "ms_call": (C.c_int, [_P, C.POINTER(Gene), C.c_int32, C.c_char_p, C.POINTER(CallParams), C.POINTER(Variant),
                          C.c_int64, C.POINTER(C.c_int64)]),
    "ms_phase_begin": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int64]),
    "ms_phase_dev": (C.c_int, [_P, _P, C.c_int64]),
    "ms_phase_groups": (C.c_int, [_P, _P, _P, C.c_int64, C.POINTER(C.c_int64), C.POINTER(PhaseCounters)]),
    "ms_haplotype_order": (C.c_int, [_P, _P, C.c_int64, C.c_int32, C.c_int32, C.POINTER(C.c_int64),
                                     C.POINTER(C.c_int64), C.POINTER(PhaseCounters)]),
    "ms_haplotype_name": (None, [C.c_int64, C.c_char_p]),
    "ms_phase_assign": (C.c_int, [_P, _P, C.c_int64, _P]),
    "ms_align_refs": (C.c_int, [_P, C.c_char_p, C.c_int32, C.c_char_p, C.c_int32, _P, C.c_int64, _P, _P]),
    "ms_align_params_default": (None, [C.POINTER(AlignParams)]),
    "ms_align_set_reference": (C.c_int, [_P, C.c_char_p, C.c_int32]),
    "ms_align_reads": (C.c_int, [_P, C.POINTER(AlignParams), C.c_char_p, _P, C.c_int64, _P, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "ms_set_cooccurrence_variant": (C.c_int, [_P, C.c_int32]),
    "ms_phase_haplotypes": (C.c_int, [_P, C.c_int32, _P, _P, C.c_int64, _P, _P, _P, _P]),
    "ms_phase_device": (C.c_int, [_P, C.POINTER(_P), C.POINTER(_P), C.POINTER(C.c_int64)]),
    "ms_cooccurrence": (C.c_int, [_P, C.POINTER(_P)]),
    "ms_linkage_params_default": (None, [C.POINTER(LinkageParams)]),
    "ms_set_linkage": (C.c_int, [_P, C.c_int]),
    "ms_linkage": (C.c_int, [_P, C.POINTER(LinkageParams), C.POINTER(LinkagePair), C.c_int64, C.POINTER(C.c_int64),
                             C.POINTER(C.c_int64)]),
    "ms_linkage_device": (C.c_int, [_P, C.POINTER(_P), C.POINTER(C.c_int32)]),
    "ms_abundance_params_default": (None, [C.POINTER(AbundanceParams)]),
    "ms_set_abundance": (C.c_int, [_P, C.c_int]),
    "ms_haplotype_abundance": (C.c_int, [_P, C.POINTER(AbundanceParams), _P, C.c_int64, C.POINTER(AbundanceRow), C.c_int64,
                                         C.POINTER(AbundanceCounters), C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_double)]),
    "ms_juliet_pass_dev": (C.c_int, [_P, _P, C.c_int64, C.POINTER(Gene), C.c_int32, C.c_char_p, C.POINTER(CallParams), C.c_int32,
                                   C.c_int32, C.POINTER(JulietResult)]),
    "ms_juliet_pass_host": (C.c_int, [_P, _P, C.c_int64, C.POINTER(Gene), C.c_int32, C.c_char_p, C.POINTER(CallParams), C.c_int32,
                                    C.c_int32, C.POINTER(JulietResult)]),
    "ms_events_bound": (C.c_int64, [C.c_int32]),
    "ms_encode_states": (C.c_int, [_P, C.c_int64, C.c_int32, _P, _P, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "ms_encode_rows": (C.c_int, [_P, C.c_int64, C.c_int32, _P, _P, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "ms_base_planes": (C.c_int, [_P, C.c_int32, _P]),
    "ms_encode_row": (C.c_int, [_P, C.c_int32, _P, _P, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "ms_events_seal": (C.c_int, [_P, C.c_int64, C.c_int64, _P, C.c_int32]),
    "ms_set_base": (C.c_int, [_P, _P]),
    "ms_expand_events_dev": (C.c_int, [_P, _P, _P, C.c_int64, _P]),
    "ms_pileup_events_host": (C.c_int, [_P, _P, _P, C.c_int64, C.POINTER(_P)]),
    "ms_juliet_pass_events_host": (C.c_int, [_P, _P, _P, C.c_int64, C.POINTER(Gene), C.c_int32, C.c_char_p, C.POINTER(CallParams), C.c_int32,
                                           C.c_int32, C.POINTER(JulietResult)]),
    "ms_fuse_params_default": (None, [C.POINTER(FuseParams)]),
    "ms_fuse": (C.c_int, [_P, C.POINTER(FuseParams), _P, _P, _P, C.c_int64, _P, C.c_int64, _P, C.c_int64,
                          C.POINTER(C.c_int64)]),
    "ms_synth_dev": (C.c_int, [_P, C.POINTER(SynthParams), _P, _P, _P, C.c_int64, C.c_int64, _P]),
    "ms_set_groups": (C.c_int, [_P, C.c_int32]),
    "ms_group_pileup_dev": (C.c_int, [_P, _P, _P, C.c_int64]),
    "ms_allreduce_group_counts": (C.c_int, [_P]),
    "ms_get_group_counts": (C.c_int, [_P, _P]),
    "ms_phase_hap_device": (C.c_int, [_P, C.POINTER(_P), C.POINTER(C.c_int64)]),
    "ms_group_consensus": (C.c_int, [_P, C.POINTER(FuseParams), _P, _P, _P, _P, C.c_int64, _P, C.c_int64, _P, C.c_int64, _P]),
    "ms_indel_params_default": (None, [C.POINTER(IndelParams)]),
    "ms_indel_count_dev": (C.c_int, [_P, _P, C.c_int64, C.c_int64, _P, _P, _P, _P, C.c_int64, _P, C.c_int64]),
    "ms_indel_counts": (C.c_int, [_P, _P, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "ms_indel_inserted": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_int32), _P, C.c_int64, C.POINTER(C.c_int64)]),
    "ms_indel_call": (C.c_int, [_P, C.POINTER(Gene), C.c_int32, C.c_char_p, C.POINTER(IndelParams), C.POINTER(Indel), C.c_int64,
                                C.POINTER(C.c_int64)]),
    "ms_phase_begin_indels": (C.c_int, [_P, _P, _P, C.c_int32, _P, C.c_int32, _P, C.c_int32, C.c_int64]),
    "ms_rare_params_default": (None, [C.POINTER(RareParams)]),
    "ms_rare_candidates": (C.c_int, [_P, C.POINTER(Gene), C.c_int32, C.c_char_p, C.POINTER(CallParams), C.POINTER(RareParams),
                                     C.POINTER(Variant), C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "ms_rare_linkage": (C.c_int, [_P, C.c_int32, C.POINTER(LinkageParams), C.POINTER(LinkagePair), C.c_int64, C.POINTER(C.c_int64),
                                  C.POINTER(C.c_int64)]),
    "ms_rare_support": (C.c_int, [_P, _P, C.c_int64, _P, _P]),
    "ms_rare_groups": (C.c_int, [C.POINTER(LinkagePair), C.c_int64, C.c_int32, C.c_int32, _P]),
    "ms_control_capture": (C.c_int, [_P]),
    "ms_control_call": (C.c_int, [_P, C.POINTER(Gene), C.c_int32, C.c_char_p, C.POINTER(CallParams), C.POINTER(Variant), C.c_int64,
                                  C.POINTER(ControlVariant), C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def load():
    """Load the shared library, raising (never falling back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m minorseq_b200.build` "
            "(minorseq_b200 has no CPU fallback)")
    lib = C.CDLL(os.environ.get("MS_LIB_PATH", LIB_PATH))   # the override is for A/B builds of the same ABI (tools/)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class MsError(RuntimeError):
    pass


def check(rc, handle=None):
    if rc != MS_OK:
        msg = load().ms_last_error(handle)
        raise MsError(f"minorseq_b200 error {rc}: {msg.decode() if msg else ''}")
