"""minorseq_b200 -- B200-native juliet/fuse hot path (pileup, codon test, phasing, consensus).

The compute path is libminorseq_b200.so (hand-written CUDA for sm_100a behind the C ABI in
include/minorseq_b200.h).  There is no CPU fallback.
"""
from . import _lib  # noqa: F401
from .api import (CODONS, Aligner, Fuse, Handle, Juliet, decode_events, device_rows, encode_rows, encode_states, host_rows, synth_device,  # noqa: F401
                  translate)
from .synth import (SynthConfig, make_tables, pack_states, start_mask_words, synth_states, tile_rows, unpack_states,  # noqa: F401
                    untile_rows)

__version__ = "0.1.0"
