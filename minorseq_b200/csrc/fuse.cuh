// fuse.cuh -- K4's insertion tally, shared by ms_fuse (fuse.cu) and the per-group consensus (group.cu).
//
// An insertion event is keyed by an int32 "column" and its string.  ms_fuse keys by the reference column; the
// per-group consensus keys by g * L + column, so that the flattened group count tensor [g][L][8] is the `colcnt` the
// evaluation reads, and each group's insertions are tallied and judged against that group's own column votes.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace ms {

struct InsCand { int32_t col, len; long long rep; uint32_t cnt, pad; };

// (column, string) -> count and lowest event index, in an open-addressing table of mask + 1 slots
__global__ void ins_tally_kernel(const int32_t* __restrict__ col, const long long* __restrict__ off,
                                 const int32_t* __restrict__ len, int64_t nins, const char* __restrict__ pool,
                                 unsigned long long* tab_key, uint32_t* tab_cnt, long long* tab_rep, int64_t mask);
// table slots whose string is in frame (length a multiple of 3) and seen in more than frac * votes reads of its column
__global__ void ins_eval_kernel(const uint32_t* __restrict__ tab_cnt, const long long* __restrict__ tab_rep, int64_t tab_size,
                                const int32_t* __restrict__ col, const int32_t* __restrict__ len,
                                const uint32_t* __restrict__ colcnt, int32_t L, double frac,
                                InsCand* __restrict__ out, unsigned long long* nout, int64_t cap);

}  // namespace ms
