// link_table.cuh -- the 2x2 table of a key pair from the stacked Gram matrix [B | M]^T [B | M] (linkage.cu, rare.cu).
#pragma once
#include <stdint.h>

namespace ms {

struct LinkTable { uint32_t a, b, c, n; };

// the 2x2 table of pair (v, w) from the stacked Gram matrix (dim x dim, half = dim / 2)
__device__ __forceinline__ LinkTable link_table(const int32_t* __restrict__ G, int32_t dim, int32_t v, int32_t w) {
    const int32_t half = dim >> 1;
    LinkTable t;
    t.a = static_cast<uint32_t>(G[static_cast<size_t>(v) * dim + w]);
    t.n = static_cast<uint32_t>(G[static_cast<size_t>(half + v) * dim + half + w]);
    t.b = static_cast<uint32_t>(G[static_cast<size_t>(v) * dim + half + w]) - t.a;     // B_v . M_w - a
    t.c = static_cast<uint32_t>(G[static_cast<size_t>(w) * dim + half + v]) - t.a;     // M_v . B_w - a
    return t;
}

}  // namespace ms
