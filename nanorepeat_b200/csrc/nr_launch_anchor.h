// nr_launch_anchor.h -- Step 1's anchor kernel (nr_launch_anchor.cu) as the host side (nr_anchor.cu) sees it.  A header
// of its own: the other kernel families' translation units stay byte for byte what they were (their code placement,
// and with it their speed, follows the exact text they are compiled from, DESIGN.md section 9).
#pragma once
#include "nr_launch.h"

namespace nr {
namespace pr {
// one read strand (template) against its region's two anchors (queries, one per half)
struct AnchorPair {
    uint32_t t_word; int32_t t_len;
    uint32_t qa_word; int32_t q_a;     // left anchor: high half
    uint32_t qb_word; int32_t q_b;     // right anchor: low half (0: none)
    int32_t R, S;                      // rows per lane (a paired stripe height), stripes: 32 * R * S >= max(q_a, q_b)
    int32_t out;                       // keys[out] = (left key, right key)
    int32_t pad[3];
};
}  // namespace pr
}  // namespace nr

namespace nrl {
size_t anchor_smem_bytes();
cudaError_t launch_anchor_pairs(int blocks, cudaStream_t st, const nr::pr::AnchorPair* pairs, int n_pairs, const uint32_t* pool,
                                ulonglong2* scratch, size_t bnd_stride, int* counter, uint2* keys);
}  // namespace nrl
