// Consensus letter and coverage statistics per position, read straight from the persistent count tables.
//
// The rule (include/lvc.h, lvc_consensus): per position the A/C/G/T counts of the group-0 planes, the other nibble codes
// of groups 1..3 (nO) and the deletion entries give the depth d.  Below min_depth (or d == 0) the letter is 'N'.  Otherwise
// the members A, C, G, T, deletion with a non-zero count are taken in descending count order (ties by that rank order)
// until the taken share cum / d reaches the threshold; a deletion on top gives '-', else the IUPAC code of the taken
// bases, which is the BAM nibble alphabet indexed by their A=1 C=2 G=4 T=8 mask.  Insertions are not in the tables.
//
// Everything is a function of the integer tables alone (no first-seen ordinals), so the result is the same whatever
// deposit kernel, batch form, checkpoint or reduction produced them.
#pragma once
#include "lvc_common.cuh"

namespace lvc {

constexpr int kConsThreads = 128;           // one thread per position, a warp covers 32 consecutive positions
constexpr int kConsBatch = 8;               // plane rows requested together (ONT tables have ~61 planes)
constexpr int kConsMaxThr = 8;

// device counters, in the order of lvc_consensus_stats
enum { CS_POSITIONS = 0, CS_DEPTH_SUM, CS_DEPTH_MAX, CS_LOW_DEPTH, CS_N, CS_DELETED, CS_AMBIGUOUS, CS_MISMATCH, CS_GE,
       CS_WORDS = CS_GE + kConsMaxThr };

struct ConsParams {
    int64_t p0, p1;            // positions [p0, p1)
    uint64_t min_depth;
    double threshold;
    int grp_begin[5];          // planes of group g are [grp_begin[g], grp_begin[g+1]) in the ordered pointer list
    int n_thr;
    uint32_t thr[kConsMaxThr];
};

__device__ __forceinline__ uint64_t warp_sum_u64(uint64_t v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, d);
    return v;
}
__device__ __forceinline__ uint64_t warp_max_u64(uint64_t v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) { const uint64_t o = __shfl_xor_sync(0xFFFFFFFFu, v, d); v = o > v ? o : v; }
    return v;
}

// the letter of one position from its five member counts (A, C, G, T, deletion), the depth d > 0 and the threshold;
// *mask_out = the taken A/C/G/T mask (0 for 'N' by the threshold and for '-')
__device__ __forceinline__ uint8_t consensus_letter(const uint64_t (&n)[5], uint64_t d, double t, uint32_t* mask_out) {
    // rank of member i in the descending order: members with a larger count, or an equal count and a lower rank, go first
    uint64_t before[5];
    int top = 0;
    uint64_t members = 0;
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        uint64_t s = 0;
        int pos = 0;
#pragma unroll
        for (int j = 0; j < 5; ++j) {
            const bool ahead = n[j] > n[i] || (n[j] == n[i] && j < i);
            s += ahead ? n[j] : 0ull;
            pos += ahead ? 1 : 0;
        }
        before[i] = s;
        if (pos == 0) top = i;
        members += n[i];
    }
    const double dd = (double)d;
    // no member, or the members together stay below the threshold (the rest of the depth is in other codes): 'N'
    if (members == 0 || !((double)members / dd >= t)) { *mask_out = 0; return 'N'; }
    if (top == 4) { *mask_out = 0; return '-'; }
    // member i is taken iff it has a count and is on top, or the members ahead of it have not reached the threshold
    uint32_t mask = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if (n[i] > 0 && (i == top || (double)before[i] / dd < t)) mask |= 1u << i;
    *mask_out = mask;
    return (uint8_t)"=ACMGRSVTWYHKDBN"[mask];
}

__global__ void __launch_bounds__(kConsThreads) k_consensus(const __grid_constant__ ConsParams cp,
                                                            const uint32_t* const* __restrict__ plane_ptrs,
                                                            const uint32_t* __restrict__ dels,
                                                            const uint8_t* __restrict__ ref,
                                                            uint8_t* __restrict__ seq_out,
                                                            unsigned long long* __restrict__ stats) {
    __shared__ const uint32_t* s_planes[kMaxKeys];
    __shared__ unsigned long long s_stats[CS_WORDS];
    const int tid = threadIdx.x;
    const int n_planes = cp.grp_begin[4];
    for (int k = tid; k < n_planes; k += kConsThreads) s_planes[k] = plane_ptrs[k];
    if (tid < CS_WORDS) s_stats[tid] = 0ull;
    __syncthreads();

    const int g0_end = cp.grp_begin[1];
    uint64_t depth_sum = 0, depth_max = 0;
    uint32_t c_pos = 0, c_low = 0, c_n = 0, c_del = 0, c_amb = 0, c_mis = 0;
    uint32_t c_ge[kConsMaxThr];
#pragma unroll
    for (int i = 0; i < kConsMaxThr; ++i) c_ge[i] = 0;

    const int64_t stride = (int64_t)gridDim.x * kConsThreads;
    for (int64_t base = cp.p0 + (int64_t)blockIdx.x * kConsThreads; base < cp.p1; base += stride) {
        const int64_t p = base + tid;
        const bool live = p < cp.p1;
        const int64_t pc = live ? p : cp.p1 - 1;            // the tail lanes read a valid row and contribute nothing
        const uint32_t nd32 = __ldcg(dels + pc);
        const uint8_t rb = ref[pc];
        uint64_t n[5] = {0, 0, 0, 0, 0};
        uint64_t n_other = 0;
        // group 0: one 16-byte row per plane, kConsBatch rows in flight
        for (int k0 = 0; k0 < g0_end; k0 += kConsBatch) {
            uint4 r[kConsBatch];
#pragma unroll
            for (int j = 0; j < kConsBatch; ++j)
                r[j] = k0 + j < g0_end ? __ldcg(reinterpret_cast<const uint4*>(s_planes[k0 + j]) + pc) : make_uint4(0, 0, 0, 0);
#pragma unroll
            for (int j = 0; j < kConsBatch; ++j) { n[0] += r[j].x; n[1] += r[j].y; n[2] += r[j].z; n[3] += r[j].w; }
        }
        // groups 1..3: every slot counts towards the depth only
        for (int k0 = g0_end; k0 < n_planes; k0 += kConsBatch) {
            uint4 r[kConsBatch];
#pragma unroll
            for (int j = 0; j < kConsBatch; ++j)
                r[j] = k0 + j < n_planes ? __ldcg(reinterpret_cast<const uint4*>(s_planes[k0 + j]) + pc) : make_uint4(0, 0, 0, 0);
#pragma unroll
            for (int j = 0; j < kConsBatch; ++j) n_other += (uint64_t)r[j].x + r[j].y + r[j].z + r[j].w;
        }
        n[4] = nd32;
        const uint64_t d = n[0] + n[1] + n[2] + n[3] + n[4] + n_other;
        const bool low = d < cp.min_depth;
        uint8_t letter = 'N';
        uint32_t mask = 0;
        if (d != 0 && !low) letter = consensus_letter(n, d, cp.threshold, &mask);
        if (live) seq_out[p - cp.p0] = letter;

        const uint32_t bits = __popc(mask);
        const uint8_t ru = (rb >= 'a' && rb <= 'z') ? (uint8_t)(rb - 32) : rb;
        const bool ref_acgt = ru == 'A' || ru == 'C' || ru == 'G' || ru == 'T';
        c_pos += __popc(__ballot_sync(0xFFFFFFFFu, live));
        c_low += __popc(__ballot_sync(0xFFFFFFFFu, live && low));
        c_n += __popc(__ballot_sync(0xFFFFFFFFu, live && letter == 'N'));
        c_del += __popc(__ballot_sync(0xFFFFFFFFu, live && letter == '-'));
        c_amb += __popc(__ballot_sync(0xFFFFFFFFu, live && (bits == 2 || bits == 3)));
        c_mis += __popc(__ballot_sync(0xFFFFFFFFu, live && bits == 1 && ref_acgt && letter != ru));
#pragma unroll
        for (int i = 0; i < kConsMaxThr; ++i)                // unrolled: the counters stay in registers
            if (i < cp.n_thr) c_ge[i] += __popc(__ballot_sync(0xFFFFFFFFu, live && d >= cp.thr[i]));
        const uint64_t dl = live ? d : 0ull;
        depth_sum += dl;
        depth_max = dl > depth_max ? dl : depth_max;
    }
    // the ballot counts are already per warp; sums and maxima of the depth are reduced over the warp here
    depth_sum = warp_sum_u64(depth_sum);
    depth_max = warp_max_u64(depth_max);
    if ((tid & 31) == 0) {
        atomicAdd(&s_stats[CS_POSITIONS], (unsigned long long)c_pos);
        atomicAdd(&s_stats[CS_DEPTH_SUM], (unsigned long long)depth_sum);
        atomicMax(&s_stats[CS_DEPTH_MAX], (unsigned long long)depth_max);
        atomicAdd(&s_stats[CS_LOW_DEPTH], (unsigned long long)c_low);
        atomicAdd(&s_stats[CS_N], (unsigned long long)c_n);
        atomicAdd(&s_stats[CS_DELETED], (unsigned long long)c_del);
        atomicAdd(&s_stats[CS_AMBIGUOUS], (unsigned long long)c_amb);
        atomicAdd(&s_stats[CS_MISMATCH], (unsigned long long)c_mis);
#pragma unroll
        for (int i = 0; i < kConsMaxThr; ++i)
            if (i < cp.n_thr) atomicAdd(&s_stats[CS_GE + i], (unsigned long long)c_ge[i]);
    }
    __syncthreads();
    if (tid < CS_GE + cp.n_thr) {
        if (tid == CS_DEPTH_MAX) atomicMax(&stats[tid], s_stats[tid]);
        else atomicAdd(&stats[tid], s_stats[tid]);
    }
}

}  // namespace lvc
