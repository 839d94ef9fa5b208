// Position-parallel fp64 genotype-likelihood kernel.
//
// Replaces prepare_variants (live_variant_caller.py:120-231) + utils.genotype_likelihood
// (utils.py:16-24) up to, but not including, the log10/round/format of the few emitted records
// (done on the host with the host libm, SURVEY A6).
//
// The reference multiplies per-read error probabilities sequentially in fp64 and lets the product
// underflow to exactly 0.0.  Here every product  prod_q e[q]^n[q]  is evaluated from the integer quality
// histogram in the log2 domain with double-double arithmetic:  S = sum_q n[q] * log2(e[q]),  the logarithms
// being double-double constants computed on the host in 80-bit arithmetic from the SAME e[q] / 1-e[q] doubles
// the reference uses (math.pow; never pow() on the device).  S carries ~100 bits, so 2^S is good to ~1e-15
// relative whatever the depth; it is split into an integer exponent and a fraction in [0,1), and the result
// is rounded to fp64 ONCE (ldexp): exactly 0.0 where the true product is below 2^-1075, a correctly rounded
// denormal inside the denormal band (where the reference itself is order dependent).  Three fused multiply-adds
// per (plane, allele, logarithm) on exactly summable pieces of the constants (Acc3 below): no data-dependent loop,
// no divergence, a third of the fp64 operations of a double-double update.
#pragma once
#include "lvc_common.cuh"

namespace lvc {

struct DD {            // value = h + l, |l| <= ulp(h)/2
    double h, l;
};

__device__ __forceinline__ DD dd_add(DD a, DD b) {
    const double t = a.h + b.h;
    const double bp = t - a.h;
    const double se = (a.h - (t - bp)) + (b.h - bp);
    const double lo = se + a.l + b.l;
    const double h = t + lo;
    return DD{h, lo - (h - t)};
}

__device__ __forceinline__ DD dd_sub(DD a, DD b) { return dd_add(a, DD{-b.h, -b.l}); }

__device__ __forceinline__ DD dd_shfl_xor(DD v, int lanemask) {
    return DD{__shfl_xor_sync(0xFFFFFFFFu, v.h, lanemask), __shfl_xor_sync(0xFFFFFFFFu, v.l, lanemask)};
}

// 2^(h + l) rounded once to fp64 (gradual underflow; 0.0 below the denormal range)
__device__ __forceinline__ double dd_exp2(DD s) {
    const double t = s.h + s.l;
    if (!(t > -1200.0)) return 0.0;
    const double i = floor(s.h);
    const double f = (s.h - i) + s.l;                      // in [0, 1] up to the low part
    return ldexp(exp2(f), (int)i);
}

struct GenoParams {
    int64_t G;
    int64_t p0, p1;          // positions [p0, p1) are genotyped (the whole contig by default)
    int64_t min_total_depth;
    int64_t min_allele_depth;
    double min_ratio;
    uint32_t flags;
    int n_planes;            // all planes, ordered by key (group 0 first)
    int grp_begin[5];        // planes of group g are [grp_begin[g], grp_begin[g+1])
    uint32_t cand_cap;
};

constexpr int kGenoThreads = 128;            // 32 positions x 4 allele slots
#ifndef LVC_GENO_BATCH
#define LVC_GENO_BATCH 8
#endif
constexpr int kGenoBatch = LVC_GENO_BATCH;                // plane counts requested together

// Exact accumulation without double-double arithmetic in the loop.  Each logarithm c is split ON THE HOST into
//   c = c1 + c2 + c3,   c1 a multiple of 2^-10 (|c1| < 2^8),  c2 a multiple of 2^-36 (|c2| <= 2^-11),  |c3| <= 2^-37,
// so for counts n the partial sums  sum n*c1  (multiples of 2^-10, < 2^43 for 2^35 deposited bases) and  sum n*c2
// (multiples of 2^-36, < 2^17 for 2^28 bases) are EXACT in fp64 with one FMA each, and  sum n*c3  is tiny (its
// rounding error is far below 2^-60).  Three FMAs per (plane, allele, logarithm) replace the 12-operation
// double-double update; the three sums are folded into one double-double after the loop.  ~95 bits survive, as
// before.  (A logarithm of 0 probability is stored as c1 = -1e290: the product vanishes, which is what it must do.)
struct Acc3 {
    double s1, s2, s3;
};
__device__ __forceinline__ void acc3_fma(Acc3& a, double n, double c1, double c2, double c3) {
    a.s1 = fma(n, c1, a.s1);
    a.s2 = fma(n, c2, a.s2);
    a.s3 = fma(n, c3, a.s3);
}
__device__ __forceinline__ DD acc3_fold(const Acc3& a) {
    const double t = a.s1 + a.s2;
    const double bp = t - a.s1;
    const double e = (a.s1 - (t - bp)) + (a.s2 - bp);          // exact error of s1 + s2
    const double lo = e + a.s3;
    const double h = t + lo;
    return DD{h, lo - (h - t)};
}

struct AlleleStat {
    Acc3 pe;     // log2 prod e
    Acc3 p1;     // log2 prod (1-e)
    double es;   // sum e
    uint32_t ad;
};

// per-plane constants, built on the host: log2(e) and log2(1-e) in three exact pieces each, and e itself
struct PlaneConst {
    double le1, le2, le3, lo1, lo2, lo3, e;
};

// One lane per (position, allele slot); the 4 slots of a position sit in 4 adjacent lanes and are combined with
// shuffles.  Alleles of the rare groups 1..3 are handled by the same lanes in turn.
template <int NG>      // NG = 1: only the A/C/G/T group has planes (the usual case), 4: all groups
__global__ void __launch_bounds__(kGenoThreads) k_genotype(GenoParams gp, const uint32_t* const* __restrict__ plane_ptrs,
                                                           const PlaneConst* __restrict__ pconst,
                                                           const uint32_t* __restrict__ dels,
                                                           const uint8_t* __restrict__ ref,
                                                           const uint32_t* const* __restrict__ first,
                                                           uint32_t* __restrict__ out_depth, uint32_t* __restrict__ out_ad,
                                                           double* __restrict__ out_lik, lvc_candidate* __restrict__ cand,
                                                           uint32_t* __restrict__ cand_count,
                                                           uint32_t* __restrict__ cand_count_next,
                                                           uint32_t* __restrict__ seen) {
    const int tid = threadIdx.x;
    // per-plane constants in shared memory: every lane of a warp reads the same entry
    extern __shared__ __align__(16) unsigned char geno_smem[];
    PlaneConst* s_pc = reinterpret_cast<PlaneConst*>(geno_smem);
    // the per-plane constants were uploaded by a copy that precedes the previous kernel of the stream (or this launch,
    // which a copy node serialises fully): they can be staged while that kernel drains
    {
        const double* src = reinterpret_cast<const double*>(pconst);
        double* dst = reinterpret_cast<double*>(geno_smem);
        const int nd = gp.n_planes * (int)(sizeof(PlaneConst) / sizeof(double));
        for (int k = tid; k < nd; k += kGenoThreads) dst[k] = src[k];
    }
    // everything below reads tables written by the deposit kernel launched before this one
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;");        // the next deposit kernel may start reading its batch
    if (blockIdx.x == 0 && tid == 0) *cand_count_next = 0;
    const int slot = tid & 3;
    // the first position of a block is a multiple of 8 (a warp writes one word of `seen`)
    const int64_t p = (gp.p0 & ~7ll) + (int64_t)blockIdx.x * (kGenoThreads / 4) + (tid / 4);
    const bool live = p >= gp.p0 && p < gp.p1;
    const int64_t pc = p < gp.p0 ? gp.p0 : (p < gp.p1 ? p : gp.p1 - 1);   // clamp: every lane takes part in the shuffles
    // requested now, used after the plane loop: deletion entries of the position and (for the hint) the first-seen cell
    const uint32_t dels_p = dels[pc];
    uint32_t first_p = kUnsetOrdinal;
    if (seen && first[0]) first_p = first[0][pc * 4 + slot];
    __syncthreads();

    AlleleStat st[NG];
#pragma unroll
    for (int g = 0; g < NG; ++g) { st[g].pe = Acc3{0.0, 0.0, 0.0}; st[g].p1 = Acc3{0.0, 0.0, 0.0}; st[g].es = 0.0; st[g].ad = 0; }
    DD pe_dd[NG], p1_dd[NG];

#pragma unroll
    for (int g = 0; g < NG; ++g) {
        // counts of up to kGenoBatch planes are requested together (one memory latency per batch, not per plane);
        // a count of 0 adds 0 to every sum, so nothing branches on the data
        for (int k0 = gp.grp_begin[g]; k0 < gp.grp_begin[g + 1]; k0 += kGenoBatch) {
            uint32_t cnt[kGenoBatch];
#pragma unroll
            for (int j = 0; j < kGenoBatch; ++j)
                cnt[j] = k0 + j < gp.grp_begin[g + 1] ? __ldcg(&plane_ptrs[k0 + j][pc * 4 + slot]) : 0u;
#pragma unroll
            for (int j = 0; j < kGenoBatch; ++j) {
                if (k0 + j < gp.grp_begin[g + 1]) {                       // uniform over the block
                    const PlaneConst& pcn = s_pc[k0 + j];
                    const double nd = (double)cnt[j];
                    st[g].ad += cnt[j];
                    st[g].es = fma(nd, pcn.e, st[g].es);
                    acc3_fma(st[g].pe, nd, pcn.le1, pcn.le2, pcn.le3);
                    acc3_fma(st[g].p1, nd, pcn.lo1, pcn.lo2, pcn.lo3);
                }
            }
        }
        pe_dd[g] = acc3_fold(st[g].pe);
        p1_dd[g] = acc3_fold(st[g].p1);
    }
    // ---- combine the (up to 16) alleles of the position: log2 of the product of e over ALL of them
    constexpr bool has_other = NG > 1;
    DD own = pe_dd[0];
    uint32_t own_ad = st[0].ad;
    if (has_other) {
#pragma unroll
        for (int g = 1; g < NG; ++g) { own = dd_add(own, pe_dd[g]); own_ad += st[g].ad; }
    }
    DD tot = dd_add(own, dd_shfl_xor(own, 1));
    tot = dd_add(tot, dd_shfl_xor(tot, 2));
    uint32_t dsum = own_ad + __shfl_xor_sync(0xFFFFFFFFu, own_ad, 1);
    dsum += __shfl_xor_sync(0xFFFFFFFFu, dsum, 2);
    const uint64_t depth = (uint64_t)dels_p + dsum;
    // L(a) = prod(1-e | a) * prod over b != a of prod(e | b)      (utils.py:16-24)
    double L[NG];
    double Ssum = 0.0;
#pragma unroll
    for (int g = 0; g < NG; ++g) {
        L[g] = 0.0;
        if ((g == 0 || has_other) && st[g].ad) {
            L[g] = dd_exp2(dd_add(p1_dd[g], dd_sub(tot, pe_dd[g])));
            Ssum += L[g];
        }
    }
    Ssum += __shfl_xor_sync(0xFFFFFFFFu, Ssum, 1);
    Ssum += __shfl_xor_sync(0xFFFFFFFFu, Ssum, 2);
    const double S = Ssum == 0.0 ? 1.0 : Ssum;                                   // live_variant_caller.py:146
    if (seen) {
        // hint for the deposit kernels (TableView::seen): which A/C/G/T alleles of these 8 positions have a first-seen
        // ordinal now -- no later batch can lower it.  Lane = position * 4 + slot is exactly the nibble layout.
        const bool has = live && first_p != kUnsetOrdinal;
        const uint32_t word = __ballot_sync(0xFFFFFFFFu, has);
        if ((tid & 31) == 0) seen[p >> 3] = word;
    }
    if (!live) return;
    const uint32_t depth32 = (uint32_t)(depth > 0xFFFFFFFFull ? 0xFFFFFFFFull : depth);
    if (slot == 0) out_depth[p] = depth32;
    out_ad[p * 4 + slot] = st[0].ad;
    out_lik[p * 4 + slot] = L[0];

    if ((int64_t)depth < gp.min_total_depth) return;                 // :131
    if (depth == 0) return;
    const uint8_t rb = ref[p];
    const bool all = gp.flags & 1u;
    const double ddepth = (double)depth;
#pragma unroll
    for (int g = 0; g < NG; ++g) {
        if (!((g == 0 || has_other) && st[g].ad)) continue;
        const uint32_t gs = (uint32_t)(g * 4 + slot);
        const uint32_t nib = gs_nibble(gs);
        const char letter = "=ACMGRSVTWYHKDBN"[nib];
        const bool ok = all || ((uint8_t)letter != rb && (int64_t)st[g].ad >= gp.min_allele_depth &&
                                ((double)st[g].ad / ddepth) >= gp.min_ratio);     // :151-155
        if (!ok) continue;
        const uint32_t idx = atomicAdd(cand_count, 1u);
        if (idx >= gp.cand_cap) continue;
        lvc_candidate c;
        c.pos = (int32_t)p; c.code = (uint8_t)nib; c.ref = rb; c.pad0 = 0;
        c.ad = st[g].ad; c.dp = depth32;
        const uint32_t* f = first[g];
        c.first = f ? f[p * 4 + slot] : kUnsetOrdinal;
        c.pad1 = 0; c.L = L[g]; c.S = S; c.esum = st[g].es;
        cand[idx] = c;
    }
}

}  // namespace lvc
