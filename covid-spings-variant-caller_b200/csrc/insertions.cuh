// Insertion counts for the consensus genome (include/lvc.h, lvc_enable_insertions / lvc_insertion_calls).
//
// Counting rule: a read that the deposit walks (read_passes_filter, at least one reference-consuming op, inside [0, G))
// counts each I op whose predecessor -- ignoring P ops and ops of length 0 -- is a match op (M, =, X) and whose anchor,
// the last base of that match op at reference position p, has quality >= min_bq.  Key: (p, len, seq) when
// len <= 32 and every inserted base is A/C/G/T with quality >= min_bq (seq = 2-bit codes, base k in bits 2k), else
// the unresolved key (p, 0, 0).  Base codes never need to represent a base below the threshold, so every batch form
// counts the same keys.
//
// The table is open addressing in HBM: 16-byte key slots claimed with one 128-bit atomicCAS, a parallel u32 count array
// incremented with atomicAdd.  The key set and the counts do not depend on the order in which reads arrive, only the slot
// a key lands in does.  A key is dropped (counted in `dropped`) only when every slot holds another key.
#pragma once
#include "lvc_common.cuh"
#include "consensus.cuh"

namespace lvc {

constexpr int kInsThreads = 256;            // k_count_insertions: one thread per read
constexpr int kInsScanThreads = 256;        // passes over the table slots
constexpr uint32_t kInsMaxLen = 32;         // longest insertion whose bases are kept (2 bits each in a 64-bit word)

struct InsTable {
    ulonglong2* keys;       // [mask + 1]; x = p << 32 | len << 1 | 1 (0: empty slot), y = seq
    uint32_t* counts;       // [mask + 1]
    uint32_t* dropped;      // [1]
    uint32_t mask;          // slots - 1 (a power of two minus one)
};

// one entry of lvc_copy_insertions / lvc_insertion_calls (mirrors lvc_insertion in include/lvc.h)
struct InsEntry {
    int32_t pos;
    uint32_t len;
    uint64_t seq;
    uint32_t count;
    uint32_t depth;
};

__device__ __forceinline__ uint64_t ins_mix(uint64_t x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdull;
    x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull;
    return x ^ (x >> 33);
}

__device__ __forceinline__ ulonglong2 ins_load_slot(const ulonglong2* s) {
    ulonglong2 v;
    asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(v.x), "=l"(v.y) : "l"(s) : "memory");
    return v;
}

// count one key; linear probing over at most every slot
__device__ __forceinline__ void ins_add(const InsTable& t, uint64_t k0, uint64_t k1) {
    uint32_t s = (uint32_t)ins_mix(k0 ^ ins_mix(k1 + 0x9E3779B97F4A7C15ull)) & t.mask;
    for (uint32_t probe = 0; probe <= t.mask; ++probe, s = (s + 1u) & t.mask) {
        ulonglong2 cur = ins_load_slot(t.keys + s);
        // a slot goes from empty to its key once.  The two words of a relaxed 16-byte load are each atomic, but not
        // together: x == 0, or the own x with y == 0, may be a torn read of a slot being claimed -- the CAS tells.
        if (cur.x == 0 || (cur.x == k0 && cur.y == 0)) {
            cur = atomicCAS(t.keys + s, make_ulonglong2(0ull, 0ull), make_ulonglong2(k0, k1));
            if (cur.x == 0) { atomicAdd(t.counts + s, 1u); return; }     // claimed
        }
        if (cur.x == k0 && cur.y == k1) { atomicAdd(t.counts + s, 1u); return; }
    }
    atomicAdd(t.dropped, 1u);
}

struct InsCountParams {
    int64_t G;
    int min_bq, min_mq;
};

// One thread per read.  Dead reads leave after their `keep` byte; reads without an I op read only their headers and
// CIGAR; only the anchors and inserted bases of counted insertions are read from the payload.
__global__ void __launch_bounds__(kInsThreads) k_count_insertions(const __grid_constant__ BatchView b,
                                                                  const __grid_constant__ InsTable t,
                                                                  const __grid_constant__ InsCountParams cp, uint32_t n) {
    const uint32_t i = blockIdx.x * kInsThreads + threadIdx.x;
    if (i < n) {
        const uint32_t keep = b.keep[i];
        if ((keep & 1u) && read_passes_filter(b.flag[i], b.mapq[i], keep, cp.min_mq)) {
            const uint32_t c0 = b.cigar_off[i], c1 = b.cigar_off[i + 1];
            int64_t rlen = 0;
            bool any_ins = false;
            for (uint32_t k = c0; k < c1; ++k) {
                const uint32_t c = b.cigar[k], op = c & 15u, len = c >> 4;
                if (op_consumes_ref(op)) rlen += len;
                any_ins |= op == 1u && len != 0u;
            }
            const int64_t pos = b.pos[i];
            // the deposit's conditions: no reference-consuming op, or outside [0, G) (LVC_ERANGE), deposits nothing
            if (any_ins && rlen != 0 && pos >= 0 && pos + rlen <= cp.G) {
                const uint64_t qb = b.seq_off[i];
                int64_t r = pos;
                uint32_t qi = 0, prev = 15u;                    // 15: no op yet
                for (uint32_t k = c0; k < c1; ++k) {
                    const uint32_t c = b.cigar[k], op = c & 15u, len = c >> 4;
                    if (len == 0u || op == 6u) continue;        // P and empty ops are transparent
                    if (op == 1u && op_is_match(prev) && (int)batch_qual(b, qb + qi - 1) >= cp.min_bq) {
                        bool resolved = len <= kInsMaxLen;
                        uint64_t seq = 0;
                        for (uint32_t j = 0; j < len && resolved; ++j) {
                            const uint32_t nib = batch_nibble(b, qb + qi + j);
                            resolved = (int)batch_qual(b, qb + qi + j) >= cp.min_bq && __popc(nib) == 1;
                            seq |= (uint64_t)(__ffs(nib) - 1) << (2 * j);     // A, C, G, T = 1, 2, 4, 8 -> 0..3
                        }
                        const uint64_t k0 = ((uint64_t)(r - 1) << 32) | (resolved ? (uint64_t)len << 1 : 0ull) | 1ull;
                        ins_add(t, k0, resolved ? seq : 0ull);
                    }
                    if (op_consumes_ref(op)) r += len;
                    if (op_consumes_query(op)) qi += len;
                    prev = op;
                }
            }
        }
    }
    // launched with programmatic serialization behind the deposit: the next kernel of the stream may only be released
    // once the deposit has completed, so nothing of this grid exits before it
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

__device__ __forceinline__ int32_t ins_pos(uint64_t k0) { return (int32_t)(k0 >> 32); }
__device__ __forceinline__ uint32_t ins_len(uint64_t k0) { return (uint32_t)(k0 >> 1) & 63u; }

// every occupied slot -> out[atomicAdd(n_out)] (at most cap entries written)
__global__ void __launch_bounds__(kInsScanThreads) k_insertion_list(const __grid_constant__ InsTable t, InsEntry* __restrict__ out,
                                                                   uint32_t cap, uint32_t* __restrict__ n_out) {
    const uint32_t s = blockIdx.x * kInsScanThreads + threadIdx.x;
    if (s > t.mask) return;
    const ulonglong2 k = t.keys[s];
    if (k.x == 0) return;
    const uint32_t j = atomicAdd(n_out, 1u);
    if (j < cap) out[j] = InsEntry{ins_pos(k.x), ins_len(k.x), k.y, t.counts[s], 0u};
}

// per anchor p in [p0, p1) (index p - p0): total[] = every count, unres[] = unresolved counts, best[] = the largest
// resolved count
__global__ void __launch_bounds__(kInsScanThreads) k_insertion_tally(const __grid_constant__ InsTable t, int64_t p0, int64_t p1,
                                                                    uint32_t* __restrict__ total, uint32_t* __restrict__ unres,
                                                                    uint32_t* __restrict__ best) {
    const uint32_t s = blockIdx.x * kInsScanThreads + threadIdx.x;
    if (s > t.mask) return;
    const ulonglong2 k = t.keys[s];
    const int64_t p = ins_pos(k.x);
    if (k.x == 0 || p < p0 || p >= p1) return;
    const uint32_t c = t.counts[s];
    atomicAdd(total + (p - p0), c);
    if (ins_len(k.x) == 0u) atomicAdd(unres + (p - p0), c);
    else atomicMax(best + (p - p0), c);
}

// n_best[] = the number of resolved keys whose count is best[]
__global__ void __launch_bounds__(kInsScanThreads) k_insertion_ties(const __grid_constant__ InsTable t, int64_t p0, int64_t p1,
                                                                   const uint32_t* __restrict__ best, uint32_t* __restrict__ n_best) {
    const uint32_t s = blockIdx.x * kInsScanThreads + threadIdx.x;
    if (s > t.mask) return;
    const ulonglong2 k = t.keys[s];
    const int64_t p = ins_pos(k.x);
    if (k.x == 0 || ins_len(k.x) == 0u || p < p0 || p >= p1) return;
    if (t.counts[s] == best[p - p0]) atomicAdd(n_best + (p - p0), 1u);
}

struct InsCallParams {
    int64_t p0, p1;
    uint64_t min_depth;
    double threshold;
    int grp_begin[5];          // the consensus pass's ordered plane list (ConsParams::grp_begin)
};

// The call rule: the unique best resolved key s at p is emitted, with depth d, iff the consensus letter of p is neither
// 'N' nor '-', count(s) > d - total (the reads without an insertion), count(s) > unresolved, and count(s) / d >= threshold.
__global__ void __launch_bounds__(kInsScanThreads) k_insertion_call(const __grid_constant__ InsTable t,
                                                                   const __grid_constant__ InsCallParams ip,
                                                                   const uint32_t* const* __restrict__ plane_ptrs,
                                                                   const uint32_t* __restrict__ dels,
                                                                   const uint32_t* __restrict__ total,
                                                                   const uint32_t* __restrict__ unres,
                                                                   const uint32_t* __restrict__ best,
                                                                   const uint32_t* __restrict__ n_best,
                                                                   InsEntry* __restrict__ out, uint32_t* __restrict__ n_out) {
    const uint32_t s = blockIdx.x * kInsScanThreads + threadIdx.x;
    if (s > t.mask) return;
    const ulonglong2 k = t.keys[s];
    const int64_t p = ins_pos(k.x);
    if (k.x == 0 || ins_len(k.x) == 0u || p < ip.p0 || p >= ip.p1) return;
    const int64_t x = p - ip.p0;
    const uint32_t c = t.counts[s];
    if (c != best[x] || n_best[x] != 1u || c <= unres[x]) return;
    // the position's counts as the consensus pass sums them
    uint64_t m[5] = {0, 0, 0, 0, __ldcg(dels + p)};
    uint64_t other = 0;
    for (int j = 0; j < ip.grp_begin[1]; ++j) {
        const uint4 v = __ldcg(reinterpret_cast<const uint4*>(plane_ptrs[j]) + p);
        m[0] += v.x; m[1] += v.y; m[2] += v.z; m[3] += v.w;
    }
    for (int j = ip.grp_begin[1]; j < ip.grp_begin[4]; ++j) {
        const uint4 v = __ldcg(reinterpret_cast<const uint4*>(plane_ptrs[j]) + p);
        other += (uint64_t)v.x + v.y + v.z + v.w;
    }
    const uint64_t d = m[0] + m[1] + m[2] + m[3] + m[4] + other;
    if (d == 0 || d < ip.min_depth) return;                                     // 'N'
    uint32_t mask = 0;
    const uint8_t letter = consensus_letter(m, d, ip.threshold, &mask);
    if (letter == 'N' || letter == '-') return;
    if ((uint64_t)c + total[x] <= d) return;                                    // count > d - total
    if (!((double)c / (double)d >= ip.threshold)) return;
    const uint32_t j = atomicAdd(n_out, 1u);
    out[j] = InsEntry{(int32_t)p, ins_len(k.x), k.y, c, (uint32_t)d};
}

}  // namespace lvc
