// Strand counts for strand-bias statistics (include/lvc.h, lvc_enable_strand_counts / lvc_strand_counts).
//
// Rule: a read that the deposit walks (read_passes_filter, at least one reference-consuming op, inside [0, G)) and whose
// flag has 0x10 (reverse strand) adds 1, for every pileup entry at p that the deposit adds to totalDepth, to
//   rev[gs][p]    for a base with BAM nibble n, gs = nibble_gs(n) (the plane group << 2 | slot), quality >= min_bq;
//   rev[16][p]    for a deletion / ref-skip entry whose deciding quality -- the query base at the start of the op, 0 past
//                 the end of the read, the quality htslib's resolve_cigar2 assigns -- is >= min_bq.
// The forward counts are the plane sums minus rev (and dels minus rev[16]): both come from the same pushes.  Only bases at
// or above the threshold are ever read, so every batch form counts the same values.
//
// Kernel: one CTA per chunk of kStrandReads consecutive reads.  Forward and dead reads leave after their flag and keep
// bytes; each warp takes reverse reads in turn.  A read's CIGAR is taken 32 ops at a time (one op per lane, scanned across
// the warp), and its counted entries -- the bases of its match ops and the columns of its passing deletions -- are
// flattened, so the lanes stride over them whatever the op lengths are (coalesced payload loads, every lane busy on ONT
// reads of short ops).  A/C/G/T and deletion entries whose column lies in the tile [base, base + kStrandTile), base the
// lowest start of the chunk's reverse reads, go to a shared count tile; the flush adds each non-zero cell to the table with
// one global atomic.  Other nibble codes and columns past the tile go to global atomics directly.
#pragma once
#include "lvc_common.cuh"

namespace lvc {

constexpr int kStrandThreads = 256;          // k_count_strands: 8 warps
constexpr uint32_t kStrandReads = 256;       // reads per CTA (one header load per thread)
constexpr uint32_t kStrandTile = 1024;       // tile columns: rows A, C, G, T and deletions, 20 KB
constexpr uint32_t kStrandRows = 17;         // table rows: the 16 slots (gs), then deletions
constexpr int kStrandQueryThreads = 256;     // k_strand_query: one thread per query

struct StrandCountParams {
    int64_t G;
    int min_bq, min_mq;
};

// one counted entry of a reverse read at column col: row 0..15 (gs) or 16 (deletion)
__device__ __forceinline__ void strand_add(uint32_t* tile, uint32_t* rev, int64_t G, int64_t base, int64_t col, uint32_t row) {
    const uint64_t t = (uint64_t)(col - base);
    const uint32_t trow = row < 4u ? row : row == 16u ? 4u : 5u;          // tile rows: A, C, G, T, deletion
    if (trow < 5u && t < kStrandTile) atomicAdd(tile + trow * kStrandTile + (uint32_t)t, 1u);
    else atomicAdd(rev + (int64_t)row * G + col, 1u);
}

__global__ void __launch_bounds__(kStrandThreads) k_count_strands(const __grid_constant__ BatchView b, uint32_t* __restrict__ rev,
                                                                  const __grid_constant__ StrandCountParams cp, uint32_t n) {
    __shared__ uint32_t tile[5 * kStrandTile];
    __shared__ uint32_t list[kStrandReads];
    __shared__ uint32_t n_list;
    __shared__ int64_t base;
    __shared__ int64_t top;                      // one past the last tile column a read of this chunk reaches
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint32_t i0 = blockIdx.x * kStrandReads;
    if (tid == 0) { n_list = 0; base = INT64_MAX; top = 0; }
    __syncthreads();
    if (tid < kStrandReads && i0 + tid < n) {
        const uint32_t i = i0 + tid;
        const uint32_t keep = b.keep[i];
        if (keep & 1u) {
            const uint32_t flag = b.flag[i];
            if ((flag & 0x10u) && read_passes_filter(flag, b.mapq[i], keep, cp.min_mq)) {
                list[atomicAdd(&n_list, 1u)] = i;
                atomicMin((unsigned long long*)&base, (unsigned long long)(int64_t)b.pos[i]);   // the deposit skips pos < 0
            }
        }
    }
    __syncthreads();
    const uint32_t nl = n_list;
    if (nl != 0) {
        for (uint32_t k = tid; k < 5 * kStrandTile; k += kStrandThreads) tile[k] = 0;
        __syncthreads();
        const int64_t tb = base;
        for (uint32_t e = warp; e < nl; e += kStrandThreads / 32) {
            const uint32_t i = list[e];
            const uint32_t c0 = b.cigar_off[i], c1 = b.cigar_off[i + 1];
            const int64_t pos = b.pos[i];
            // reference length and l_qseq
            uint32_t rlen = 0, lq = 0;
            for (uint32_t k = c0 + lane; k < c1; k += 32) {
                const uint32_t c = b.cigar[k], op = c & 15u, len = c >> 4;
                if (op_consumes_ref(op)) rlen += len;
                if (op_consumes_query(op)) lq += len;
            }
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) {
                rlen += __shfl_xor_sync(0xFFFFFFFFu, rlen, d);
                lq += __shfl_xor_sync(0xFFFFFFFFu, lq, d);
            }
            // the deposit's conditions: no reference-consuming op, or outside [0, G) (LVC_ERANGE), deposits nothing
            if (rlen == 0 || pos < 0 || pos + (int64_t)rlen > cp.G) continue;
            if (lane == 0) atomicMax((unsigned long long*)&top, (unsigned long long)(pos + rlen));
            const uint64_t qb = b.seq_off[i];
            int64_t r = pos;                     // reference column and query index at the start of the op group
            uint32_t qi = 0;
            for (uint32_t g0 = c0; g0 < c1; g0 += 32) {
                const uint32_t c = g0 + lane < c1 ? b.cigar[g0 + lane] : 0u;      // padding: a match of length 0
                const uint32_t op = c & 15u, len = c >> 4;
                const uint32_t rl = op_consumes_ref(op) ? len : 0u, ql = op_consumes_query(op) ? len : 0u;
                uint32_t r_in = rl, q_in = ql;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const uint32_t ur = __shfl_up_sync(0xFFFFFFFFu, r_in, d), uq = __shfl_up_sync(0xFFFFFFFFu, q_in, d);
                    if ((int)lane >= d) { r_in += ur; q_in += uq; }
                }
                const uint32_t r_op = r_in - rl, q_op = q_in - ql;                // offsets of this op inside the group
                // entries of this op: every base of a match op (tested below), every column of a passing deletion
                uint32_t ne = 0;
                if (op_is_match(op)) ne = len;
                else if (op == 2u || op == 3u) {
                    const uint32_t qx = qi + q_op;
                    ne = (int)(qx < lq ? batch_qual(b, qb + qx) : 0u) >= cp.min_bq ? len : 0u;
                }
                uint32_t e_in = ne;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const uint32_t u = __shfl_up_sync(0xFFFFFFFFu, e_in, d);
                    if ((int)lane >= d) e_in += u;
                }
                const uint32_t total = __shfl_sync(0xFFFFFFFFu, e_in, 31);
                for (uint32_t j0 = 0; j0 < total; j0 += 32) {
                    const uint32_t j = j0 + lane;
                    // the op holding entry j: the first lane whose inclusive entry sum exceeds j
                    uint32_t k = 0;
#pragma unroll
                    for (uint32_t s = 16; s > 0; s >>= 1) {
                        const uint32_t v = __shfl_sync(0xFFFFFFFFu, e_in, k + s - 1u);
                        if (v <= j) k += s;
                    }
                    const uint32_t k_op = __shfl_sync(0xFFFFFFFFu, op, k);
                    const uint32_t k_r = __shfl_sync(0xFFFFFFFFu, r_op, k);
                    const uint32_t k_q = __shfl_sync(0xFFFFFFFFu, q_op, k);
                    const uint32_t k_e = __shfl_sync(0xFFFFFFFFu, e_in - ne, k);
                    if (j >= total) continue;
                    const uint32_t off = j - k_e;
                    const int64_t col = r + k_r + off;
                    if (op_is_match(k_op)) {
                        const uint64_t x = qb + qi + k_q + off;
                        if ((int)batch_qual(b, x) >= cp.min_bq) strand_add(tile, rev, cp.G, tb, col, nibble_gs(batch_nibble(b, x)));
                    } else {
                        strand_add(tile, rev, cp.G, tb, col, 16u);
                    }
                }
                r += __shfl_sync(0xFFFFFFFFu, r_in, 31);
                qi += __shfl_sync(0xFFFFFFFFu, q_in, 31);
            }
        }
        __syncthreads();
        // flush: one global atomic per non-zero cell of the columns the chunk reached
        const uint32_t width = (uint32_t)min((int64_t)kStrandTile, top > tb ? top - tb : (int64_t)0);
        for (uint32_t row = 0; row < 5; ++row)
            for (uint32_t t = tid; t < width; t += kStrandThreads) {
                const uint32_t v = tile[row * kStrandTile + t];
                if (v) atomicAdd(rev + (int64_t)(row < 4u ? row : 16u) * cp.G + tb + t, v);
            }
    }
    // launched with programmatic serialization behind the deposit: the next kernel of the stream may only be released
    // once the deposit has completed, so nothing of this grid exits before it
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

// lvc_strand_counts: one thread per query (pos, row): the allele's count summed over its planes (rows 0..15: the planes of
// group row >> 2, slot row & 3; row 16: dels), and rev of the same cell.  `planes` are ordered by key, the planes of group
// g being [grp_begin[g], grp_begin[g + 1]).
struct StrandQueryParams {
    int64_t G;
    int grp_begin[5];
};

__global__ void __launch_bounds__(kStrandQueryThreads) k_strand_query(const __grid_constant__ StrandQueryParams qp,
                                                                      const uint32_t* const* __restrict__ planes,
                                                                      const uint32_t* __restrict__ dels,
                                                                      const uint32_t* __restrict__ rev,
                                                                      const int32_t* __restrict__ pos, const uint8_t* __restrict__ row,
                                                                      uint32_t* __restrict__ fwd_out, uint32_t* __restrict__ rev_out,
                                                                      uint32_t n) {
    const uint32_t k = blockIdx.x * kStrandQueryThreads + threadIdx.x;
    if (k >= n) return;
    const int64_t p = pos[k];
    const uint32_t w = row[k];
    uint32_t total = 0;
    if (w == 16u) total = dels[p];
    else
        for (int pl = qp.grp_begin[w >> 2]; pl < qp.grp_begin[(w >> 2) + 1]; ++pl) total += planes[pl][p * 4 + (w & 3u)];
    const uint32_t rv = rev[(int64_t)w * qp.G + p];
    fwd_out[k] = total - rv;
    rev_out[k] = rv;
}

}  // namespace lvc
