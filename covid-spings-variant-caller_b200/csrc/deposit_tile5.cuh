// Tiled deposit kernel, generation 5: bit-sliced counters, 32-column units, per-task flush.
//
// Front half as in deposit_tile4.cuh (chunk of 256 coordinate-sorted reads per CTA, classification into match runs,
// payload reduced to 4-bit one-hot KEYS while it is copied from global memory).  What changed is everything after the
// keys are staged (DESIGN.md section 3.1):
//   * unit   = 32 columns of one run per lane (4 key words from 5 aligned shared words), so the per-unit overhead
//              (run record, offsets, edge test) is paid once per 32 bases instead of once per 16;
//   * counts = BIT-SLICED.  A key word holds 8 columns x 4 one-hot allele bits = 32 one-bit counters; a lane adds
//              its units into three bit planes with a carry-save ripple (4 LOP3 per word, all four alleles at once,
//              no shifts, no per-allele masks; <= 7 units per lane per task);
//   * reduce = the 32 lanes of a warp hold 32 different runs of the same 32 columns.  Two exchange levels split the
//              four words over the lane groups (bit-sliced full adders), three more levels are an all-reduce inside
//              groups of 8 lanes on whole registers: after them lane L holds the task's A/C/G/T counts of column L
//              of the slab as 8 planes, turned into four byte fields with one multiply per plane;
//   * flush  = straight to the tables from the task (one RED per non-zero (column, allele) per task): no shared
//              count table, no zeroing, no shared atomics, and no barrier between the task loop and the flush -- a
//              warp that runs out of tasks is done with the column window.
// Launched with programmatic stream serialization: everything before `griddepcontrol.wait` only reads the batch.
#pragma once
#include "deposit_tile4.cuh"
#include "qcode.hpp"

namespace lvc {

#ifndef LVC5_CTAS_PER_SM
#define LVC5_CTAS_PER_SM 7
#endif
#ifndef LVC5_THREADS
#define LVC5_THREADS 192
#endif
// CTA = 192 threads = 192 reads: a chunk of 150 bp shotgun reads at 1,000x then spans 6 slabs of 32 columns whose
// candidate runs fit ONE task each (<= 224 runs): 6 tasks for 6 warps, one reduction per warp per chunk, where 256
// reads gave 12 tasks for 8 warps (two rounds, a quarter of the task phase idle)
constexpr int kT5Threads = LVC5_THREADS;
constexpr int kT5Warps = kT5Threads / 32;
constexpr int kT5Reads = kT5Threads;              // one read header per thread
static_assert(kT5Threads % 32 == 0 && kT5Threads <= 256, "read index in a chunk is stored in 8 bits");
constexpr uint32_t kT5WinStride = kT5Reads * 160u;                   // payload bytes per staged window
constexpr uint32_t kT5KeyCapBases = kT5WinStride + kMaxReadBytes;    // + one longest tileable read
constexpr int kTile5CtasPerSM = LVC5_CTAS_PER_SM;
// Where the kernel waits for the previous kernel of the stream (programmatic dependent launch):
//   0  before the byte extents (everything after the read-level filter follows the wait)
//   1  before the coverage atomics (extents, payload prefetch and classification precede it)
//   2  after the first window is staged: the coverage / deletion updates are parked in shared memory, so that headers,
//      classification AND the payload loads of a chunk overlap the tail of the previous kernel
// Measured (config 2 / config 5 step): 0: 75.0 / 539 us, 1: 74.1 / 538 us, 2: 77.9 / 582 us -- the parked update costs more
// than the overlap returns; 1 is the default.
#ifndef LVC5_WAIT
#define LVC5_WAIT 1
#endif
constexpr int kTask5Runs = 224;                  // runs per task: 7 units per lane, three bit planes hold <= 7

// Run table: per run only what the task table and the pass loop need -- the read's start column (s_rs), the packed
// (start column, key offset | length) record (s_pk) and (window << 8 | read index) (s_rix).  The cold-path deposit, the
// first-seen scan and multi-window chunks derive a run's column, length and payload offset from s_pk: inside one staged
// window a run's payload offset is w_rel + (s_pk.y & 0xFFFF).
struct Tile5Smem {
    static constexpr uint32_t key_off = 0;                                     // 4-bit keys, little-endian nibble order
    static constexpr uint32_t key_bytes = kSlack + kT5KeyCapBases / 2 + 32 + kSlack;
    static constexpr uint32_t rs_off = key_off + key_bytes;                    // i32 [kMaxRuns] start column of the run's read
    static constexpr uint32_t rix_off = rs_off + kMaxRuns * 4;                 // u16 [kMaxRuns]
    static constexpr uint32_t dlist_off = rix_off + kMaxRuns * 2;              // u16 [kT5Reads]
    static constexpr uint32_t slab_a_off = dlist_off + kT5Reads * 2;         // u32 [kMaxSlabs]
    static constexpr uint32_t slab_pre_off = slab_a_off + kMaxSlabs * 4;       // u32 [kMaxSlabs+1]
    static constexpr uint32_t slab_n_off = slab_pre_off + (kMaxSlabs + 1) * 4; // u32 [kMaxSlabs]
    static constexpr uint32_t slab_per_off = slab_n_off + kMaxSlabs * 4;       // u32 [kMaxSlabs] runs per task of the slab
    static constexpr uint32_t misc_off = (slab_per_off + kMaxSlabs * 4 + 15) & ~15u;
    static constexpr uint32_t lut_off = misc_off + 256;                        // uint4 [2][33] edge masks
    static constexpr uint32_t pk_off = lut_off + 2 * 33 * 16;                  // uint2 [kMaxRuns]: what the pass loop reads
    static constexpr uint32_t cov_off = pk_off + kMaxRuns * 8;                 // uint2 [kT5Reads]: parked coverage update
    static constexpr uint32_t del_off = cov_off + (LVC5_WAIT == 2 ? kT5Reads * 8 : 0);   // uint4 [kT5Reads]: parked deletions
    static constexpr uint32_t total = del_off + (LVC5_WAIT == 2 ? kT5Reads * 16 : 0);
};
constexpr size_t kTile5SmemBytes = Tile5Smem::total;
static_assert((kTile5SmemBytes + 1024) * kTile5CtasPerSM <= 227 * 1024, "the intended CTAs per SM must fit");

// Phase clocks (build with -DLVC5_PHASE_CLOCKS; tools/bench_phases.py reads them through lvc_phase_clocks): thread 0
// of every CTA of the last launch records its SM and clock64() at the phase boundaries below (0 = not reached).
#ifdef LVC5_PHASE_CLOCKS
enum { T5P_ENTRY, T5P_HEADERS, T5P_EXTENTS, T5P_BARRIER_A, T5P_BARRIER_B, T5P_BARRIER_C, T5P_TASKS_END, T5P_EXIT, T5P_N };
constexpr uint32_t kT5PhaseMaxCtas = 1u << 16;
__device__ unsigned long long g_t5_phase[kT5PhaseMaxCtas][1 + T5P_N];     // [cta] = smid, stamps
#define T5_STAMP(k)                                                                                        \
    do {                                                                                                   \
        if (threadIdx.x == 0 && blockIdx.x < kT5PhaseMaxCtas) g_t5_phase[blockIdx.x][1 + (k)] = clock64(); \
    } while (0)
#else
#define T5_STAMP(k) do {} while (0)
#endif

__device__ __forceinline__ uint32_t lop3_xor3(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ uint32_t lop3_maj(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, 0xE8;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
// a ^ (b & c)
__device__ __forceinline__ uint32_t lop3_xor_and(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, 0x78;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
// bit-sliced add of two N-plane numbers (32 independent counters per register): s gets N+1 planes
template <int N>
__device__ __forceinline__ void bs_add(const uint32_t (&a)[N], const uint32_t (&b)[N], uint32_t (&s)[N + 1]) {
    s[0] = a[0] ^ b[0];
    uint32_t c = a[0] & b[0];
#pragma unroll
    for (int k = 1; k < N; ++k) {
        s[k] = lop3_xor3(a[k], b[k], c);
        c = lop3_maj(a[k], b[k], c);
    }
    s[N] = c;
}

// kernel parameters stay in the constant bank even where their address is taken (the warp-per-read helper takes
// the views by reference): without this every thread copies them to local memory first
// PEER: lvc_peer_attach is active -- columns another rank owns are reduced into that rank's tables (lvc_common.cuh)
// QC: quality-code batch (lvc_batch::qual_bits == 2): `b.qual` holds 2-bit codes, 16 bases per 32-bit word; a group of
//     16 bases is staged from ONE code word + 8 sequence bytes (0.75 bytes per base instead of 1.5); the key transform is
//     qc_keys16 (qcode.hpp).  Everything after the keys are staged is the same code.
// B2 (with QC): the batch carries 2-bit BASE codes as well (BatchView::sbits == 2): a group of 16 bases is staged from one
//     word of quality codes + one word of base codes (0.5 bytes per base); b2_onehot16 (qcode.hpp) turns the base codes
//     into the one-hot nibbles the 4-bit form holds.  Everything after the keys are staged is the same code.
template <bool GE_ALL, bool PEER, bool QC = false, bool B2 = false>
__global__ void __launch_bounds__(kT5Threads, kTile5CtasPerSM)
k_deposit_tile5(LVC_GC BatchView b, LVC_GC TableView tv, LVC_GC DepositParams dp, LVC_GC TileParams tp) {
    extern __shared__ __align__(128) unsigned char smem[];
    const uint32_t sbase = smem_u32(smem);
    int32_t* s_rs = reinterpret_cast<int32_t*>(smem + Tile5Smem::rs_off);
    uint16_t* s_rix = reinterpret_cast<uint16_t*>(smem + Tile5Smem::rix_off);
    uint16_t* s_dlist = reinterpret_cast<uint16_t*>(smem + Tile5Smem::dlist_off);
    uint32_t* s_slab_a = reinterpret_cast<uint32_t*>(smem + Tile5Smem::slab_a_off);
    uint32_t* s_slab_pre = reinterpret_cast<uint32_t*>(smem + Tile5Smem::slab_pre_off);
    uint32_t* s_slab_n = reinterpret_cast<uint32_t*>(smem + Tile5Smem::slab_n_off);
    uint32_t* s_slab_per = reinterpret_cast<uint32_t*>(smem + Tile5Smem::slab_per_off);
    uint4* s_lut = reinterpret_cast<uint4*>(smem + Tile5Smem::lut_off);
    uint32_t* s_misc = reinterpret_cast<uint32_t*>(smem + Tile5Smem::misc_off);
    uint2* s_pk = reinterpret_cast<uint2*>(smem + Tile5Smem::pk_off);
    // s_misc: [2] task counter  [4] window max end column (long reads only)  [6] deferred reads
    //         [5] run table end (overflow only)
    //         [8..11] min read byte, max read end byte, max reference span, max end column   [32..39] runs per warp
    const uint32_t k_smem = sbase + Tile5Smem::key_off + kSlack;      // staged keys start here

    // let a kernel launched with programmatic stream serialization (the genotype pass) become resident while this
    // grid drains; it still waits for this grid's completion before reading
    asm volatile("griddepcontrol.launch_dependents;");
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#ifdef LVC5_PHASE_CLOCKS
    if (tid == 0 && blockIdx.x < kT5PhaseMaxCtas) {
        uint32_t smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        g_t5_phase[blockIdx.x][0] = smid;
        for (int k = 1; k < T5P_N; ++k) g_t5_phase[blockIdx.x][1 + k] = 0;
    }
    T5_STAMP(T5P_ENTRY);
#endif
    const uint32_t qprim4 = tp.qprim * 0x01010101u;
    const int mbq = dp.min_bq < 1 ? 1 : (dp.min_bq > 128 ? 128 : dp.min_bq);
    const uint32_t ge_add4 = (uint32_t)(0x80 - mbq) * 0x01010101u;

    // ---- (1) this chunk's read headers: issue the global loads first, then set up shared memory
    const uint32_t cur = blockIdx.x;
    ReadHdr hd;
    uint64_t so0;
    if (b.hdr_lazy) {
        const uint32_t i = cur * kT5Reads + (uint32_t)tid;
        hd.keep = i < b.n_reads ? (uint32_t)b.keep[i] : 0u;
    } else hdr_load1<kT5Reads>(b, cur, tid, hd, so0);
    uint32_t* sc = s_misc + 8;                                       // per-chunk scalars
    uint32_t* wc = s_misc + 32;                                      // runs per warp
    if (tid == 0) {
        s_misc[6] = 0;
        sc[0] = 0xFFFFFFFFu; sc[1] = 0; sc[2] = 0; sc[3] = 0;
    }
    // a chunk in which the host admission (htslib max_depth) dropped every read ends here, after ONE load per thread:
    // nothing else of its headers is waited for
    if (!__syncthreads_or(hd.keep & 1u)) { T5_STAMP(T5P_EXIT); return; }
    if (b.hdr_lazy) hdr_load1<kT5Reads>(b, cur, tid, hd, so0);
    if (tid < 66) {
        // edge masks of a 32-column unit, one nibble per column: [0][n] keeps the columns >= n, [1][n] the columns < n
        const uint32_t n = tid < 33 ? (uint32_t)tid : (uint32_t)tid - 33u;
        uint32_t m[4];
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            const int32_t d = (int32_t)n - 8 * w;                      // columns of word w below n
            const uint32_t below = d <= 0 ? 0u : (d >= 8 ? 0xFFFFFFFFu : ((1u << (4 * d)) - 1u));
            m[w] = tid < 33 ? ~below : below;
        }
        s_lut[tid] = make_uint4(m[0], m[1], m[2], m[3]);
    }
    hdr_load2(b, hd, dp.min_mq);       // CIGAR ops, only for reads that pass the read-level filter
    // a chunk in which no read passes the read-level filter ends here
    if (!__syncthreads_or(read_passes_filter(hd.flag, hd.mapq, hd.keep, dp.min_mq))) { T5_STAMP(T5P_EXIT); return; }
    T5_STAMP(T5P_HEADERS);
    // Up to here only the batch was read.  The tables may still be in use by the previous kernel of the stream (this
    // kernel is launched with programmatic stream serialization): wait for it before the first table access.
#if LVC5_WAIT == 0
    asm volatile("griddepcontrol.wait;" ::: "memory");
#endif
    // byte extent of the reads that pass the read-level filter (a superset of what will be deposited):
    // known before the CIGARs arrive, so the bulk copy overlaps classification
    const uint32_t so_rel = hd.so - (uint32_t)so0, so1_rel = hd.so1 - (uint32_t)so0;
    // "every base of the read is A, C, G or T" (keep bit 1).  A base-code batch holds nothing else by construction: what
    // was another code had a quality below the threshold and is code 0 now, which the quality test still drops -- so a read
    // with a no-call takes the tiled path there instead of the one-warp-per-read path
    const bool acgt = B2 || (hd.keep & 2u);
    {
        const bool pass = read_passes_filter(hd.flag, hd.mapq, hd.keep, dp.min_mq) && acgt &&
                          (so1_rel - so_rel) <= kMaxReadBytes && so1_rel > so_rel;
        uint32_t lo = pass ? so_rel : 0xFFFFFFFFu, hi = pass ? so1_rel : 0u;
        lo = __reduce_min_sync(0xFFFFFFFFu, lo);
        hi = __reduce_max_sync(0xFFFFFFFFu, hi);
        if (lane == 0 && hi) { atomicMin(&sc[0], lo); atomicMax(&sc[1], hi); }
    }
    __syncthreads();
    T5_STAMP(T5P_EXTENTS);
    const uint32_t min_rel = sc[0], max_rel = sc[1];
    if (max_rel == 0) {
        // no read of this chunk can take the tiled path: hand over what must be deposited and leave
        if (read_passes_filter(hd.flag, hd.mapq, hd.keep, dp.min_mq) && hd.nc) {
            bool any_ref = false;
            for (uint32_t k = 0; k < hd.nc; ++k) any_ref |= op_consumes_ref(b.cigar[hd.c0 + k] & 15u);
            if (any_ref) s_dlist[atomicAdd(&s_misc[6], 1u)] = (uint16_t)tid;
        }
        __syncthreads();
        const uint32_t n_def = s_misc[6];
        asm volatile("griddepcontrol.wait;" ::: "memory");
        for (uint32_t d = warp; d < n_def; d += kT5Warps) (PEER ? deposit_read_warp_peer : deposit_read_warp)(b, tv, dp, cur * kT5Reads + s_dlist[d], lane);
        T5_STAMP(T5P_EXIT);
        return;
    }
    // staging base: 16-byte aligned start of the first such read
    const uint64_t base_abs = (so0 + min_rel) & ~15ull;
    const uint32_t base_rel = (uint32_t)(base_abs - so0);            // may wrap below zero: used mod 2^32
#ifndef LVC5_NO_PREFETCH
    {
        // ask L2 for the chunk's payload now: classification and the run table hide the DRAM latency of the staging
        // loads (measured on config 5: 0.524 -> 0.498 ms).  The 128-byte lines of the quality array, then those of the
        // base array, numbered from the (16-base aligned) staging base: one line per thread for a chunk of short reads
        const uint32_t span = max_rel - base_rel;                    // bases from the staging base to the last read's end
        constexpr int qsh = QC ? 2 : 0, ssh = B2 ? 2 : 1;            // log2 bases per byte
        const uint32_t nq = (((span + (1u << qsh) - 1u) >> qsh) + 127u) >> 7;
        const uint32_t ns = (((span + (1u << ssh) - 1u) >> ssh) + 127u) >> 7;
        const uint8_t* pq = b.qual + (base_abs >> qsh);
        const uint8_t* ps = b.seq4 + (base_abs >> ssh);
        for (uint32_t l = (uint32_t)tid; l < nq + ns; l += kT5Threads)
            asm volatile("prefetch.global.L2 [%0];" ::"l"(l < nq ? pq + 128u * l : ps + 128u * (l - nq)));
    }
#endif
    {
        const uint32_t chunk0 = cur * kT5Reads;
        // ---- (2) classify this thread's read: filter, match runs, deletion entries
        int32_t run_pos[kMaxRunsPerRead] = {0, 0, 0};
        uint32_t run_len[kMaxRunsPerRead] = {0, 0, 0}, run_q[kMaxRunsPerRead] = {0, 0, 0};
        int32_t del_pos[kMaxDelsPerRead] = {0, 0};
        uint32_t del_len[kMaxDelsPerRead] = {0, 0}, del_q[kMaxDelsPerRead] = {0, 0};
        uint32_t nr = 0, nd = 0, rspan = 0;
        bool defer = false;
        const bool rpass = read_passes_filter(hd.flag, hd.mapq, hd.keep, dp.min_mq);
        // warp-uniform shortcut: every read of the warp that passes the filter is one match op (150M): no CIGAR walk
        const uint32_t l0 = hd.cg0 >> 4;
        const bool one_m = hd.nc == 1 && op_is_match(hd.cg0 & 15u) && acgt && (hd.so1 - hd.so) <= kMaxReadBytes &&
                           l0 >= 1u && l0 <= 65535u;
        if (__all_sync(0xFFFFFFFFu, !rpass || one_m)) {
            if (rpass) {
                if (hd.pos < 0 || (int64_t)hd.pos + l0 > tv.G) atomicAdd(&tv.status[ST_RANGE_ERR], 1u);
                else { nr = 1; run_pos[0] = hd.pos; run_len[0] = l0; run_q[0] = 0; rspan = l0; }
            }
        } else if (__all_sync(0xFFFFFFFFu, !rpass || (hd.nc >= 1u && hd.nc <= 3u && acgt &&
                                                        (hd.so1 - hd.so) <= kMaxReadBytes))) {
            // second warp-uniform shortcut: at most 3 CIGAR ops per read (one indel or soft clips), all of them
            // already in registers: straight-line code, same results as the general walk below
            if (rpass) {
                const bool p1 = hd.nc > 1u, p2 = hd.nc > 2u;
                const uint32_t o0 = hd.cg0 & 15u, o1 = hd.cg1 & 15u, o2 = hd.cg2 & 15u;
                const uint32_t n0 = hd.cg0 >> 4, n1 = p1 ? hd.cg1 >> 4 : 0u, n2 = p2 ? hd.cg2 >> 4 : 0u;
                const bool m0 = op_is_match(o0), m1 = p1 && op_is_match(o1), m2 = p2 && op_is_match(o2);
                const bool d0 = o0 == 2 || o0 == 3, d1 = p1 && (o1 == 2 || o1 == 3), d2 = p2 && (o2 == 2 || o2 == 3);
                const uint32_t qc0 = op_consumes_query(o0) ? n0 : 0u, qc1 = (p1 && op_consumes_query(o1)) ? n1 : 0u,
                               qc2 = (p2 && op_consumes_query(o2)) ? n2 : 0u;
                const uint32_t rc0 = (m0 || d0) ? n0 : 0u, rc1 = (m1 || d1) ? n1 : 0u, rc2 = (m2 || d2) ? n2 : 0u;
                const uint32_t qo1 = qc0, qo2 = qc0 + qc1, lq = qo2 + qc2;
                const uint32_t ro1 = rc0, ro2 = rc0 + rc1;
                rspan = ro2 + rc2;
                // match runs: a run starts at a match op that does not follow a match op
                const bool s0 = m0, s1 = m1 && !m0, s2 = m2 && !m1;
                const uint32_t len2 = n2, len1 = n1 + (m2 ? n2 : 0u), len0 = n0 + (m1 ? len1 : 0u);
                nr = (uint32_t)s0 + (uint32_t)s1 + (uint32_t)s2;
                if (s0) { run_pos[0] = hd.pos; run_len[0] = len0; run_q[0] = 0; }
                else if (s1) { run_pos[0] = hd.pos + (int32_t)ro1; run_len[0] = len1; run_q[0] = qo1; }
                else if (s2) { run_pos[0] = hd.pos + (int32_t)ro2; run_len[0] = len2; run_q[0] = qo2; }
                if (s0 && s2) { run_pos[1] = hd.pos + (int32_t)ro2; run_len[1] = len2; run_q[1] = qo2; }
                // deletion / ref-skip entries, in op order; their quality (the NEXT query base, 0 past the end) is
                // requested here and tested where the entries are deposited
                const uint32_t ndel = (uint32_t)d0 + (uint32_t)d1 + (uint32_t)d2;
                bool tileable = ndel <= (uint32_t)kMaxDelsPerRead;
                if (tileable && ndel) {
                    const uint64_t qrd0 = so0 + so_rel;
                    auto qrd = [&](uint32_t k) -> uint32_t { return QC ? batch_qual(b, qrd0 + k) : (uint32_t)b.qual[qrd0 + k]; };
                    if (d0) { del_pos[0] = hd.pos; del_len[0] = n0; del_q[0] = 0u < lq ? qrd(0) : 0u; nd = 1; }
                    if (d1) {
                        const uint32_t qv = qo1 < lq ? qrd(qo1) : 0u;
                        if (nd == 0) { del_pos[0] = hd.pos + (int32_t)ro1; del_len[0] = n1; del_q[0] = qv; }
                        else { del_pos[1] = hd.pos + (int32_t)ro1; del_len[1] = n1; del_q[1] = qv; }
                        ++nd;
                    }
                    if (d2) {
                        const uint32_t qv = qo2 < lq ? qrd(qo2) : 0u;
                        if (nd == 0) { del_pos[0] = hd.pos + (int32_t)ro2; del_len[0] = n2; del_q[0] = qv; }
                        else { del_pos[1] = hd.pos + (int32_t)ro2; del_len[1] = n2; del_q[1] = qv; }
                        ++nd;
                    }
                }
                bool any_ref = m0 || m1 || m2 || d0 || d1 || d2;
                if (tileable && any_ref && (hd.pos < 0 || (int64_t)hd.pos + rspan > tv.G)) {
                    atomicAdd(&tv.status[ST_RANGE_ERR], 1u);
                    nr = 0; nd = 0; rspan = 0; any_ref = false;
                }
                if ((nr >= 1 && run_len[0] > 65535u) || (nr >= 2 && run_len[1] > 65535u)) tileable = false;
                if (!tileable) { defer = any_ref; nr = 0; nd = 0; rspan = 0; }
                else if (!any_ref) { nr = 0; nd = 0; rspan = 0; }
            }
        } else if (rpass) {
            bool tileable = hd.nc <= (uint32_t)kMaxCigarTile && hd.nc > 0 && (hd.so1 - hd.so) <= kMaxReadBytes &&
                            acgt;
            uint32_t lq = 0;
            bool any_ref = false;
            if (tileable) {
                // l_qseq first (a deletion at the very end tests a quality that does not exist)
                for (uint32_t k = 0; k < hd.nc; ++k) {
                    const uint32_t c = k == 0 ? hd.cg0 : (k == 1 ? hd.cg1 : (k == 2 ? hd.cg2 : b.cigar[hd.c0 + k]));
                    if (op_consumes_query(c & 15u)) lq += c >> 4;
                }
                uint32_t qi = 0;
                int32_t r = hd.pos;
                bool prev_match = false;
                for (uint32_t k = 0; k < hd.nc && tileable; ++k) {
                    const uint32_t c = k == 0 ? hd.cg0 : (k == 1 ? hd.cg1 : (k == 2 ? hd.cg2 : b.cigar[hd.c0 + k]));
                    const uint32_t op = c & 15u, l = c >> 4;
                    if (op_is_match(op)) {
                        any_ref = true;
                        if (prev_match) {
                            if (nr == 1) run_len[0] += l; else if (nr == 2) run_len[1] += l; else run_len[2] += l;
                        } else if (nr == (uint32_t)kMaxRunsPerRead) tileable = false;
                        else {
                            if (nr == 0) { run_pos[0] = r; run_len[0] = l; run_q[0] = qi; }
                            else if (nr == 1) { run_pos[1] = r; run_len[1] = l; run_q[1] = qi; }
                            else { run_pos[2] = r; run_len[2] = l; run_q[2] = qi; }
                            ++nr;
                        }
                        qi += l; r += (int32_t)l; prev_match = true;
                    } else {
                        prev_match = false;
                        if (op == 2 || op == 3) {
                            any_ref = true;
                            // kept iff the NEXT query base passes the quality rule (0 if past the end).  The quality
                            // is only requested here; it is tested where the entries are deposited, after the barrier,
                            // so its latency does not hold up the chunk
                            if (nd == (uint32_t)kMaxDelsPerRead) tileable = false;
                            else {
                                const uint32_t q = qi < lq ? (QC ? batch_qual(b, so0 + so_rel + qi) : (uint32_t)b.qual[so0 + so_rel + qi]) : 0u;
                                if (nd == 0) { del_pos[0] = r; del_len[0] = l; del_q[0] = q; }
                                else { del_pos[1] = r; del_len[1] = l; del_q[1] = q; }
                                ++nd;
                            }
                            r += (int32_t)l;
                        } else if (op == 1 || op == 4) qi += l;
                    }
                }
                rspan = (uint32_t)(r - hd.pos);
                if (tileable && any_ref && (hd.pos < 0 || (int64_t)hd.pos + rspan > tv.G)) {
                    atomicAdd(&tv.status[ST_RANGE_ERR], 1u);
                    nr = 0; nd = 0; rspan = 0; tileable = true; any_ref = false;
                }
#pragma unroll
                for (int k = 0; k < kMaxRunsPerRead; ++k) if ((uint32_t)k < nr && run_len[k] > 65535u) tileable = false;
            }
            if (!tileable) {
                // a record with no reference-consuming op at all is skipped everywhere
                if (!any_ref)
                    for (uint32_t k = 0; k < hd.nc; ++k) any_ref |= op_consumes_ref(b.cigar[hd.c0 + k] & 15u);
                defer = any_ref;
                nr = 0; nd = 0; rspan = 0;
            } else if (!any_ref) { nr = 0; nd = 0; rspan = 0; }
        }
        // ---- (3) warp-level compaction bookkeeping + chunk extents, then ONE barrier
        const uint32_t b1 = __ballot_sync(0xFFFFFFFFu, nr >= 1), b2 = __ballot_sync(0xFFFFFFFFu, nr >= 2),
                       b3 = __ballot_sync(0xFFFFFFFFu, nr >= 3);
        const uint32_t lt = (1u << lane) - 1u;
        const uint32_t wprefix = __popc(b1 & lt) + __popc(b2 & lt) + __popc(b3 & lt);
        {
            uint32_t sp = nr ? rspan : 0u;
            int32_t ce = nr ? (int32_t)(hd.pos + rspan) : 0;
            sp = __reduce_max_sync(0xFFFFFFFFu, sp);
            ce = __reduce_max_sync(0xFFFFFFFFu, ce);
            if (lane == 0) {
                wc[warp] = __popc(b1) + __popc(b2) + __popc(b3);
                if (sp) { atomicMax(&sc[2], sp); atomicMax(reinterpret_cast<int32_t*>(&sc[3]), ce); }
            }
        }
        __syncthreads();                                                   // barrier A
        T5_STAMP(T5P_BARRIER_A);
        uint32_t n_runs = 0, my_base = 0;
#pragma unroll
        for (int w = 0; w < kT5Warps; ++w) {
            const uint32_t c = wc[w];
            if (w < warp) my_base += c;
            n_runs += c;
        }
        const uint32_t maxspan = sc[2];
        const int32_t chunk_cmax = (int32_t)sc[3];
        if (n_runs > (uint32_t)kMaxRuns) {                                // run table full (indel-dense chunk): rare
            // reads whose runs do not fit are handed to the general kernel; the table ends where the first
            // such read would have started (prefix sums are monotone, so everything after it overflows too)
            if (tid == 0) s_misc[5] = 0;
            __syncthreads();
            const uint32_t my_end = my_base + wprefix + nr;
            if (nr && my_end > (uint32_t)kMaxRuns) { defer = true; nr = 0; nd = 0; rspan = 0; }
            uint32_t ok_end = nr ? my_end : 0u;
            ok_end = __reduce_max_sync(0xFFFFFFFFu, ok_end);
            if (lane == 0) atomicMax(&s_misc[5], ok_end);
            __syncthreads();
            n_runs = s_misc[5];
        }
        const bool active = rspan != 0;                                   // deposited by this kernel
        if (defer) s_dlist[atomicAdd(&s_misc[6], 1u)] = (uint16_t)tid;
        // coverage difference array (one atomic per distinct start / end among the warp's reads) and deletion entries:
        // the first table accesses of the chunk.  All 32 lanes of every warp call this together.
        auto deposit_cov = [&](bool act, int32_t rpos, uint32_t span, uint32_t n_del, int32_t dpos0, uint32_t dlen0, int32_t dpos1,
                               uint32_t dlen1) {
            asm volatile("griddepcontrol.wait;" ::: "memory");
            const int32_t ks = act ? rpos : (int32_t)(0x80000000u + lane);
            const uint32_t ms = __match_any_sync(0xFFFFFFFFu, ks);
            if (act && lane == __ffs(ms) - 1) atomicAdd(PEER ? covdiff_cell(tv, rpos) : tv.covdiff + rpos, (int32_t)__popc(ms));
            const int32_t ke = act ? (int32_t)(rpos + span) : (int32_t)(0x80000000u + lane);
            const uint32_t me = __match_any_sync(0xFFFFFFFFu, ke);
            if (act && lane == __ffs(me) - 1) atomicAdd(PEER ? covdiff_cell(tv, (int64_t)rpos + span) : tv.covdiff + rpos + span, -(int32_t)__popc(me));
            if (n_del) {
                for (uint32_t j = 0; j < dlen0; ++j) atomicAdd(PEER ? dels_cell(tv, (int64_t)dpos0 + j) : tv.dels + dpos0 + j, 1u);
                for (uint32_t j = 0; j < dlen1; ++j) atomicAdd(PEER ? dels_cell(tv, (int64_t)dpos1 + j) : tv.dels + dpos1 + j, 1u);
            }
        };
        // deletion entries that passed the quality rule (a failed one keeps length 0)
        const uint32_t dl0 = (nd >= 1 && (int)del_q[0] >= dp.min_bq) ? del_len[0] : 0u;
        const uint32_t dl1 = (nd >= 2 && (int)del_q[1] >= dp.min_bq) ? del_len[1] : 0u;
#if LVC5_WAIT == 2
        // parked: the update is issued once the first window is staged (or right away if nothing is staged)
        uint2* s_cov = reinterpret_cast<uint2*>(smem + Tile5Smem::cov_off);
        uint4* s_del = reinterpret_cast<uint4*>(smem + Tile5Smem::del_off);
        s_cov[tid] = make_uint2((uint32_t)hd.pos, (active ? rspan : 0u) | ((dl0 | dl1) ? 0x80000000u : 0u));
        if (dl0 | dl1) s_del[tid] = make_uint4((uint32_t)del_pos[0], dl0, (uint32_t)del_pos[1], dl1);
        bool cov_parked = true;
        auto deposit_parked = [&]() {
            if (!cov_parked) return;                          // (uniform over the CTA)
            cov_parked = false;
            const uint2 cv = s_cov[tid];
            uint4 dv = make_uint4(0, 0, 0, 0);
            if (cv.y & 0x80000000u) dv = s_del[tid];
            const uint32_t span = cv.y & 0x7FFFFFFFu;
            deposit_cov(span != 0, (int32_t)cv.x, span, cv.y >> 31, (int32_t)dv.x, dv.y, (int32_t)dv.z, dv.w);
        };
        if (!n_runs) deposit_parked();
#else
        deposit_cov(active, hd.pos, rspan, (dl0 | dl1) ? 1u : 0u, del_pos[0], dl0, del_pos[1], dl1);
#endif
        if (n_runs) {
            if (nr) {
                const uint32_t off = so_rel - base_rel;                   // read's first byte relative to the base
                const uint32_t win = off / kT5WinStride;
                const uint32_t idx0 = my_base + wprefix;
#pragma unroll
                for (int k = 0; k < kMaxRunsPerRead; ++k) {
                    if ((uint32_t)k < nr) {
                        const uint32_t idx = idx0 + k;
                        s_rs[idx] = hd.pos;
                        s_rix[idx] = (uint16_t)((win << 8) | (uint32_t)tid);
                        // (start column, key offset inside the read's window | length << 16): one 8-byte load per unit
                        s_pk[idx] = make_uint2((uint32_t)run_pos[k], ((off + run_q[k] - win * kT5WinStride) & 0xFFFFu) | (run_len[k] << 16));
                    }
                }
            }
            __syncthreads();                                               // barrier B: run table visible
            T5_STAMP(T5P_BARRIER_B);
        }

        // ---- (5) staged windows of runs (one per chunk unless reads are long)
        if (n_runs) {
            const uint32_t n_win = (uint32_t)(s_rix[n_runs - 1] >> 8) + 1u;
            uint32_t a0 = 0;
            for (uint32_t win = 0; win < n_win; ++win) {
                uint32_t a1 = n_runs;
                if (win + 1 < n_win) {            // first run of a later window
                    uint32_t lo = a0, hi = n_runs;
                    while (lo < hi) { const uint32_t m = (lo + hi) >> 1; if ((uint32_t)(s_rix[m] >> 8) <= win) lo = m + 1; else hi = m; }
                    a1 = lo;
                }
                if (a1 == a0 && win > 0) continue;
                const uint32_t w_rel = win * kT5WinStride;                   // window start relative to the base
                const uint64_t qbeg = base_abs + w_rel;                    // 16-byte aligned
                // column range of these runs
                const int32_t cmin = s_rs[a0];
                int32_t cmax = chunk_cmax;                                 // chunk-wide (an upper bound for any window)
                if (n_win > 1) {                                           // long reads: exact range of this window's runs
                    __syncthreads();
                    if (tid == 0) s_misc[4] = 0;
                    __syncthreads();
                    int32_t e = 0;
                    for (uint32_t r = a0 + tid; r < a1; r += kT5Threads) e = max(e, (int32_t)s_pk[r].x + (int32_t)(s_pk[r].y >> 16));
                    e = __reduce_max_sync(0xFFFFFFFFu, e);
                    if (lane == 0 && e) atomicMax(reinterpret_cast<int32_t*>(&s_misc[4]), e);
                    __syncthreads();
                    cmax = (int32_t)s_misc[4];
                }
                // Task table of one column window: per 32-column slab the candidate run range and the exclusive scan of
                // the task counts.  One warp does it, before its share of the staging, and the other warps wait for it at
                // barrier C, so the two lower bounds of a slab over the read starts of the runs (non-decreasing: a batch is
                // coordinate sorted) are independent searches on two lanes: lane s finds the end of slab s's range (the
                // first run whose read starts at or after the slab's end), lane 8 + s its first run (the first run whose
                // read starts after slab start - max span).  Half the chain of dependent shared loads of one lane doing both.
                auto slab_setup = [&](int32_t wc0) {
                    const int nslab = min(kMaxSlabs, (cmax - wc0 + kSlabCols - 1) / kSlabCols);
                    uint32_t cnt = 0, first_run = 0;
                    {
                        static_assert(kMaxSlabs == 8, "two searches per slab on lanes s and 8 + s");
                        const int sl = lane & 15;
                        const int32_t s_lo = wc0 + (sl & 7) * kSlabCols;
                        const int64_t thr = sl < 8 ? (int64_t)s_lo + kSlabCols - 1 : (int64_t)s_lo - (int64_t)maxspan;
                        uint32_t lo = a0, hi = a1;               // first run whose read starts after thr
                        while (lo < hi) {
                            const uint32_t m = (lo + hi) >> 1;
                            if ((int64_t)s_rs[m] <= thr) lo = m + 1; else hi = m;
                        }
                        const uint32_t fr = __shfl_down_sync(0xFFFFFFFFu, lo, 8);
                        if (lane < nslab) { first_run = fr; cnt = lo - fr; }
                    }
                    // tasks of a slab are equal shares of its candidate runs, <= kTask5Runs each (whole passes of 32)
                    const uint32_t groups = (cnt + kTask5Runs - 1) / kTask5Runs;
                    const uint32_t per = groups ? (((cnt + groups - 1) / groups + 31u) & ~31u) : 0u;
                    uint32_t incl = groups;
#pragma unroll
                    for (int d = 1; d < kMaxSlabs; d <<= 1) {
                        const uint32_t up = __shfl_up_sync(0xFFFFFFFFu, incl, d);
                        if (lane >= d) incl += up;
                    }
                    if (lane < nslab) {
                        s_slab_a[lane] = first_run; s_slab_n[lane] = cnt; s_slab_pre[lane] = incl - groups; s_slab_per[lane] = per;
                    }
                    if (lane == nslab - 1) s_slab_pre[nslab] = incl;
                    if (lane == 0) s_misc[2] = 0;
                };
                // ---- stage this window as KEYS: coalesced 16-byte loads, 16 bases per step, written in place once
                if (a1 > a0) {
                    const uint64_t qend_all = so0 + max_rel;
                    const uint64_t qend = qend_all < qbeg + kT5KeyCapBases ? qend_all : qbeg + kT5KeyCapBases;
                    const uint32_t n_grp = (uint32_t)(((qend - qbeg) + 15) >> 4);
                    const uint32_t chunk_ord = dp.ord_base + chunk0;
                    const uint4* gq = reinterpret_cast<const uint4*>(b.qual + qbeg);
                    const uint2* gs = reinterpret_cast<const uint2*>(b.seq4 + (qbeg >> 1));
                    // one group = 16 bases: 16 quality bytes + 8 sequence bytes -> 16 keys
                    auto stage_group = [&](uint32_t gg, const uint4& q, const uint2& sraw) {
                        // base nibbles in little-endian nibble order (base k at bits 4k)
                        const uint32_t s0 = bitsel(sraw.x >> 4, sraw.x << 4, 0x0F0F0F0Fu);
                        const uint32_t s1 = bitsel(sraw.y >> 4, sraw.y << 4, 0x0F0F0F0Fu);
                        // Qualities below 128 (every real file): no carries between bytes, so per word
                        //   bit 7 of (q ^ qprim) + 0x7F = "differs from the primary quality"
                        //   bit 7 of  q + (0x80 - minBQ) = "passes the base-quality threshold"
                        const uint32_t t0 = (q.x ^ qprim4) + 0x7F7F7F7Fu, t1 = (q.y ^ qprim4) + 0x7F7F7F7Fu;
                        const uint32_t t2 = (q.z ^ qprim4) + 0x7F7F7F7Fu, t3 = (q.w ^ qprim4) + 0x7F7F7F7Fu;
                        uint32_t cold = q.x | q.y | q.z | q.w;                       // a byte >= 128: exact path
                        if (GE_ALL) cold |= t0 | t1 | t2 | t3;
                        else cold |= (t0 & (q.x + ge_add4)) | (t1 & (q.y + ge_add4)) | (t2 & (q.z + ge_add4)) |
                                     (t3 & (q.w + ge_add4));                          // passing, not primary
                        // "differs" flags of the even / odd bases gathered and widened to bytes (PRMT sign mode)
                        uint32_t k0 = s0 & ~bitsel(prmt_sign(t0, t1, 0xECA8u), prmt_sign(t0, t1, 0xFDB9u), 0x0F0F0F0Fu);
                        uint32_t k1 = s1 & ~bitsel(prmt_sign(t2, t3, 0xECA8u), prmt_sign(t2, t3, 0xFDB9u), 0x0F0F0F0Fu);
                        if (cold & 0x80808080u) {
                            // rare: exact flags; a passing quality other than the primary one is deposited individually
                            k0 = 0; k1 = 0;
#pragma unroll 1
                            for (int w = 0; w < 4; ++w) {
                                const uint32_t qv = w == 0 ? q.x : (w == 1 ? q.y : (w == 2 ? q.z : q.w));
                                const uint32_t e80 = bytes_eq80(qv, qprim4);
                                const uint32_t sx = ((w < 2) ? s0 : s1) >> (16 * (w & 1));     // these 4 bases' nibbles
                                const uint32_t kw = sx & flags_to_nibbles(e80);
                                if (w < 2) k0 |= kw << (16 * (w & 1)); else k1 |= kw << (16 * (w & 1));
                                uint32_t m80 = (GE_ALL ? 0x80808080u : bytes_ge80(qv, ge_add4)) & ~e80;
                                while (m80) {
                                    const int bb = (__ffs(m80) - 1) >> 3;
                                    m80 &= ~(0x80u << (8 * bb));
                                    const uint32_t x_win = 16u * gg + 4u * (uint32_t)w + (uint32_t)bb;
                                    uint32_t lo = a0, hi = a1;             // last run whose payload starts at or before x_win
                                    while (lo < hi) { const uint32_t m = (lo + hi) >> 1; if ((s_pk[m].y & 0xFFFFu) <= x_win) lo = m + 1; else hi = m; }
                                    if (lo > a0) {
                                        const uint2 pk = s_pk[lo - 1];
                                        const uint32_t r = lo - 1, d = x_win - (pk.y & 0xFFFFu);
#if LVC5_WAIT == 2
                                        asm volatile("griddepcontrol.wait;" ::: "memory");
#endif
                                        if (d < (pk.y >> 16))
                                            deposit_base<PEER>(tv, dp, (int64_t)(int32_t)pk.x + d, (sx >> (4 * bb)) & 15u,
                                                         (qv >> (8 * bb)) & 255u, chunk_ord + (s_rix[r] & 255u));
                                    }
                                }
                            }
                        }
                        asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(k_smem + 8u * gg), "r"(k0), "r"(k1) : "memory");
                    };
                    // two groups per iteration, loaded then reduced.  (A software-pipelined version with the next two
                    // groups in flight costs 12 more live registers under the 48-register cap and measured 4 % slower:
                    // with 5 CTAs per SM the load latency is covered by the other CTAs.  One group per iteration is 8 % slower.)
                    // the same for a quality-code batch: one word of 16 codes + 8 sequence bytes -> 16 keys
                    auto stage_group_qc = [&](uint32_t gg, uint32_t w, const uint2& sraw) {
                        // base nibbles in little-endian nibble order: from the 4-bit form by swapping the nibbles of every
                        // byte, from the 2-bit form (sraw.x = 16 codes) by b2_onehot16
                        uint32_t s0, s1;
                        if (B2) b2_onehot16(sraw.x, s0, s1);
                        else { s0 = bitsel(sraw.x >> 4, sraw.x << 4, 0x0F0F0F0Fu); s1 = bitsel(sraw.y >> 4, sraw.y << 4, 0x0F0F0F0Fu); }
                        uint32_t k0, k1;
                        qc_keys16(s0, s1, w, tp.qc_pcode, k0, k1);
                        if (tp.qc_cold) {
                            // some code other than the primary one passes the threshold (uniform over the grid): its bases
                            // are deposited individually, exactly as in the byte form
                            uint32_t cold = qc_cold_flags(w, tp.qc_cold);
                            while (cold) {
                                const uint32_t bb = (uint32_t)(__ffs(cold) - 1) >> 1;          // base 0..15 of the group
                                cold &= cold - 1;
                                const uint32_t x_win = 16u * gg + bb;
                                uint32_t lo = a0, hi = a1;             // last run whose payload starts at or before x_win
                                while (lo < hi) { const uint32_t m = (lo + hi) >> 1; if ((s_pk[m].y & 0xFFFFu) <= x_win) lo = m + 1; else hi = m; }
                                if (lo > a0) {
                                    const uint2 pk = s_pk[lo - 1];
                                    const uint32_t r = lo - 1, d = x_win - (pk.y & 0xFFFFu);
#if LVC5_WAIT == 2
                                    asm volatile("griddepcontrol.wait;" ::: "memory");
#endif
                                    if (d < (pk.y >> 16))
                                        deposit_base<PEER>(tv, dp, (int64_t)(int32_t)pk.x + d, ((bb < 8u ? s0 : s1) >> (4u * (bb & 7u))) & 15u,
                                                           (b.qdict >> (8u * ((w >> (2u * bb)) & 3u))) & 255u, chunk_ord + (s_rix[r] & 255u));
                                }
                            }
                        }
                        asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(k_smem + 8u * gg), "r"(k0), "r"(k1) : "memory");
                    };
                    if (warp == 0 && cmin < cmax) slab_setup(cmin);
                    if (QC && B2) {
                        const uint32_t* gc = reinterpret_cast<const uint32_t*>(b.qual + (qbeg >> 2));
                        const uint32_t* gb = reinterpret_cast<const uint32_t*>(b.seq4 + (qbeg >> 2));
                        for (uint32_t g = tid; g < n_grp; g += 2 * kT5Threads) {
                            const bool hasB = g + kT5Threads < n_grp;
                            const uint32_t wA = __ldcs(gc + g);
                            const uint32_t bA = __ldcs(gb + g);
                            uint32_t wB = 0, bB = 0;
                            if (hasB) { wB = __ldcs(gc + g + kT5Threads); bB = __ldcs(gb + g + kT5Threads); }
                            stage_group_qc(g, wA, make_uint2(bA, 0));
                            if (hasB) stage_group_qc(g + kT5Threads, wB, make_uint2(bB, 0));
                        }
                    } else if (QC) {
                        const uint32_t* gc = reinterpret_cast<const uint32_t*>(b.qual + (qbeg >> 2));
                        for (uint32_t g = tid; g < n_grp; g += 2 * kT5Threads) {
                            const bool hasB = g + kT5Threads < n_grp;
                            const uint32_t wA = __ldcs(gc + g);
                            const uint2 sA = __ldcs(gs + g);
                            uint32_t wB = 0;
                            uint2 sB = make_uint2(0, 0);
                            if (hasB) { wB = __ldcs(gc + g + kT5Threads); sB = __ldcs(gs + g + kT5Threads); }
                            stage_group_qc(g, wA, sA);
                            if (hasB) stage_group_qc(g + kT5Threads, wB, sB);
                        }
                    } else
                    for (uint32_t g = tid; g < n_grp; g += 2 * kT5Threads) {
                        const bool hasB = g + kT5Threads < n_grp;
                        // streaming loads: the payload is read exactly once and should not displace the few hot lines
                        // (plane pointers, key LUT) in the 38 KB of L1 left beside the shared memory: -4 %
                        const uint4 qA = __ldcs(gq + g);
                        const uint2 sA = __ldcs(gs + g);
                        uint4 qB = make_uint4(0, 0, 0, 0);
                        uint2 sB = make_uint2(0, 0);
                        if (hasB) { qB = __ldcs(gq + g + kT5Threads); sB = __ldcs(gs + g + kT5Threads); }
                        stage_group(g, qA, sA);
                        if (hasB) stage_group(g + kT5Threads, qB, sB);
                    }
                }

#if LVC5_WAIT == 2
                deposit_parked();                                          // first window staged: the tables are needed from here on
#endif
                // ---- column windows of kTabCols (one for amplicon / deep shotgun chunks)
                const uint32_t chunk_ord0 = dp.ord_base + chunk0;
                uint32_t* plane = tv.planes[tp.prim_plane];
                uint32_t* first0 = tv.first[0];
                const uint32_t ord_lo = chunk_ord0 + (s_rix[a0] & 255u);      // first read of this window's runs
                const uint32_t pk_smem = sbase + Tile5Smem::pk_off;
                const uint32_t lut_smem = sbase + Tile5Smem::lut_off;
                for (int32_t wc0 = cmin; wc0 < cmax; wc0 += kTabCols) {
                    const int nslab = min(kMaxSlabs, (cmax - wc0 + kSlabCols - 1) / kSlabCols);
                    if (wc0 != cmin) {
                        __syncthreads();                                   // every warp has left the previous column window
                        if (warp == 0) slab_setup(wc0);
                    }
                    __syncthreads();                                       // barrier C: keys staged, task table built
                    T5_STAMP(T5P_BARRIER_C);
                    const uint32_t n_tasks = s_slab_pre[nslab];

                    // ---- tasks: (slab of 32 columns, share of its candidate runs); lane = one run per pass, all 32 columns
                    for (;;) {
                        uint32_t t = 0;
                        if (lane == 0)
                            asm volatile("atom.shared.add.u32 %0, [%1], 1;" : "=r"(t) : "r"(sbase + Tile5Smem::misc_off + 8u) : "memory");
                        t = __shfl_sync(0xFFFFFFFFu, t, 0);
                        if (t >= n_tasks) break;
                        int k = 0;
                        while (k + 1 < nslab && s_slab_pre[k + 1] <= t) ++k;
                        const uint32_t sa = s_slab_a[k], se = sa + s_slab_n[k];
                        const uint32_t ra = sa + (t - s_slab_pre[k]) * s_slab_per[k];
                        const uint32_t rb = min(se, ra + s_slab_per[k]);
                        const int32_t col0 = wc0 + k * kSlabCols;
                        // three bit planes x four key words: 128 counters (32 columns x A,C,G,T), each <= 7
                        uint32_t P0[4] = {0, 0, 0, 0}, P1[4] = {0, 0, 0, 0}, P2[4] = {0, 0, 0, 0};
#pragma unroll 1
                        for (uint32_t r0 = ra; r0 < rb; r0 += 32) {
                            const uint32_t r = r0 + (uint32_t)lane;
                            // a run that misses the slab (or a slot past the end of the share) becomes a unit of length 0,
                            // which the edge masks empty: no other branch
                            uint32_t px = (uint32_t)col0, py = 0;
                            if (r < rb) asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(px), "=r"(py) : "r"(pk_smem + 8u * r));
                            int32_t j = col0 - (int32_t)px, len = (int32_t)(py >> 16);
                            const bool on = j > -32 && j < len;
                            j = on ? j : 0; len = on ? len : 0;
                            const int32_t ka = (int32_t)(py & 0xFFFFu) + j;
                            const uint32_t a = k_smem + (uint32_t)((ka >> 3) << 2);
                            const uint32_t x0 = lds32(a), x1 = lds32(a + 4), x2 = lds32(a + 8), x3 = lds32(a + 12), x4 = lds32(a + 16);
                            const uint32_t sh = (uint32_t)(ka & 7) * 4u;
                            uint32_t kw[4];
                            kw[0] = __funnelshift_r(x0, x1, sh); kw[1] = __funnelshift_r(x1, x2, sh);
                            kw[2] = __funnelshift_r(x2, x3, sh); kw[3] = __funnelshift_r(x3, x4, sh);
                            if (__any_sync(0xFFFFFFFFu, j < 0 || j + 32 > len)) {
                                // some lane's unit overlaps a run edge: keep the keys with 0 <= j + column < len
                                const int32_t lo = j < 0 ? -j : 0, hi = (len - j) < 32 ? (len - j) : 32;
                                uint4 ml, mh;
                                asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(ml.x), "=r"(ml.y), "=r"(ml.z), "=r"(ml.w) : "r"(lut_smem + 16u * (uint32_t)lo));
                                asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(mh.x), "=r"(mh.y), "=r"(mh.z), "=r"(mh.w) : "r"(lut_smem + 16u * (33u + (uint32_t)hi)));
                                kw[0] &= ml.x & mh.x; kw[1] &= ml.y & mh.y; kw[2] &= ml.z & mh.z; kw[3] &= ml.w & mh.w;
                            }
                            // carry-save ripple: +1 into the three planes wherever a key bit is set
#pragma unroll
                            for (int w = 0; w < 4; ++w) {
                                const uint32_t c0 = P0[w] & kw[w];
                                P2[w] = lop3_xor_and(P2[w], P1[w], c0);
                                P1[w] ^= c0;
                                P0[w] ^= kw[w];
                            }
                        }
                        // ---- reduce over the 32 runs of the passes (DESIGN.md 3.1)
                        // level A (lane bit 4): words {0,1} stay with the low half of the warp, words {2,3} go to the high half
                        uint32_t Q[2][4];                                   // [word][plane], 4 planes
                        {
                            const bool hiA = lane & 16;
#pragma unroll
                            for (int w = 0; w < 2; ++w) {
                                uint32_t mine[3], got[3];
                                mine[0] = hiA ? P0[w + 2] : P0[w]; mine[1] = hiA ? P1[w + 2] : P1[w]; mine[2] = hiA ? P2[w + 2] : P2[w];
                                got[0] = __shfl_xor_sync(0xFFFFFFFFu, hiA ? P0[w] : P0[w + 2], 16);
                                got[1] = __shfl_xor_sync(0xFFFFFFFFu, hiA ? P1[w] : P1[w + 2], 16);
                                got[2] = __shfl_xor_sync(0xFFFFFFFFu, hiA ? P2[w] : P2[w + 2], 16);
                                bs_add<3>(mine, got, Q[w]);
                            }
                        }
                        // level B (lane bit 3): one word per lane
                        uint32_t R5[5];
                        {
                            const bool hiB = lane & 8;
                            uint32_t mine[4], got[4];
#pragma unroll
                            for (int p = 0; p < 4; ++p) {
                                mine[p] = hiB ? Q[1][p] : Q[0][p];
                                got[p] = __shfl_xor_sync(0xFFFFFFFFu, hiB ? Q[0][p] : Q[1][p], 8);
                            }
                            bs_add<4>(mine, got, R5);
                        }
                        // levels C, D, E (lane bits 2, 1, 0): the 8 lanes that hold the same word add whole registers
                        // (an all-reduce: counters are independent bit positions, nothing to select or shift)
                        uint32_t R6[6], R7[7], R8[8];
                        {
                            uint32_t got[5];
#pragma unroll
                            for (int p = 0; p < 5; ++p) got[p] = __shfl_xor_sync(0xFFFFFFFFu, R5[p], 4);
                            bs_add<5>(R5, got, R6);
                        }
                        {
                            uint32_t got[6];
#pragma unroll
                            for (int p = 0; p < 6; ++p) got[p] = __shfl_xor_sync(0xFFFFFFFFu, R6[p], 2);
                            bs_add<6>(R6, got, R7);
                        }
                        {
                            uint32_t got[7];
#pragma unroll
                            for (int p = 0; p < 7; ++p) got[p] = __shfl_xor_sync(0xFFFFFFFFu, R7[p], 1);
                            bs_add<7>(R7, got, R8);
                        }
                        // lane L = column L of the slab: its nibble of the word (bits 4*(L&7)..) holds, plane by plane,
                        // the A,C,G,T bits of the four counts (<= 224).  One multiply spreads a nibble to four bytes.
                        uint32_t cnt4 = 0;
                        {
                            const uint32_t s4 = (uint32_t)(lane & 7) * 4u;
#pragma unroll
                            for (int p = 7; p >= 0; --p)
                                cnt4 = cnt4 * 2u + ((((R8[p] >> s4) & 15u) * 0x00204081u) & 0x01010101u);
                        }
                        // ---- flush: one global RED per non-zero (column, allele) of the task; new pairs get their
                        //      exact first-seen ordinal below
                        const int32_t col = col0 + lane;
                        uint32_t fresh = 0;
                        if (cnt4) {
                            // the four first-seen ordinals of the column come with ONE 16-byte load (requested before
                            // the reductions are issued)
                            const int64_t cell = (int64_t)col * 4;
                            uint32_t* prow = plane + cell;
                            const uint32_t* frow = first0 + cell;
                            if (PEER && peer_remote(tv.peer, col)) {       // a column another rank owns: its tables, over NVLink
                                prow = plane_row(tv, tp.prim_plane, col);
                                frow = first_row(tv, 0, col);
                            }
                            const uint4 ff = *reinterpret_cast<const uint4*>(frow);
#pragma unroll
                            for (int c = 0; c < 4; ++c) {
                                const uint32_t f = (cnt4 >> (8 * c)) & 255u;
                                if (f) atomicAdd(prow + c, f);
                            }
                            if ((cnt4 & 0x000000FFu) && ff.x > ord_lo) fresh |= 1u;
                            if ((cnt4 & 0x0000FF00u) && ff.y > ord_lo) fresh |= 2u;
                            if ((cnt4 & 0x00FF0000u) && ff.z > ord_lo) fresh |= 4u;
                            if ((cnt4 & 0xFF000000u) && ff.w > ord_lo) fresh |= 8u;
                        }
                        if (__any_sync(0xFFFFFFFFu, fresh != 0)) {
                            // exact first-seen ordinal for new (column, allele) pairs: scan the slab's candidate runs in
                            // read order (all of them, not only this task's share)
#pragma unroll 1
                            for (int c = 0; c < 4; ++c) {
                                uint32_t todo = __ballot_sync(0xFFFFFFFFu, (fresh >> c) & 1u);
                                while (todo) {
                                    const int src = __ffs(todo) - 1;
                                    todo &= todo - 1;
                                    const int32_t icol = col0 + src;
                                    const uint32_t want = 1u << c;
                                    for (uint32_t q0 = sa; q0 < se; q0 += 32) {
                                        const uint32_t r = q0 + (uint32_t)lane;
                                        bool hit = false;
                                        if (r < se) {
                                            const uint2 pk = s_pk[r];
                                            const int32_t jj = icol - (int32_t)pk.x;
                                            if (jj >= 0 && jj < (int32_t)(pk.y >> 16)) {
                                                const uint32_t kk = (pk.y & 0xFFFFu) + (uint32_t)jj;
                                                const uint32_t key = (lds32(k_smem + ((kk >> 3) << 2)) >> ((kk & 7u) * 4u)) & 15u;
                                                hit = key == want;
                                            }
                                        }
                                        const uint32_t hb = __ballot_sync(0xFFFFFFFFu, hit);
                                        if (hb) {
                                            if (lane == 0)
                                                atomicMin((PEER ? first_row(tv, 0, icol) : first0 + (int64_t)icol * 4) + c,
                                                          chunk_ord0 + (s_rix[q0 + (__ffs(hb) - 1)] & 255u));
                                            break;
                                        }
                                    }
                                }
                            }
                        }
                    }
                }
                if (win + 1 < n_win) __syncthreads();                      // staging buffer is reused by the next window
                a0 = a1;
            }
        }
#if LVC5_WAIT == 2
        deposit_parked();                                                  // (no-op unless no window was staged)
#endif
        // ---- reads the tiled path could not take (many runs, long, exotic base codes): general path, one warp each
        __syncthreads();
        T5_STAMP(T5P_TASKS_END);
        const uint32_t n_def = s_misc[6];
        for (uint32_t d = warp; d < n_def; d += kT5Warps) (PEER ? deposit_read_warp_peer : deposit_read_warp)(b, tv, dp, chunk0 + s_dlist[d], lane);
    }
    T5_STAMP(T5P_EXIT);
}

}  // namespace lvc
