// Shared device-side definitions for the live-variant-caller kernels (sm_100a).
#pragma once
#include <stdint.h>
#include <cuda_runtime.h>

namespace lvc {

constexpr uint16_t kNoPlane = 0xFFFFu;
constexpr uint32_t kUnsetOrdinal = 0xFFFFFFFFu;
constexpr int kMaxKeys = 1024;          // 4 allele groups x 256 qualities
constexpr uint32_t kFlagFilter = 0x4u | 0x100u | 0x200u | 0x400u;   // UNMAP|SECONDARY|QCFAIL|DUP (SURVEY B1)

// status words written by the deposit kernels
enum { ST_UNMAPPED = 0, ST_RANGE_ERR = 1, ST_WORDS = 8 };

// BAM nibble -> (group<<2 | slot).  A,C,G,T (1,2,4,8) are group 0 slots 0..3; the other 12 codes fill
// groups 1..3 in ascending nibble order.  Packed 4 bits per nibble, nibble 0 in the low digit.
constexpr uint64_t kNibbleToGS = 0xFEDCBA9387625104ull;
__host__ __device__ __forceinline__ uint32_t nibble_gs(uint32_t nib) {
    return (uint32_t)(kNibbleToGS >> (nib * 4)) & 0xFu;
}
// inverse: (group<<2|slot) -> nibble
__host__ __device__ __forceinline__ uint32_t gs_nibble(uint32_t gs) {
    constexpr uint64_t inv = 0xFEDCBA9765308421ull;   // gs 0..15 -> 1,2,4,8, 0,3,5,6, 7,9,10,11, 12..15
    return (uint32_t)(inv >> (gs * 4)) & 0xFu;
}

// Position ownership over NVLink peer memory (lvc_peer_attach): rank r owns the columns [r*per, (r+1)*per) and its tables
// hold the history of those columns only.  A deposit into a column owned by another rank is reduced directly into THAT
// rank's table through its peer-mapped pointer (a RED that travels over NVLink / NVSwitch and is resolved in the owner's
// L2): the exchange step of the read-chunk sharding disappears into the deposit kernel.
constexpr int kMaxPeers = 8;
struct PeerView {
    int32_t n_ranks, rank;
    int64_t per;                              // columns per rank (lvc_position_slice)
    int64_t lo, hi;                           // this rank's columns [lo, hi)
    uint32_t* dels[kMaxPeers];                // [rank] -> that rank's table ([rank] of this rank = its own pointer)
    int32_t* covdiff[kMaxPeers];
    uint32_t* first[kMaxPeers][4];
    uint32_t* const* planes[kMaxPeers];       // [rank] -> device array indexed by THIS rank's plane id
};

// Persistent per-handle tables as the kernels see them.
struct TableView {
    int64_t G;                    // reference length
    uint32_t* const* planes;      // [n_planes] -> uint32 [G][4]
    const uint16_t* lut;          // [1024] key -> plane id or kNoPlane
    uint32_t* dels;               // [G]
    int32_t* covdiff;             // [G+1]
    uint32_t* first[4];           // per group [G][4] (nullptr if the group has no plane yet)
    uint32_t* newkeys;            // [32] bitmap of keys seen without a plane
    uint32_t* status;             // [ST_WORDS]
    const uint32_t* seen;         // hint, may be null: one nibble per column (8 columns per word), bit = "this A/C/G/T
                                  // allele had a first-seen ordinal after an EARLIER batch" (written by k_genotype);
                                  // readable from column -16 to G + 31
    const PeerView* peer;         // null unless lvc_peer_attach was called (device memory)
};

// One batch of reads, device pointers (mirrors lvc_batch in include/lvc.h).
struct BatchView {
    uint32_t n_reads;
    const int32_t* pos;
    const uint16_t* flag;
    const uint8_t* mapq;
    const uint8_t* keep;
    const uint32_t* cigar_off;
    const uint32_t* cigar;
    const uint64_t* seq_off;
    const uint8_t* seq4;
    const uint8_t* qual;
    uint32_t qbits = 0;           // 2: `qual` holds 2-bit codes (four bases per byte, low bits first), phred = byte `code` of qdict
    uint32_t qdict = 0;           // lvc_batch::qual_dict, code 0 in the low byte
    uint32_t sbits = 0;           // 2: `seq4` holds 2-bit base codes (A,C,G,T = 0..3; four bases per byte, low bits first)
    uint32_t hdr_lazy = 0;        // the per-read arrays other than `keep` sit in host memory (read in place over PCIe): a
                                  // chunk asks for them only after its `keep` bytes say that some read is admitted
};

// quality of the base with quality index x (= seq_off[read] + query index), either batch form
__device__ __forceinline__ uint32_t batch_qual(const BatchView& b, uint64_t x) {
    if (b.qbits == 2u) {
        const uint32_t c = ((uint32_t)b.qual[x >> 2] >> (2u * ((uint32_t)x & 3u))) & 3u;
        return (b.qdict >> (8u * c)) & 255u;
    }
    return b.qual[x];
}

// BAM nibble code of the base with quality index x (= seq_off[read] + query index; seq_off is even), either batch form
__device__ __forceinline__ uint32_t batch_nibble(const BatchView& b, uint64_t x) {
    if (b.sbits == 2u) return 1u << (((uint32_t)b.seq4[x >> 2] >> (2u * ((uint32_t)x & 3u))) & 3u);
    const uint32_t byte = b.seq4[x >> 1];
    return (x & 1u) ? (byte & 15u) : (byte >> 4);
}

struct DepositParams {
    int min_bq;
    int min_mq;
    uint32_t ord_base;            // ordinal of read 0 of this batch
    int replay;                   // 0: normal pass; 1: deposit only keys in `replay_keys`, no dels/cov
    const uint32_t* replay_keys;  // [32] bitmap (device) when replay
};

// ---- table cells by column, routed to the owning rank when peer tables are attached (the local slice takes the first branch)
__device__ __forceinline__ int peer_owner(const PeerView* pv, int64_t col) {
    const uint32_t r = (uint32_t)col / (uint32_t)pv->per;
    return (int)(r < (uint32_t)pv->n_ranks ? r : (uint32_t)pv->n_ranks - 1u);
}
__device__ __forceinline__ bool peer_remote(const PeerView* pv, int64_t col) { return pv && (col < pv->lo || col >= pv->hi); }
// covdiff has G + 1 entries; entry i belongs to the owner of column min(i, G - 1)
__device__ __forceinline__ int32_t* covdiff_cell(const TableView& tv, int64_t i) {
    const int64_t c = i < tv.G ? i : tv.G - 1;
    if (peer_remote(tv.peer, c)) return tv.peer->covdiff[peer_owner(tv.peer, c)] + i;
    return tv.covdiff + i;
}
__device__ __forceinline__ uint32_t* dels_cell(const TableView& tv, int64_t col) {
    if (peer_remote(tv.peer, col)) return tv.peer->dels[peer_owner(tv.peer, col)] + col;
    return tv.dels + col;
}
// row (4 cells) of plane `pl` / of the first-seen table of `group` at column col
__device__ __forceinline__ uint32_t* plane_row(const TableView& tv, uint32_t pl, int64_t col) {
    if (peer_remote(tv.peer, col)) return tv.peer->planes[peer_owner(tv.peer, col)][pl] + col * 4;
    return tv.planes[pl] + col * 4;
}
__device__ __forceinline__ uint32_t* first_row(const TableView& tv, uint32_t group, int64_t col) {
    if (peer_remote(tv.peer, col)) return tv.peer->first[peer_owner(tv.peer, col)][group] + col * 4;
    return tv.first[group] + col * 4;
}

__host__ __device__ __forceinline__ bool read_passes_filter(uint32_t flag, uint32_t mapq, uint32_t keep, int min_mq) {
    // pysam stepper "samtools": flag filter, mapq, ignore_orphans (SURVEY B2) + host admission bit
    if (!(keep & 1u)) return false;
    if (flag & kFlagFilter) return false;
    if ((int)mapq < min_mq) return false;
    if ((flag & 0x1u) && !(flag & 0x2u)) return false;
    return true;
}

__device__ __forceinline__ bool op_consumes_ref(uint32_t op) {   // M D N = X
    return op == 0 || op == 2 || op == 3 || op == 7 || op == 8;
}
__device__ __forceinline__ bool op_consumes_query(uint32_t op) { // M I S = X
    return op == 0 || op == 1 || op == 4 || op == 7 || op == 8;
}
__device__ __forceinline__ bool op_is_match(uint32_t op) { return op == 0 || op == 7 || op == 8; }

}  // namespace lvc
