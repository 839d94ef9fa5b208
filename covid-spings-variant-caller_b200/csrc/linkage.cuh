// Variant linkage: how chosen sites co-occur on the same reads (include/lvc.h, lvc_set_linkage_sites / lvc_copy_linkage).
//
// Rule: a read that the deposit walks (read_passes_filter, at least one reference-consuming op, inside [0, G)) has, at a
// registered site (pos, alt), the pileup entry the deposit adds to totalDepth at pos, or none.  The site's state is
//   absent  no entry (outside the aligned span, in a soft clip), or an entry that fails the base-quality rule: the base's
//           quality, or for a deletion / ref-skip entry the quality of the query base at the start of its op (0 past
//           the end of the read), the quality htslib's resolve_cigar2 assigns to it;
//   REF 0   the base is the reference letter;
//   ALT 1   the base is `alt`, or the entry is a deletion / ref-skip and `alt` is '-';
//   OTHER 2 anything else (another nibble code, N included, or a deletion / ref-skip when `alt` is a base).
// Every pair of sites a < b with pos_b - pos_a <= max_span whose two states are present on the read adds 1 to
// count[state_a][state_b].  Only bases above the threshold are ever read, so every batch form counts the same values.
//
// The host guarantees that any window of max_span + 1 positions holds at most 64 sites, so the partners of a site are
// among the 63 sites before it: one thread walks its read's CIGAR and sites together and keeps the states of the last 64
// sites in three 64-bit registers.
#pragma once
#include "lvc_common.cuh"

namespace lvc {

constexpr int kLinkThreads = 256;           // k_count_linkage: one thread per read
constexpr uint32_t kLinkMaxWindow = 64;     // sites inside any window of max_span + 1 positions
constexpr uint8_t kLinkDeletion = 16;       // LinkSite::alt_nib of a '-' site: equal to no nibble code ('=' is 0)

// per registered site, beside its position
struct LinkSite {
    uint32_t off;           // index of the pair (this site, the next site)
    uint8_t ref_nib;        // BAM nibble of the reference letter (1, 2, 4, 8)
    uint8_t alt_nib;        // BAM nibble of the alt base, kLinkDeletion for '-'
    uint8_t back;           // partners before this site: sites a with pos - pos_a <= max_span (<= 63)
    uint8_t pad;
};

struct LinkTable {
    const int32_t* pos;     // [n_sites], strictly ascending
    const LinkSite* site;   // [n_sites]
    uint32_t* counts;       // [n_pairs][3][3]
    uint32_t n_sites;
};

struct LinkCountParams {
    int64_t G;
    int min_bq, min_mq;
};

// One thread per read.  Dead reads leave after their `keep` byte; reads whose span holds no site leave after their
// headers and CIGAR; the payload is read only at sites and at the qualities that decide deletion entries.
__global__ void __launch_bounds__(kLinkThreads) k_count_linkage(const __grid_constant__ BatchView b,
                                                                const __grid_constant__ LinkTable t,
                                                                const __grid_constant__ LinkCountParams cp, uint32_t n) {
    const uint32_t i = blockIdx.x * kLinkThreads + threadIdx.x;
    if (i < n) {
        const uint32_t keep = b.keep[i];
        if ((keep & 1u) && read_passes_filter(b.flag[i], b.mapq[i], keep, cp.min_mq)) {
            const int64_t pos = b.pos[i];
            const uint32_t c0 = b.cigar_off[i], c1 = b.cigar_off[i + 1];
            // first site at or after the read start: a chain of loads independent of the CIGAR's, so the two overlap
            uint32_t s = 0, hi = t.n_sites;
            while (s < hi) {
                const uint32_t mid = (s + hi) >> 1;
                if (t.pos[mid] < pos) s = mid + 1; else hi = mid;
            }
            int64_t sp = s < t.n_sites ? t.pos[s] : INT64_MAX;
            int64_t rlen = 0;
            uint32_t lq = 0;
            for (uint32_t k = c0; k < c1; ++k) {
                const uint32_t c = b.cigar[k], op = c & 15u, len = c >> 4;
                if (op_consumes_ref(op)) rlen += len;
                if (op_consumes_query(op)) lq += len;
            }
            // the deposit's conditions: no reference-consuming op, or outside [0, G) (LVC_ERANGE), deposits nothing
            if (rlen != 0 && pos >= 0 && pos + rlen <= cp.G) {
                if (sp < pos + rlen) {
                    const uint64_t qb = b.seq_off[i];
                    // the last 64 sites, newest in bit 0: present, and the two bits of the state
                    uint64_t pres = 0, st0 = 0, st1 = 0;
                    int64_t r = pos;
                    uint32_t qi = 0;
                    for (uint32_t k = c0; k < c1 && sp < pos + rlen; ++k) {
                        const uint32_t c = b.cigar[k], op = c & 15u, len = c >> 4;
                        if (op_consumes_ref(op)) {
                            const int64_t r_end = r + len;
                            // deletion / ref-skip entries: the quality of the query base at the start of the op
                            const bool del_ok = (op == 2u || op == 3u) && sp < r_end &&
                                                (int)(qi < lq ? batch_qual(b, qb + qi) : 0u) >= cp.min_bq;
                            for (; sp < r_end; sp = ++s < t.n_sites ? t.pos[s] : INT64_MAX) {
                                const LinkSite ls = t.site[s];
                                uint32_t st = 3u;                               // absent
                                if (op_is_match(op)) {
                                    const uint64_t x = qb + qi + (uint32_t)(sp - r);
                                    if ((int)batch_qual(b, x) >= cp.min_bq) {
                                        const uint32_t nib = batch_nibble(b, x);
                                        st = nib == ls.ref_nib ? 0u : nib == ls.alt_nib ? 1u : 2u;
                                    }
                                } else if (del_ok) {
                                    st = ls.alt_nib == kLinkDeletion ? 1u : 2u;
                                }
                                pres <<= 1; st0 <<= 1; st1 <<= 1;
                                if (st == 3u) continue;
                                pres |= 1u; st0 |= st & 1u; st1 |= st >> 1;
                                // partners: ring bits 1..back (2 << 63 wraps to 0, giving bits 1..63)
                                uint64_t cand = pres & ((2ull << ls.back) - 2ull);
                                while (cand) {
                                    const uint32_t j = __ffsll((long long)cand) - 1;
                                    cand &= cand - 1;
                                    const uint32_t sa = (uint32_t)((st0 >> j) & 1u) | (uint32_t)((st1 >> j) & 1u) << 1;
                                    const uint32_t pair = t.site[s - j].off + (j - 1u);
                                    // amplicon reads of a warp share their pairs and mostly their cells: one atomic per
                                    // distinct cell among the lanes here (config 2, 1,000 sites: 87 against 197 us)
                                    const uint32_t cell = pair * 9u + sa * 3u + st;
                                    const uint32_t peers = __match_any_sync(__activemask(), cell);
                                    if ((threadIdx.x & 31u) == (uint32_t)(__ffs(peers) - 1))
                                        atomicAdd(t.counts + cell, (uint32_t)__popc(peers));
                                }
                            }
                            r = r_end;
                        }
                        if (op_consumes_query(op)) qi += len;
                    }
                }
            }
        }
    }
    // launched with programmatic serialization behind the deposit: the next kernel of the stream may only be released
    // once the deposit has completed, so nothing of this grid exits before it
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

}  // namespace lvc
