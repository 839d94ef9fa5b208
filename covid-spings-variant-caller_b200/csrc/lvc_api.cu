// liblvc_b200.so -- C-ABI (include/lvc.h) over the sm_100a kernels.  No torch types, no CPU fallback.
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <mutex>
#include <string>
#include <vector>

#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>          // header-only NVTX 3: ranges cost nothing unless a tool injects itself

#include "../../include/lvc.h"
#include "lvc_common.cuh"
#include "deposit_general.cuh"
#include "deposit_tile.cuh"
#include "deposit_tile4.cuh"
#include "deposit_tile5.cuh"
#include "deposit_ont.cuh"
#include "genotype.cuh"
#include "consensus.cuh"
#include "insertions.cuh"
#include "deposit_select.hpp"
#include "overlap.hpp"
#include "qcode.hpp"

// NVTX range around the host side of an entry point (SURVEY section 5: ingest / push / genotype / exchange show up
// as named ranges in Nsight Systems).
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
};

using namespace lvc;

static thread_local std::string g_create_error;
// every per-position table is allocated with this many extra rows, so that an in-place reduce-scatter onto position
// slices of ceil((G+1)/n) rows (lvc_reduce_tables) stays inside the allocation for any n < kRowSlack - 1
constexpr int kRowSlack = 258;

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
};

struct lvc_handle {
    int device = 0;
    int64_t G = 0;
    int min_bq = 0, min_mq = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::string err;
    int impl = 0;
    int sm_count = 148;
    uint64_t launches = 0;
    bool zero_copy_ok = true;                // read page-locked caller payload in place (LVC_ZERO_COPY=0 disables)
    bool zc_headers = false;                 // also read the per-read arrays (all but `keep`) in place (LVC_ZC_HEADERS=1)
    uint64_t h2d_payload_bytes = 0;          // payload bytes actually copied by lvc_push_batch (cumulative)
    uint64_t ordinal = 0;
    int qprim = 255;                         // primary quality of the current batch (tiled kernel)
    uint8_t* h_sample = nullptr;             // pinned quality sample for device-resident batches

    // persistent tables
    uint8_t* d_ref = nullptr;
    std::vector<uint32_t*> planes;           // device pointers, index = plane id
    std::vector<uint16_t> plane_key;         // plane id -> key
    uint16_t lut[kMaxKeys];
    uint32_t** d_planes = nullptr;           // [kMaxKeys]
    uint16_t* d_lut = nullptr;               // [kMaxKeys]
    uint32_t* d_dels = nullptr;
    int32_t* d_covdiff = nullptr;
    PeerView* d_peer = nullptr;              // lvc_peer_attach: tables of the other ranks (peer.hpp)
    uint32_t** d_peer_planes = nullptr;
    std::vector<void*> peer_opened;
    int peer_ranks = 0;
    size_t peer_planes_at_attach = 0;
    uint32_t* d_seen = nullptr;              // first-seen hint nibbles (TableView::seen), 2 words of padding in front
    size_t seen_words = 0;
    bool seen_off = false;                   // someone took a raw pointer to a first-seen table: no hints any more
    uint32_t* d_first[4] = {nullptr, nullptr, nullptr, nullptr};
    uint32_t** d_first_arr = nullptr;        // [4] device copy of d_first
    uint32_t* d_newkeys = nullptr;           // [32]
    uint32_t* d_replay = nullptr;            // [32]
    uint32_t* d_status = nullptr;            // [ST_WORDS]
    uint32_t* h_status = nullptr;            // pinned [ST_WORDS + 32]
    uint8_t* d_keymap = nullptr;             // [kMaxKeys] plane presence map (lvc_reduce_tables)
    uint64_t last_exchange_bytes = 0;        // bytes this rank put into the last lvc_reduce_tables

    // batch staging (device copies of host batches)
    DevBuf b_pos, b_flag, b_mapq, b_keep, b_coff, b_cig, b_soff, b_seq, b_qual;

    // genotype
    DevBuf g_order_ptrs, g_order_keys, g_cand, g_pconst;
    std::vector<PlaneConst> pconst_host;     // staging of the per-plane constants (kept alive for the async copy)
    double* d_elut = nullptr;                // [512] e, 1-e
    uint32_t* d_out_depth = nullptr;
    uint32_t* d_out_ad = nullptr;
    double* d_out_lik = nullptr;
    uint32_t* d_cand_count = nullptr;           // [2]: the genotype kernel counts in one and clears the other for the next call
    int cand_slot = 0;
    uint32_t cand_cap = 0;
    uint32_t last_cand_count = 0;
    int64_t geno_p0 = 0, geno_p1 = -1;       // genotype position range (p1 < 0: whole contig)
    bool geno_pending = false;               // an async genotype launch whose count has not been read yet
    size_t geno_planes_uploaded = (size_t)-1; // number of planes the device-side ordered plane list reflects
    double lut_host[512];                    // last uploaded e / 1-e tables
    bool lut_valid = false;

    // consensus (lvc_consensus): its own ordered plane list, output letters and counters
    DevBuf c_order_ptrs, c_seq, c_stats;
    size_t cons_planes_uploaded = (size_t)-1;
    int cons_grp_begin[5] = {0, 0, 0, 0, 0};

    // insertion counts (lvc_enable_insertions): ins.keys == nullptr while counting is off
    InsTable ins = {nullptr, nullptr, nullptr, 0};
    bool tables_touched = false;             // a push, import or reduction since lvc_create / lvc_reset
    bool ins_uncovered = false;              // an import or reduction since lvc_reset: counts the insertion table lacks
    DevBuf i_list, i_scratch;

    // optional per-kernel timing (CUDA events on the launching stream)
    bool timing = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev[5];   // 0 tiled deposit, 1 general deposit, 2 genotype, 3 consensus,
                                                              // 4 insertion counts
    std::vector<cudaEvent_t> ev_pool;
};

static cudaEvent_t get_event(lvc_handle* h) {
    if (!h->ev_pool.empty()) { cudaEvent_t e = h->ev_pool.back(); h->ev_pool.pop_back(); return e; }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}
struct KernelTimer {
    lvc_handle* h; int which; cudaEvent_t a = nullptr, b = nullptr;
    KernelTimer(lvc_handle* h_, int w) : h(h_), which(w) {
        if (h->timing) { a = get_event(h); b = get_event(h); cudaEventRecord(a, h->stream); }
    }
    ~KernelTimer() {
        if (h->timing) { cudaEventRecord(b, h->stream); h->ev[which].push_back({a, b}); }
    }
};

static int fail(lvc_handle* h, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (h) h->err = buf; else g_create_error = buf;
    return code;
}

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(h, LVC_ECUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

static int ensure(lvc_handle* h, DevBuf& b, size_t bytes) {
    if (bytes <= b.cap && b.p) return LVC_OK;
    size_t want = std::max<size_t>(bytes + bytes / 8, 256);
    if (b.p) CU(cudaFree(b.p));
    b.p = nullptr; b.cap = 0;
    CU(cudaMalloc(&b.p, want));
    b.cap = want;
    return LVC_OK;
}

static TableView table_view(lvc_handle* h) {
    TableView tv;
    tv.G = h->G;
    tv.planes = h->d_planes;
    tv.lut = h->d_lut;
    tv.dels = h->d_dels;
    tv.covdiff = h->d_covdiff;
    for (int g = 0; g < 4; ++g) tv.first[g] = h->d_first[g];
    tv.newkeys = h->d_newkeys;
    tv.status = h->d_status;
    tv.seen = (h->d_seen && !h->seen_off) ? h->d_seen + 2 : nullptr;
    tv.peer = h->peer_ranks > 1 ? h->d_peer : nullptr;
    return tv;
}

// One kernel launch on the handle's stream, counted in lvc_launch_count.  `pdl`: programmatic stream serialization -- the
// kernel may become resident while the previous kernel of the stream drains, so it must execute griddepcontrol.wait
// before it reads or writes anything that kernel touches.
static cudaError_t launch_kernel(lvc_handle* h, const void* kern, dim3 grid, dim3 block, size_t smem, bool pdl, void** args) {
    cudaLaunchAttribute at;
    at.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at.val.programmaticStreamSerializationAllowed = 1;
    const cudaLaunchConfig_t cfg = {grid, block, smem, h->stream, &at, pdl ? 1u : 0u};
    const cudaError_t e = cudaLaunchKernelExC(&cfg, kern, args);
    if (e == cudaSuccess) h->launches++;
    return e;
}
// the same with the arguments converted to the kernel's parameter types
template <typename... P, typename... A>
static cudaError_t launch_kernel(lvc_handle* h, void (*kern)(P...), dim3 grid, dim3 block, size_t smem, bool pdl, A&&... args) {
    return [&](P... p) {
        void* pargs[] = {&p...};
        return launch_kernel(h, (const void*)kern, grid, block, smem, pdl, pargs);
    }(std::forward<A>(args)...);
}

// Every instantiation of the tiled deposit kernels: by GE_ALL (threshold <= 0), and for generation 5 by PEER and by the
// batch's payload form (phred bytes, quality codes, quality and base codes).  launch_deposit picks from these tables and
// lvc_create raises the dynamic shared memory limit of every entry.
using TileKernel = void (*)(BatchView, TableView, DepositParams, TileParams);
static const TileKernel kTile3[2] = {k_deposit_tile<false>, k_deposit_tile<true>};
static const TileKernel kTile4[2] = {k_deposit_tile4<false>, k_deposit_tile4<true>};
static const TileKernel kTile5[2][2][3] = {
    {{k_deposit_tile5<false, false>, k_deposit_tile5<false, false, true>, k_deposit_tile5<false, false, true, true>},
     {k_deposit_tile5<false, true>, k_deposit_tile5<false, true, true>, k_deposit_tile5<false, true, true, true>}},
    {{k_deposit_tile5<true, false>, k_deposit_tile5<true, false, true>, k_deposit_tile5<true, false, true, true>},
     {k_deposit_tile5<true, true>, k_deposit_tile5<true, true, true>, k_deposit_tile5<true, true, true, true>}}};

// allocate the first-seen table of allele group g if it has none yet (all cells unset); uploads its pointer
static int ensure_first_table(lvc_handle* h, int g) {
    if (h->d_first[g]) return LVC_OK;
    const size_t bytes = ((size_t)h->G + kRowSlack) * 4 * sizeof(uint32_t);
    CU(cudaMalloc(&h->d_first[g], bytes));
    CU(cudaMemsetAsync(h->d_first[g], 0xFF, bytes, h->stream));
    CU(cudaMemcpyAsync(h->d_first_arr + g, &h->d_first[g], sizeof(uint32_t*), cudaMemcpyHostToDevice, h->stream));
    return LVC_OK;
}

// allocate a plane for `key` (and the group's first-seen table); uploads pointer + lut entry
static int add_plane(lvc_handle* h, uint16_t key) {
    if (key >= kMaxKeys) return fail(h, LVC_EINVAL, "plane key %u out of range", key);
    if (h->lut[key] != kNoPlane) return LVC_OK;
    int rc = ensure_first_table(h, key >> 8);
    if (rc) return rc;
    const size_t bytes = ((size_t)h->G + kRowSlack) * 4 * sizeof(uint32_t);
    uint32_t* p = nullptr;
    CU(cudaMalloc(&p, bytes));
    CU(cudaMemsetAsync(p, 0, bytes, h->stream));
    const uint16_t id = (uint16_t)h->planes.size();
    h->planes.push_back(p);
    h->plane_key.push_back(key);
    h->lut[key] = id;
    CU(cudaMemcpyAsync(h->d_planes + id, &h->planes[id], sizeof(uint32_t*), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_lut + key, &h->lut[key], sizeof(uint16_t), cudaMemcpyHostToDevice, h->stream));
    // pageable sources: the runtime stages them before returning, so the host vectors may move later
    return LVC_OK;
}

extern "C" {

int lvc_version(void) { return 1; }

const char* lvc_last_error(const lvc_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int lvc_create(lvc_handle** out, int device, int64_t ref_len, const uint8_t* ref_bytes, int min_base_quality,
               int min_mapping_quality, void* stream) {
    lvc_handle* h = nullptr;
    if (!out || ref_len <= 0 || !ref_bytes) return fail(nullptr, LVC_EINVAL, "lvc_create: bad arguments");
    if (min_base_quality < 0) min_base_quality = 0;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(nullptr, LVC_ENODEVICE, "lvc_create: no CUDA device visible; this library has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(nullptr, LVC_EINVAL, "lvc_create: device %d of %d", device, ndev);
    h = new lvc_handle();
    h->device = device;
    h->G = ref_len;
    h->min_bq = min_base_quality;
    h->min_mq = min_mapping_quality;
    for (int k = 0; k < kMaxKeys; ++k) h->lut[k] = kNoPlane;
    if (const char* zc = getenv("LVC_ZERO_COPY")) h->zero_copy_ok = atoi(zc) != 0;
    if (const char* zh = getenv("LVC_ZC_HEADERS")) h->zc_headers = atoi(zh) != 0;
    auto body = [&]() -> int {
        CU(cudaSetDevice(device));
        cudaDeviceProp prop;
        CU(cudaGetDeviceProperties(&prop, device));
        h->sm_count = prop.multiProcessorCount;
        if (stream) { h->stream = (cudaStream_t)stream; h->own_stream = false; }
        else { CU(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)); h->own_stream = true; }
        const size_t G = (size_t)ref_len;
        CU(cudaMalloc(&h->d_ref, G));
        CU(cudaMemcpyAsync(h->d_ref, ref_bytes, G, cudaMemcpyHostToDevice, h->stream));
        CU(cudaMalloc(&h->d_planes, kMaxKeys * sizeof(uint32_t*)));
        CU(cudaMemsetAsync(h->d_planes, 0, kMaxKeys * sizeof(uint32_t*), h->stream));
        CU(cudaMalloc(&h->d_lut, kMaxKeys * sizeof(uint16_t)));
        CU(cudaMemsetAsync(h->d_lut, 0xFF, kMaxKeys * sizeof(uint16_t), h->stream));
        CU(cudaMalloc(&h->d_dels, (G + kRowSlack) * sizeof(uint32_t)));
        CU(cudaMemsetAsync(h->d_dels, 0, (G + kRowSlack) * sizeof(uint32_t), h->stream));
        CU(cudaMalloc(&h->d_covdiff, (G + kRowSlack) * sizeof(int32_t)));
        CU(cudaMemsetAsync(h->d_covdiff, 0, (G + kRowSlack) * sizeof(int32_t), h->stream));
        h->seen_words = (G + 7) / 8 + 8;
        CU(cudaMalloc(&h->d_seen, h->seen_words * sizeof(uint32_t)));
        CU(cudaMemsetAsync(h->d_seen, 0, h->seen_words * sizeof(uint32_t), h->stream));
        CU(cudaMalloc(&h->d_first_arr, 4 * sizeof(uint32_t*)));
        CU(cudaMemsetAsync(h->d_first_arr, 0, 4 * sizeof(uint32_t*), h->stream));
        CU(cudaMalloc(&h->d_newkeys, 32 * sizeof(uint32_t)));
        CU(cudaMemsetAsync(h->d_newkeys, 0, 32 * sizeof(uint32_t), h->stream));
        CU(cudaMalloc(&h->d_replay, 32 * sizeof(uint32_t)));
        CU(cudaMemsetAsync(h->d_replay, 0, 32 * sizeof(uint32_t), h->stream));
        CU(cudaMalloc(&h->d_status, ST_WORDS * sizeof(uint32_t)));
        CU(cudaMemsetAsync(h->d_status, 0, ST_WORDS * sizeof(uint32_t), h->stream));
        CU(cudaHostAlloc(&h->h_status, (ST_WORDS + 32) * sizeof(uint32_t), cudaHostAllocDefault));
        CU(cudaMalloc(&h->d_elut, 512 * sizeof(double)));
        CU(cudaMalloc(&h->d_out_depth, G * sizeof(uint32_t)));
        CU(cudaMalloc(&h->d_out_ad, G * 4 * sizeof(uint32_t)));
        CU(cudaMalloc(&h->d_out_lik, G * 4 * sizeof(double)));
        // positions outside a restricted genotype range are never written: they read back as zero, not as garbage
        CU(cudaMemsetAsync(h->d_out_depth, 0, G * sizeof(uint32_t), h->stream));
        CU(cudaMemsetAsync(h->d_out_ad, 0, G * 4 * sizeof(uint32_t), h->stream));
        CU(cudaMemsetAsync(h->d_out_lik, 0, G * 4 * sizeof(double), h->stream));
        CU(cudaMalloc(&h->d_cand_count, 2 * sizeof(uint32_t)));
        CU(cudaMemsetAsync(h->d_cand_count, 0, 2 * sizeof(uint32_t), h->stream));
        for (TileKernel k : kTile3) CU(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTileSmemBytes));
        for (TileKernel k : kTile4) CU(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTile4SmemBytes));
        for (auto& by_peer : kTile5) for (auto& by_form : by_peer) for (TileKernel k : by_form)
            CU(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTile5SmemBytes));
        CU(cudaStreamSynchronize(h->stream));
        return LVC_OK;
    };
    int rc = body();
    if (rc != LVC_OK) {
        g_create_error = h->err;
        lvc_destroy(h);
        return rc;
    }
    *out = h;
    return LVC_OK;
}

void lvc_destroy(lvc_handle* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    for (auto p : h->planes) cudaFree(p);
    for (int g = 0; g < 4; ++g) cudaFree(h->d_first[g]);
    cudaFree(h->d_ref); cudaFree(h->d_planes); cudaFree(h->d_lut); cudaFree(h->d_dels); for (void* q : h->peer_opened) cudaIpcCloseMemHandle(q);
    cudaFree(h->d_peer); cudaFree(h->d_peer_planes);
    cudaFree(h->d_covdiff); cudaFree(h->d_seen);
    cudaFree(h->d_first_arr); cudaFree(h->d_newkeys); cudaFree(h->d_replay); cudaFree(h->d_status); cudaFree(h->d_keymap);
    if (h->h_status) cudaFreeHost(h->h_status);
    if (h->h_sample) cudaFreeHost(h->h_sample);
    for (int w = 0; w < 5; ++w) for (auto& pr : h->ev[w]) { cudaEventDestroy(pr.first); cudaEventDestroy(pr.second); }
    for (auto e : h->ev_pool) cudaEventDestroy(e);
    cudaFree(h->d_elut); cudaFree(h->d_out_depth); cudaFree(h->d_out_ad); cudaFree(h->d_out_lik);
    cudaFree(h->d_cand_count);
    cudaFree(h->ins.keys); cudaFree(h->ins.counts); cudaFree(h->ins.dropped);
    for (DevBuf* b : {&h->b_pos, &h->b_flag, &h->b_mapq, &h->b_keep, &h->b_coff, &h->b_cig, &h->b_soff, &h->b_seq,
                      &h->b_qual, &h->g_order_ptrs, &h->g_order_keys, &h->g_cand, &h->g_pconst, &h->c_order_ptrs,
                      &h->c_seq, &h->c_stats, &h->i_list, &h->i_scratch})
        cudaFree(b->p);
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

int lvc_set_stream(lvc_handle* h, void* stream) {
    if (!h) return LVC_EINVAL;
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    if (h->own_stream) { cudaStreamDestroy(h->stream); h->own_stream = false; }
    if (stream) h->stream = (cudaStream_t)stream;
    else { CU(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)); h->own_stream = true; }
    return LVC_OK;
}

int lvc_sync(lvc_handle* h) {
    if (!h) return LVC_EINVAL;
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    return LVC_OK;
}

int lvc_set_impl(lvc_handle* h, int impl) {
    if (!h || impl < 0 || impl > 6) return LVC_EINVAL;
    h->impl = impl;
    return LVC_OK;
}

int lvc_reset(lvc_handle* h) {
    if (!h) return LVC_EINVAL;
    CU(cudaSetDevice(h->device));
    const size_t G = (size_t)h->G;
    for (auto p : h->planes) CU(cudaMemsetAsync(p, 0, G * 4 * sizeof(uint32_t), h->stream));
    for (int g = 0; g < 4; ++g)
        if (h->d_first[g]) CU(cudaMemsetAsync(h->d_first[g], 0xFF, G * 4 * sizeof(uint32_t), h->stream));
    CU(cudaMemsetAsync(h->d_dels, 0, G * sizeof(uint32_t), h->stream));
    CU(cudaMemsetAsync(h->d_covdiff, 0, (G + 1) * sizeof(int32_t), h->stream));
    CU(cudaMemsetAsync(h->d_seen, 0, h->seen_words * sizeof(uint32_t), h->stream));
    CU(cudaMemsetAsync(h->d_out_depth, 0, G * sizeof(uint32_t), h->stream));
    CU(cudaMemsetAsync(h->d_out_ad, 0, G * 4 * sizeof(uint32_t), h->stream));
    CU(cudaMemsetAsync(h->d_out_lik, 0, G * 4 * sizeof(double), h->stream));
    if (h->ins.keys) {
        const size_t slots = (size_t)h->ins.mask + 1;
        CU(cudaMemsetAsync(h->ins.keys, 0, slots * sizeof(ulonglong2), h->stream));
        CU(cudaMemsetAsync(h->ins.counts, 0, slots * sizeof(uint32_t), h->stream));
        CU(cudaMemsetAsync(h->ins.dropped, 0, sizeof(uint32_t), h->stream));
    }
    h->tables_touched = false;
    h->ins_uncovered = false;
    h->ordinal = 0;
    CU(cudaStreamSynchronize(h->stream));
    return LVC_OK;
}

void* lvc_host_alloc(uint64_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}
void lvc_host_free(void* p) { if (p) cudaFreeHost(p); }

// ------------------------------------------------------------------------------------------------
// host-side admission: SURVEY B2 (read filter) + B4 (htslib bam_plp_push maxcnt rule)
// ------------------------------------------------------------------------------------------------
int lvc_admit(uint32_t n, const int32_t* pos, const uint16_t* flag, const uint8_t* mapq, const uint32_t* cigar_off,
              const uint32_t* cigar, int min_mq, int max_depth, uint8_t* keep) {
    if (n && (!pos || !flag || !mapq || !cigar_off || !cigar || !keep)) return LVC_EINVAL;
    auto no_name = [](uint32_t) { return lvc_overlap::NameKey{nullptr, 0}; };
    return lvc_overlap::admit_core(n, pos, flag, mapq, cigar_off, cigar, nullptr, nullptr, nullptr, no_name, nullptr, nullptr,
                                   nullptr, min_mq, max_depth, LVC_OVERLAP_OFF, keep, nullptr, nullptr);
}

int lvc_admit_overlaps(uint32_t n, const int32_t* pos, const uint16_t* flag, const uint8_t* mapq, const uint32_t* cigar_off,
                       const uint32_t* cigar, const uint64_t* seq_off, const uint8_t* seq4, uint8_t* qual,
                       const uint32_t* name_off, const char* names, const int32_t* mate_pos, const int8_t* mate_ref,
                       const int32_t* tlen, int min_mq, int max_depth, int overlap_model, uint8_t* keep, uint64_t* n_pairs,
                       uint64_t* n_bases) {
    if (n && (!pos || !flag || !mapq || !cigar_off || !cigar || !keep)) return LVC_EINVAL;
    if (overlap_model < LVC_OVERLAP_OFF || overlap_model > LVC_OVERLAP_HTSLIB_1_13) return LVC_EINVAL;
    if (overlap_model != LVC_OVERLAP_OFF && n && (!seq_off || !seq4 || !qual || !name_off || !names)) return LVC_EINVAL;
    auto name = [&](uint32_t i) { return lvc_overlap::NameKey{names + name_off[i], name_off[i + 1] - name_off[i]}; };
    return lvc_overlap::admit_core(n, pos, flag, mapq, cigar_off, cigar, seq_off, seq4, qual, name, mate_pos, mate_ref, tlen,
                                   min_mq, max_depth, overlap_model, keep, n_pairs, n_bases);
}

int lvc_pack_quality_codes(const uint8_t* qual, uint64_t n_qual_bytes, uint32_t n_reads, const uint8_t* keep,
                           const uint64_t* seq_off, const uint32_t* cigar_off, const uint32_t* cigar, int n_threads,
                           uint8_t dict_out[4], uint8_t* codes_out) {
    if ((n_qual_bytes && !qual) || !dict_out || !codes_out) return LVC_EINVAL;
    if (n_threads <= 0) n_threads = (int)std::max(1u, std::thread::hardware_concurrency());
    return lvc::pack_quality_codes(qual, n_qual_bytes, n_reads, keep, seq_off, cigar_off, cigar, n_threads, dict_out, codes_out);
}

int lvc_pack_base_codes(const uint8_t* seq4, const uint8_t* qual, uint64_t n_qual_bytes, uint32_t n_reads, const uint8_t* keep,
                        const uint64_t* seq_off, const uint32_t* cigar_off, const uint32_t* cigar, int min_base_quality,
                        int n_threads, uint8_t* codes_out) {
    if (!seq4 || !qual || !keep || !seq_off || !cigar_off || !cigar || !codes_out) return LVC_EINVAL;
    if (n_threads <= 0) n_threads = (int)std::max(1u, std::thread::hardware_concurrency());
    return lvc::pack_base_codes(seq4, qual, n_qual_bytes, n_reads, keep, seq_off, cigar_off, cigar, min_base_quality, n_threads,
                                codes_out);
}

// ------------------------------------------------------------------------------------------------
// deposit
// ------------------------------------------------------------------------------------------------
static int launch_deposit(lvc_handle* h, const BatchView& bv, int replay, uint64_t n_cigar_ops, uint64_t n_qual) {
    TableView tv = table_view(h);
    DepositParams dp;
    dp.min_bq = h->min_bq;
    dp.min_mq = h->min_mq;
    dp.ord_base = (uint32_t)h->ordinal;
    dp.replay = replay;
    dp.replay_keys = h->d_replay;
    const uint32_t n = bv.n_reads;
    if (n == 0) return LVC_OK;
    // quality-code batches: the code of the primary quality (4: none) and the other codes that pass the threshold
    const bool qc = bv.qbits == 2u;
    uint32_t qc_pcode = 4, qc_cold = 0;
    for (uint32_t c = 0; c < 4 && qc; ++c) {
        const int v = (int)((bv.qdict >> (8 * c)) & 255u);
        if (v == h->qprim && qc_pcode == 4) qc_pcode = c;
        else if (v >= h->min_bq) qc_cold |= 1u << c;
    }
    DepositInputs in;
    in.impl = h->impl; in.n_reads = n; in.n_cigar_ops = n_cigar_ops; in.replay = replay != 0; in.small_contig = h->G < (1ll << 30);
    in.peer = h->peer_ranks > 1; in.planes_changed = h->planes.size() != h->peer_planes_at_attach;
    // the tiled kernels' byte arithmetic assumes a primary quality and a threshold below 128
    in.tile_ok = h->qprim < 128 && h->min_bq <= 128 && h->lut[h->qprim] != kNoPlane;
    in.qc = qc; in.qc_prim_coded = qc_pcode < 4; in.base_codes = bv.sbits == 2u;
    const DepositChoice choice = select_deposit(in);
    if (choice.error == DepositError::planes_after_attach)
        return fail(h, LVC_EINVAL, "a plane was added after lvc_peer_attach: export and attach again");
    if (choice.error == DepositError::qc_impl)
        return fail(h, LVC_EINVAL, "quality-code batches run on impl 0, 1 or 5 (selected: %d)", h->impl);
    TileParams tp = make_tile_params(n, h->sm_count);
    tp.qprim = (uint32_t)h->qprim; tp.prim_plane = h->lut[h->qprim]; tp.qc_pcode = qc_pcode & 3u; tp.qc_cold = qc_cold;
    uint32_t rpc = 0;                           // k_deposit_ont: reads per CTA
    void* last_arg = (void*)&n;                 // the tiled kernels take TileParams where the others take n
    const bool peer = in.peer, ge_all = h->min_bq <= 0;
    // programmatic stream serialization (pdl): the warp, ONT and generation-4/5 tiled kernels read their chunk headers or
    // walk their CIGARs while the previous kernel of the stream drains, and wait for it before their first table access.
    // The general and generation-3 kernels never wait: they start after the previous kernel has finished.
    const void* kern = nullptr;
    dim3 grid, block;
    size_t smem = 0;
    bool pdl = true;
    int timer = 1;                              // KernelTimer slot: 0 tiled, 1 general / warp / ONT
    switch (choice.kernel) {
    case DepositKernel::general:
        kern = (const void*)(peer ? k_deposit_general<true> : k_deposit_general<false>);
        grid = dim3((n + 127) / 128); block = dim3(128); pdl = false;
        break;
    case DepositKernel::warp: {
        const unsigned wpb = kWarpKernelThreads / 32;
        kern = (const void*)(peer ? k_deposit_warp<true> : k_deposit_warp<false>);
        grid = dim3((n + wpb - 1) / wpb); block = dim3(kWarpKernelThreads);
        break;
    }
    case DepositKernel::ont: {
        // reads per CTA: as many as keep the CTA's unit list (16 query bases per unit) about three quarters full
        const uint64_t avg_q = std::max<uint64_t>(n_qual / n, 1);
        rpc = (uint32_t)std::min<uint64_t>(kOntMaxReads, std::max<uint64_t>(1, (uint64_t)kOntMaxUnits * 12 / avg_q));
        kern = (const void*)k_deposit_ont;
        grid = dim3((n + rpc - 1) / rpc); block = dim3(kOntThreads);
        break;
    }
    case DepositKernel::tile3:
        kern = (const void*)kTile3[ge_all];
        grid = dim3(tp.grid); block = dim3(kTileThreads); smem = kTileSmemBytes; pdl = false; timer = 0; last_arg = &tp;
        break;
    case DepositKernel::tile4:
        kern = (const void*)kTile4[ge_all];
        grid = dim3(tp.grid); block = dim3(kTileThreads); smem = kTile4SmemBytes; timer = 0; last_arg = &tp;
        break;
    case DepositKernel::tile5:
        kern = (const void*)kTile5[ge_all][peer][choice.t5_form];
        grid = dim3((n + kT5Reads - 1) / kT5Reads); block = dim3(kT5Threads); smem = kTile5SmemBytes; timer = 0; last_arg = &tp;
        break;
    }
    void* args[] = {(void*)&bv, &tv, &dp, last_arg, &rpc};
    { KernelTimer t(h, timer);
      CU(launch_kernel(h, kern, grid, block, smem, pdl, args)); }
    CU(cudaGetLastError());
    return LVC_OK;
}

// The insertion counts of one batch (lvc_enable_insertions), launched right behind its first deposit pass while the batch
// buffers are valid.  Programmatic serialization lets it overlap the deposit's tail; it reads no table the deposit writes.
static int launch_count_insertions(lvc_handle* h, const BatchView& bv) {
    if (!h->ins.keys || bv.n_reads == 0) return LVC_OK;
    InsCountParams cp;
    cp.G = h->G; cp.min_bq = h->min_bq; cp.min_mq = h->min_mq;
    { KernelTimer t(h, 4);
      CU(launch_kernel(h, k_count_insertions, dim3((bv.n_reads + kInsThreads - 1) / kInsThreads), dim3(kInsThreads), 0, true,
                       bv, h->ins, cp, bv.n_reads)); }
    CU(cudaGetLastError());
    return LVC_OK;
}

static int deposit_with_replay(lvc_handle* h, const BatchView& bv, uint64_t n_cigar_ops, uint64_t n_qual,
                               const lvc_batch* account = nullptr) {
    if ((uint64_t)h->ordinal + bv.n_reads >= 0xFFFFFFFFull)
        return fail(h, LVC_ERANGE, "first-seen ordinal space (2^32-1 reads per handle) exhausted");
    h->tables_touched = true;
    CU(cudaMemsetAsync(h->d_status, 0, ST_WORDS * sizeof(uint32_t), h->stream));
    int rc = launch_deposit(h, bv, 0, n_cigar_ops, n_qual);
    if (rc) return rc;
    rc = launch_count_insertions(h, bv);           // once per batch: the replay pass below does not count again
    if (rc) return rc;
    CU(cudaMemcpyAsync(h->h_status, h->d_status, ST_WORDS * sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(h->h_status + ST_WORDS, h->d_newkeys, 32 * sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    if (account) {
        // zero-copy push: what crosses PCIe is what the kernel requests -- per chunk of kT5Reads reads the 16-byte
        // groups of the byte extent [first live read, end of last live read) (dead reads in between ride along; chunks
        // with no live read request nothing).  Counted here, on the host, while the kernel runs.
        uint64_t moved = 0;
        const size_t n = account->n_reads;
        for (size_t c0 = 0; c0 < n; c0 += kT5Reads) {
            const size_t c1 = std::min(n, c0 + kT5Reads);
            uint64_t lo = ~0ull, hi = 0;
            for (size_t i = c0; i < c1; ++i) {
                const bool live = read_passes_filter(account->flag[i], account->mapq[i], account->keep[i], h->min_mq);
                if (live) { lo = std::min<uint64_t>(lo, account->seq_off[i]); hi = std::max<uint64_t>(hi, account->seq_off[i + 1]); }
            }
            if (hi > lo) { const uint64_t q = ((hi + 15) & ~15ull) - (lo & ~15ull); moved += (account->qual_bits == 2u ? q / 4 : q) + ((account->seq_form & 255u) == 2u ? q / 4 : q / 2); }
        }
        h->h2d_payload_bytes += moved;
    }
    CU(cudaStreamSynchronize(h->stream));
    if (h->h_status[ST_RANGE_ERR]) {
        h->ordinal += bv.n_reads;
        return fail(h, LVC_ERANGE, "%u read(s) extend outside the reference [0, %lld); they were skipped",
                    h->h_status[ST_RANGE_ERR], (long long)h->G);
    }
    if (h->h_status[ST_UNMAPPED]) {
        // new (allele group, quality) keys: allocate their planes and replay ONLY those keys
        for (int k = 0; k < kMaxKeys; ++k)
            if ((h->h_status[ST_WORDS + (k >> 5)] >> (k & 31)) & 1u) {
                rc = add_plane(h, (uint16_t)k);
                if (rc) return rc;
            }
        CU(cudaMemcpyAsync(h->d_replay, h->d_newkeys, 32 * sizeof(uint32_t), cudaMemcpyDeviceToDevice, h->stream));
        CU(cudaMemsetAsync(h->d_newkeys, 0, 32 * sizeof(uint32_t), h->stream));
        CU(cudaMemsetAsync(h->d_status, 0, ST_WORDS * sizeof(uint32_t), h->stream));
        rc = launch_deposit(h, bv, 1, n_cigar_ops, n_qual);
        if (rc) return rc;
        CU(cudaStreamSynchronize(h->stream));
    }
    h->ordinal += bv.n_reads;
    return LVC_OK;
}

// Sample qualities: pre-allocate planes for the passing values seen (so the first pass rarely needs a
// replay) and pick the most frequent passing value as the tiled kernel's register-path quality.
// `dict` != nullptr: the sample holds 2-bit quality codes (four per byte) of a quality-code batch
static int premap_from_sample(lvc_handle* h, const uint8_t* q, uint64_t n, uint64_t stride, const uint8_t* dict = nullptr) {
    uint32_t hist[256] = {0};
    if (dict) {
        uint32_t ch[4] = {0, 0, 0, 0};
        for (uint64_t i = 0; i < n; i += stride) { const uint32_t v = q[i]; ch[v & 3]++; ch[(v >> 2) & 3]++; ch[(v >> 4) & 3]++; ch[v >> 6]++; }
        for (int c = 0; c < 4; ++c) hist[dict[c]] += ch[c];
    } else
    for (uint64_t i = 0; i < n; i += stride) hist[q[i]]++;
    int best = 255;
    uint32_t best_n = 0;
    for (int v = h->min_bq; v < 255; ++v)
        if (hist[v]) {
            int rc = add_plane(h, (uint16_t)v);
            if (rc) return rc;
            if (hist[v] > best_n) { best_n = hist[v]; best = v; }
        }
    h->qprim = best;
    return LVC_OK;
}

static constexpr uint32_t kSampleRows = 512, kSampleRowBytes = 64;

static int premap_host(lvc_handle* h, const lvc_batch* b) {
    const uint64_t nq = b->n_qual_bytes;
    // 32768 strided probes of the caller's buffer cost ~1 ms of cache and TLB misses in front of the kernel launch.
    // The first batch of a handle pays that (it creates the planes); later batches only re-elect the primary
    // quality from 2048 probes, and a quality never seen before still gets its plane through the replay path.
    const uint64_t probes = h->planes.empty() ? 32768 : 2048;
    if (b->qual_bits == 2u) return premap_from_sample(h, b->qual, nq / 4, std::max<uint64_t>(1, nq / 4 / probes), b->qual_dict);
    return premap_from_sample(h, b->qual, nq, std::max<uint64_t>(1, nq / probes));
}

// device-resident batch: gather a strided sample (kSampleRows rows of 64 bytes) with one 2-D copy
static int premap_device(lvc_handle* h, const lvc_batch* b) {
    const bool qc = b->qual_bits == 2u;
    const uint64_t nq = qc ? b->n_qual_bytes / 4 : b->n_qual_bytes;       // bytes of the quality array
    if (nq == 0) { h->qprim = 255; return LVC_OK; }
    if (!h->h_sample) CU(cudaHostAlloc(&h->h_sample, kSampleRows * kSampleRowBytes, cudaHostAllocDefault));
    uint64_t rows = kSampleRows, width = kSampleRowBytes;
    if (nq < rows * width) { rows = 1; width = std::min<uint64_t>(nq, kSampleRows * kSampleRowBytes); }
    const uint64_t pitch = rows > 1 ? nq / rows : width;
    CU(cudaMemcpy2DAsync(h->h_sample, width, b->qual, pitch, width, rows, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return premap_from_sample(h, h->h_sample, rows * width, 1, qc ? b->qual_dict : nullptr);
}

static int validate_batch(lvc_handle* h, const lvc_batch* b) {
    if (!h || !b) return LVC_EINVAL;
    if (b->n_reads == 0) return LVC_OK;
    if (!b->pos || !b->flag || !b->mapq || !b->keep || !b->cigar_off || !b->cigar || !b->seq_off || !b->seq4 || !b->qual)
        return fail(h, LVC_EINVAL, "lvc_batch has a null array");
    if (b->qual_bits != 0 && b->qual_bits != 8 && b->qual_bits != 2)
        return fail(h, LVC_EINVAL, "lvc_batch.qual_bits must be 0 / 8 (phred bytes) or 2 (codes into qual_dict), not %u", b->qual_bits);
    const uint32_t sbits = b->seq_form & 255u, s_min_bq = (b->seq_form >> 8) & 255u;
    if (sbits != 0 && sbits != 4 && sbits != 2)
        return fail(h, LVC_EINVAL, "lvc_batch.seq_form: base width must be 0 / 4 (BAM nibbles) or 2 (codes), not %u", sbits);
    if (sbits == 2) {
        if (b->qual_bits != 2) return fail(h, LVC_EINVAL, "2-bit base codes need 2-bit quality codes (qual_bits = 2)");
        // bases whose quality is below the threshold the codes were made for are not represented (lvc_pack_base_codes)
        if ((uint32_t)std::max(h->min_bq, 0) < s_min_bq)
            return fail(h, LVC_EINVAL, "the batch's 2-bit base codes were made for a base-quality threshold of %u; this handle uses %d",
                        s_min_bq, h->min_bq);
    }
    return LVC_OK;
}

// the batch as the kernels see it: the caller's arrays and the batch's quality form
static BatchView batch_view(const lvc_batch* b) {
    BatchView bv;
    bv.n_reads = b->n_reads;
    bv.pos = b->pos; bv.flag = b->flag; bv.mapq = b->mapq; bv.keep = b->keep;
    bv.cigar_off = b->cigar_off; bv.cigar = b->cigar; bv.seq_off = b->seq_off; bv.seq4 = b->seq4; bv.qual = b->qual;
    bv.qbits = b->qual_bits == 2u ? 2u : 0u;
    bv.sbits = (b->seq_form & 255u) == 2u ? 2u : 0u;
    bv.qdict = (uint32_t)b->qual_dict[0] | ((uint32_t)b->qual_dict[1] << 8) | ((uint32_t)b->qual_dict[2] << 16) |
               ((uint32_t)b->qual_dict[3] << 24);
    return bv;
}

int lvc_push_batch(lvc_handle* h, const lvc_batch* b) {
    NvtxRange nvtx_range("lvc_push_batch");
    int rc = validate_batch(h, b);
    if (rc) return rc;
    if (b->n_reads == 0) return LVC_OK;
    CU(cudaSetDevice(h->device));
    if (b->cigar_off[b->n_reads] != b->n_cigar_ops || b->seq_off[b->n_reads] != b->n_qual_bytes)
        return fail(h, LVC_EINVAL, "lvc_batch: n_cigar_ops / n_qual_bytes do not match the offset arrays");
    const size_t n = b->n_reads;
    struct { DevBuf* d; const void* s; size_t bytes; bool copy; } cp[] = {
        {&h->b_pos, b->pos, n * 4, true},           {&h->b_flag, b->flag, n * 2, true},
        {&h->b_mapq, b->mapq, n, true},             {&h->b_keep, b->keep, n, true},
        {&h->b_coff, b->cigar_off, (n + 1) * 4, true}, {&h->b_cig, b->cigar, (size_t)b->n_cigar_ops * 4, true},
        {&h->b_soff, b->seq_off, (n + 1) * 8, true},
        {&h->b_seq, b->seq4, (size_t)((b->seq_form & 255u) == 2u ? (b->n_qual_bytes + 3) / 4 : (b->n_qual_bytes + 1) / 2), false},
        {&h->b_qual, b->qual, (size_t)(b->qual_bits == 2u ? (b->n_qual_bytes + 3) / 4 : b->n_qual_bytes), false},
    };
    const bool qc = b->qual_bits == 2u;
    const bool b2 = (b->seq_form & 255u) == 2u;              // 2-bit base codes: a quarter byte per base instead of a half
    // LVC_ZC_HEADERS=1: the per-read arrays other than `keep` are read in place too when they are page-locked -- a chunk
    // whose reads were all dropped leaves after its `keep` bytes (copied in bulk) and never asks for the rest
    const void* hdr_alias[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    bool hdr_in_place = false;
    if (h->zero_copy_ok && h->zc_headers) {
        hdr_in_place = true;
        for (int k = 0; k < 7 && hdr_in_place; ++k) {
            if (k == 3) continue;                                       // keep: always copied
            cudaPointerAttributes a;
            if (cudaPointerGetAttributes(&a, cp[k].s) == cudaSuccess && a.type == cudaMemoryTypeHost && a.devicePointer)
                hdr_alias[k] = a.devicePointer;
            else { cudaGetLastError(); hdr_in_place = false; }
        }
    }
    for (int k = 0; k < 9; ++k) {
        auto& c = cp[k];
        if (hdr_in_place && k < 7 && k != 3) continue;
        rc = ensure(h, *c.d, c.bytes + 64);     // +64: the tiled kernel reads whole 16-byte groups
        if (rc) return rc;
        if (c.bytes && c.copy) CU(cudaMemcpyAsync(c.d->p, c.s, c.bytes, cudaMemcpyHostToDevice, h->stream));
    }
    // Payload (4-bit bases + qualities).  If the caller's buffers are page-locked (lvc_host_alloc / cudaHostAlloc)
    // the kernels read them IN PLACE over PCIe: every chunk's TMA bulk copy pulls exactly the bytes of the reads
    // that will be deposited, with thousands of requests in flight, and reads dropped by the host admission are
    // never transferred.  Otherwise only the byte ranges of admitted reads are copied (pageable memory).
    const uint8_t* dev_qual = (const uint8_t*)h->b_qual.p;
    const uint8_t* dev_seq = (const uint8_t*)h->b_seq.p;
    bool zero_copy = false;
    // A batch without dropped reads (ReadBatch.admitted_only / lvc_reads_compact) has nothing to skip: its payload is one
    // contiguous range, and one bulk copy per array on the copy engine moves it a little faster than the kernel's in-place
    // reads do (config 2, 109 MB: 2.43 against 2.56 ms per step).  1024 probes of `keep`, then eight bytes per test.
    const char* dense_env = getenv("LVC_DENSE_BULK_COPY");            // 0: always read page-locked payload in place
    bool dense = dense_env ? atoi(dense_env) != 0 : true;
    if (dense) {
        const size_t stride = std::max<size_t>(1, n / 1024);
        for (size_t i = 0; i < n && dense; i += stride) dense = (b->keep[i] & 1u) != 0;
        size_t i = 0;
        for (; i + 8 <= n && dense; i += 8) {
            uint64_t w; memcpy(&w, b->keep + i, 8);
            dense = (w & 0x0101010101010101ull) == 0x0101010101010101ull;
        }
        for (; i < n && dense; ++i) dense = (b->keep[i] & 1u) != 0;
    }
    if (dense) {
        const size_t qb = (size_t)(qc ? (b->n_qual_bytes + 3) / 4 : b->n_qual_bytes);
        const size_t sb = (size_t)(b2 ? (b->n_qual_bytes + 3) / 4 : (b->n_qual_bytes + 1) / 2);
        if (qb) CU(cudaMemcpyAsync(h->b_qual.p, b->qual, qb, cudaMemcpyHostToDevice, h->stream));
        if (sb) CU(cudaMemcpyAsync(h->b_seq.p, b->seq4, sb, cudaMemcpyHostToDevice, h->stream));
        h->h2d_payload_bytes += qb + sb;
    }
    if (h->zero_copy_ok && !dense) {
        cudaPointerAttributes aq, as;
        if (cudaPointerGetAttributes(&aq, b->qual) == cudaSuccess && cudaPointerGetAttributes(&as, b->seq4) == cudaSuccess &&
            aq.type == cudaMemoryTypeHost && as.type == cudaMemoryTypeHost && aq.devicePointer && as.devicePointer &&
            ((uintptr_t)aq.devicePointer & 15u) == 0 && ((uintptr_t)as.devicePointer & 15u) == 0) {
            dev_qual = (const uint8_t*)aq.devicePointer;
            dev_seq = (const uint8_t*)as.devicePointer;
            zero_copy = true;          // (the bytes pulled over PCIe are accounted while the kernel runs, below)
        } else {
            cudaGetLastError();
        }
    }
    if (!zero_copy && !dense) {
        const uint32_t kGap = 64;                 // merge live ranges separated by fewer dropped reads than this
        size_t i = 0;
        while (i < n) {
            while (i < n && !(b->keep[i] & 1u)) ++i;
            if (i >= n) break;
            size_t j = i, last_live = i;
            while (j < n && j - last_live <= kGap) { if (b->keep[j] & 1u) last_live = j; ++j; }
            const size_t end = last_live + 1;
            const uint64_t q0 = b->seq_off[i] & ~15ull, q1 = std::min<uint64_t>((b->seq_off[end] + 15) & ~15ull, b->n_qual_bytes);
            if (q1 > q0) {
                if (qc) CU(cudaMemcpyAsync((uint8_t*)h->b_qual.p + q0 / 4, b->qual + q0 / 4, (q1 - q0 + 3) / 4, cudaMemcpyHostToDevice, h->stream));
                else
                CU(cudaMemcpyAsync((uint8_t*)h->b_qual.p + q0, b->qual + q0, q1 - q0, cudaMemcpyHostToDevice, h->stream));
                const uint64_t s0 = b2 ? q0 >> 2 : q0 >> 1;
                const uint64_t s1 = b2 ? std::min<uint64_t>((q1 + 3) >> 2, (b->n_qual_bytes + 3) >> 2) : std::min<uint64_t>((q1 + 1) >> 1, (b->n_qual_bytes + 1) >> 1);
                CU(cudaMemcpyAsync((uint8_t*)h->b_seq.p + s0, b->seq4 + s0, s1 - s0, cudaMemcpyHostToDevice, h->stream));
                h->h2d_payload_bytes += (qc ? (q1 - q0 + 3) / 4 : (q1 - q0)) + (s1 - s0);
            }
            i = end;
        }
    }
    rc = premap_host(h, b);
    if (rc) return rc;
    BatchView bv = batch_view(b);
    bv.pos = (const int32_t*)h->b_pos.p;       bv.flag = (const uint16_t*)h->b_flag.p;
    bv.mapq = (const uint8_t*)h->b_mapq.p;     bv.keep = (const uint8_t*)h->b_keep.p;
    bv.cigar_off = (const uint32_t*)h->b_coff.p; bv.cigar = (const uint32_t*)h->b_cig.p;
    bv.seq_off = (const uint64_t*)h->b_soff.p; bv.seq4 = dev_seq;
    if (hdr_in_place) {
        bv.pos = (const int32_t*)hdr_alias[0]; bv.flag = (const uint16_t*)hdr_alias[1]; bv.mapq = (const uint8_t*)hdr_alias[2];
        bv.cigar_off = (const uint32_t*)hdr_alias[4]; bv.cigar = (const uint32_t*)hdr_alias[5];
        bv.seq_off = (const uint64_t*)hdr_alias[6];
        bv.hdr_lazy = 1;
    }
    bv.qual = dev_qual;
    return deposit_with_replay(h, bv, b->n_cigar_ops, b->n_qual_bytes, zero_copy ? b : nullptr);
}

int lvc_push_batch_device(lvc_handle* h, const lvc_batch* b) {
    NvtxRange nvtx_range("lvc_push_batch_device");
    int rc = validate_batch(h, b);
    if (rc) return rc;
    if (b->n_reads == 0) return LVC_OK;
    CU(cudaSetDevice(h->device));
    const BatchView bv = batch_view(b);
    rc = premap_device(h, b);
    if (rc) return rc;
    return deposit_with_replay(h, bv, b->n_cigar_ops, b->n_qual_bytes);
}

int lvc_push_batch_device_async(lvc_handle* h, const lvc_batch* b) {
    NvtxRange nvtx_range("lvc_push_batch_device_async");
    int rc = validate_batch(h, b);
    if (rc) return rc;
    if (b->n_reads == 0) return LVC_OK;
    CU(cudaSetDevice(h->device));
    if ((uint64_t)h->ordinal + b->n_reads >= 0xFFFFFFFFull)
        return fail(h, LVC_ERANGE, "first-seen ordinal space (2^32-1 reads per handle) exhausted");
    const BatchView bv = batch_view(b);
    if (h->qprim == 255) {
        // the first push of this handle is an asynchronous one (peer tables: nothing may be deposited before the tables
        // are mapped): elect the tiled kernel's primary quality now (one small copy + stream synchronisation)
        rc = premap_device(h, b);
        if (rc) return rc;
    }
    h->tables_touched = true;
    rc = launch_deposit(h, bv, 0, b->n_cigar_ops, b->n_qual_bytes);
    if (rc) return rc;
    rc = launch_count_insertions(h, bv);
    if (rc) return rc;
    h->ordinal += b->n_reads;
    return LVC_OK;
}

int lvc_check_async(lvc_handle* h) {
    if (!h) return LVC_EINVAL;
    CU(cudaSetDevice(h->device));
    CU(cudaMemcpyAsync(h->h_status, h->d_status, ST_WORDS * sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    const uint32_t unmapped = h->h_status[ST_UNMAPPED], range = h->h_status[ST_RANGE_ERR];
    CU(cudaMemsetAsync(h->d_status, 0, ST_WORDS * sizeof(uint32_t), h->stream));
    CU(cudaMemsetAsync(h->d_newkeys, 0, 32 * sizeof(uint32_t), h->stream));
    if (range) return fail(h, LVC_ERANGE, "%u read(s) extend outside the reference; they were skipped", range);
    if (unmapped)
        return fail(h, LVC_EAGAIN, "%u base(s) had a (allele group, quality) key without a plane during async pushes; "
                    "their counts are missing -- push the first batch of a stream synchronously", unmapped);
    return LVC_OK;
}

int lvc_set_timing(lvc_handle* h, int on) {
    if (!h) return LVC_EINVAL;
    h->timing = on != 0;
    return LVC_OK;
}

int lvc_get_timing(lvc_handle* h, int which, double* ms_total, uint64_t* n_launches) {
    if (!h || which < 0 || which > 4 || !ms_total || !n_launches) return LVC_EINVAL;
    if (which == 4 && !h->ins.keys) return fail(h, LVC_EINVAL, "timer 4 (insertion counts) needs lvc_enable_insertions");
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    double tot = 0.0;
    for (auto& pr : h->ev[which]) {
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, pr.first, pr.second));
        tot += ms;
        h->ev_pool.push_back(pr.first);
        h->ev_pool.push_back(pr.second);
    }
    *ms_total = tot;
    *n_launches = h->ev[which].size();
    h->ev[which].clear();
    return LVC_OK;
}

// ------------------------------------------------------------------------------------------------
// genotype
// ------------------------------------------------------------------------------------------------
// the planes ordered by key -- group 0 (A/C/G/T) first, then groups 1..3 -- with their keys; the planes of group g are
// [grp_begin[g], grp_begin[g + 1])
static void ordered_planes(const lvc_handle* h, std::vector<uint32_t*>& ptrs, std::vector<uint16_t>& keys, int grp_begin[5]) {
    const int np = (int)h->planes.size();
    std::vector<int> order(np);
    for (int i = 0; i < np; ++i) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return h->plane_key[a] < h->plane_key[b]; });
    ptrs.assign(std::max(np, 1), nullptr);
    keys.assign(std::max(np, 1), 0);
    for (int g = 0; g < 5; ++g) grp_begin[g] = 0;
    for (int i = 0; i < np; ++i) {
        ptrs[i] = h->planes[order[i]];
        keys[i] = h->plane_key[order[i]];
        grp_begin[(keys[i] >> 8) + 1] = i + 1;
    }
    for (int g = 1; g <= 4; ++g) grp_begin[g] = std::max(grp_begin[g], grp_begin[g - 1]);
}

static int genotype_enqueue(lvc_handle* h, int64_t min_total_depth, int64_t min_allele_depth, double min_ratio,
                            const double* e_lut, const double* om_lut, uint32_t flags) {
    const int np = (int)h->planes.size();
    std::vector<uint32_t*> ptrs; std::vector<uint16_t> keys; int grp_begin[5];
    ordered_planes(h, ptrs, keys, grp_begin);
    int rc = ensure(h, h->g_order_ptrs, ptrs.size() * sizeof(uint32_t*));
    if (rc) return rc;
    rc = ensure(h, h->g_order_keys, keys.size() * sizeof(uint16_t));
    if (rc) return rc;
    if (h->cand_cap == 0) {
        h->cand_cap = 1u << 16;
        rc = ensure(h, h->g_cand, (size_t)h->cand_cap * sizeof(lvc_candidate));
        if (rc) return rc;
    }
    bool tables_stale = false;
    if (h->geno_planes_uploaded != (size_t)np) {     // planes are only ever appended: the count identifies the set
        CU(cudaMemcpyAsync(h->g_order_ptrs.p, ptrs.data(), ptrs.size() * sizeof(uint32_t*), cudaMemcpyHostToDevice, h->stream));
        CU(cudaMemcpyAsync(h->g_order_keys.p, keys.data(), keys.size() * sizeof(uint16_t), cudaMemcpyHostToDevice, h->stream));
        h->geno_planes_uploaded = (size_t)np;
        tables_stale = true;
    }
    if (!h->lut_valid || memcmp(h->lut_host, e_lut, 256 * sizeof(double)) != 0 ||
        memcmp(h->lut_host + 256, om_lut, 256 * sizeof(double)) != 0) {
        memcpy(h->lut_host, e_lut, 256 * sizeof(double));
        memcpy(h->lut_host + 256, om_lut, 256 * sizeof(double));
        h->lut_valid = true;
        tables_stale = true;
    }
    if (tables_stale && np > 0) {
        // per plane: log2(e[q]) and log2(1 - e[q]) split into exactly summable pieces, from the caller's doubles in 80-bit arithmetic.
        // A zero probability (1 - e at q = 0) becomes a huge finite negative logarithm: its products vanish.
        rc = ensure(h, h->g_pconst, (size_t)np * sizeof(PlaneConst));
        if (rc) return rc;
        CU(cudaStreamSynchronize(h->stream));                 // the staging vector may still feed an earlier copy
        h->pconst_host.resize((size_t)np);
        // log2 of a probability in three pieces (genotype.cuh Acc3): multiples of 2^-10 and 2^-36 plus a remainder
        auto split3 = [](double v, double& c1, double& c2, double& c3) {
            if (!(v > 0.0)) { c1 = -1e290; c2 = 0.0; c3 = 0.0; return; }
            const long double l = log2l((long double)v);
            const long double a = roundl(l * 1024.0L) / 1024.0L;
            const long double r1 = l - a;
            const long double bq = roundl(r1 * 68719476736.0L) / 68719476736.0L;      // 2^36
            c1 = (double)a; c2 = (double)bq; c3 = (double)(r1 - bq);
        };
        for (int k = 0; k < np; ++k) {
            const uint32_t q = keys[(size_t)k] & 255u;
            PlaneConst& pc = h->pconst_host[(size_t)k];
            split3(e_lut[q], pc.le1, pc.le2, pc.le3);
            split3(om_lut[q], pc.lo1, pc.lo2, pc.lo3);
            pc.e = e_lut[q];
        }
        CU(cudaMemcpyAsync(h->g_pconst.p, h->pconst_host.data(), (size_t)np * sizeof(PlaneConst), cudaMemcpyHostToDevice,
                           h->stream));
    }
    GenoParams gp;
    gp.G = h->G; gp.p0 = h->geno_p0; gp.p1 = h->geno_p1 < 0 ? h->G : h->geno_p1; gp.min_total_depth = min_total_depth; gp.min_allele_depth = min_allele_depth;
    gp.min_ratio = min_ratio; gp.flags = flags; gp.n_planes = np; gp.cand_cap = h->cand_cap;
    for (int g = 0; g < 5; ++g) gp.grp_begin[g] = grp_begin[g];
    // one lane per (position, slot), also for wide quality alphabets (ONT: dozens of planes) on a short contig: measured
    // best on B200 (config 3, 61 planes: 19 us; 2 / 4 / 8 lanes sharing the planes of a slot: 23 / 27 / 36 us; the 4 warps
    // of a block sharing 8 positions: 23 us) -- the pass is bound by its fixed latency chain, not by loads in flight
    const int ppb = kGenoThreads / 4;                         // positions per block
    const unsigned blocks = (unsigned)((gp.p1 - (gp.p0 & ~7ll) + ppb - 1) / ppb);          // position 0 of a block is a multiple of 8
    if (gp.p1 <= gp.p0) { h->last_cand_count = 0; h->geno_pending = false; return LVC_OK; }
    {
        // Launched with programmatic stream serialization: its blocks may become resident while the deposit kernel
        // drains (that kernel signals launch_dependents at its start); k_genotype waits for the deposit kernel's
        // completion (griddepcontrol.wait) before it reads a table.  No memset sits between the two launches: the
        // candidate counter alternates between two words, each call clearing the other one.
        KernelTimer t(h, 2);
        h->cand_slot ^= 1;
        const auto kern = grp_begin[4] > grp_begin[1] ? k_genotype<4> : k_genotype<1>;
        const size_t smem = (size_t)np * sizeof(PlaneConst);
        if (smem > 48 * 1024) {        // > 877 planes: never seen, allowed (1024 keys x 56 B = 57 KB)
            CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kMaxKeys * sizeof(PlaneConst))));
        }
        CU(launch_kernel(h, kern, dim3(blocks), dim3(kGenoThreads), smem, true, gp, (const uint32_t* const*)h->g_order_ptrs.p,
                         (const PlaneConst*)h->g_pconst.p, (const uint32_t*)h->d_dels, (const uint8_t*)h->d_ref,
                         (const uint32_t* const*)h->d_first_arr, h->d_out_depth, h->d_out_ad, h->d_out_lik,
                         (lvc_candidate*)h->g_cand.p, h->d_cand_count + h->cand_slot, h->d_cand_count + (h->cand_slot ^ 1),
                         (h->d_seen && !h->seen_off) ? h->d_seen + 2 : (uint32_t*)nullptr));
    }
    CU(cudaGetLastError());
    h->geno_pending = true;
    return LVC_OK;
}

static int genotype_read_count(lvc_handle* h) {
    CU(cudaMemcpyAsync(h->h_status, h->d_cand_count + h->cand_slot, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    h->last_cand_count = h->h_status[0];
    h->geno_pending = false;
    return LVC_OK;
}

int lvc_genotype_device(lvc_handle* h, int64_t min_total_depth, int64_t min_allele_depth, double min_ratio,
                        const double* e_lut, const double* om_lut, uint32_t flags) {
    NvtxRange nvtx_range("lvc_genotype_device");
    if (!h || !e_lut || !om_lut) return LVC_EINVAL;
    CU(cudaSetDevice(h->device));
    for (int attempt = 0; attempt < 2; ++attempt) {
        int rc = genotype_enqueue(h, min_total_depth, min_allele_depth, min_ratio, e_lut, om_lut, flags);
        if (rc) return rc;
        rc = genotype_read_count(h);
        if (rc) return rc;
        if (h->last_cand_count <= h->cand_cap) break;
        // grow and run once more (rare: more candidates than the buffer)
        h->cand_cap = h->last_cand_count + h->last_cand_count / 4 + 1024;
        rc = ensure(h, h->g_cand, (size_t)h->cand_cap * sizeof(lvc_candidate));
        if (rc) return rc;
    }
    return LVC_OK;
}

int lvc_genotype_device_async(lvc_handle* h, int64_t min_total_depth, int64_t min_allele_depth, double min_ratio,
                              const double* e_lut, const double* om_lut, uint32_t flags) {
    NvtxRange nvtx_range("lvc_genotype_device_async");
    if (!h || !e_lut || !om_lut) return LVC_EINVAL;
    CU(cudaSetDevice(h->device));
    return genotype_enqueue(h, min_total_depth, min_allele_depth, min_ratio, e_lut, om_lut, flags);
}

int lvc_set_genotype_range(lvc_handle* h, int64_t p0, int64_t p1) {
    if (!h) return LVC_EINVAL;
    if (p1 < 0) { h->geno_p0 = 0; h->geno_p1 = -1; return LVC_OK; }
    if (p0 < 0 || p1 > h->G || p0 > p1) return fail(h, LVC_EINVAL, "genotype range [%lld, %lld) outside [0, %lld)",
                                                    (long long)p0, (long long)p1, (long long)h->G);
    h->geno_p0 = p0; h->geno_p1 = p1;
    return LVC_OK;
}

int lvc_fetch_candidates(lvc_handle* h, lvc_candidate* out, uint32_t cap, uint32_t* n_out) {
    if (!h || !n_out) return LVC_EINVAL;
    CU(cudaSetDevice(h->device));
    if (h->geno_pending) { int rc = genotype_read_count(h); if (rc) return rc; }
    *n_out = h->last_cand_count;
    const uint32_t n = std::min(std::min(cap, h->last_cand_count), h->cand_cap);
    if (n && out) {
        CU(cudaMemcpyAsync(out, h->g_cand.p, (size_t)n * sizeof(lvc_candidate), cudaMemcpyDeviceToHost, h->stream));
        CU(cudaStreamSynchronize(h->stream));
    }
    return LVC_OK;
}

int lvc_genotype(lvc_handle* h, int64_t min_total_depth, int64_t min_allele_depth, double min_ratio, const double* e_lut,
                 const double* om_lut, uint32_t flags, lvc_candidate* out, uint32_t cap, uint32_t* n_out) {
    NvtxRange nvtx_range("lvc_genotype");
    int rc = lvc_genotype_device(h, min_total_depth, min_allele_depth, min_ratio, e_lut, om_lut, flags);
    if (rc) return rc;
    return lvc_fetch_candidates(h, out, cap, n_out);
}

int lvc_copy_dense(lvc_handle* h, uint32_t* depth, uint32_t* ad, double* lik) {
    if (!h) return LVC_EINVAL;
    CU(cudaSetDevice(h->device));
    const size_t G = (size_t)h->G;
    if (depth) CU(cudaMemcpyAsync(depth, h->d_out_depth, G * 4, cudaMemcpyDeviceToHost, h->stream));
    if (ad) CU(cudaMemcpyAsync(ad, h->d_out_ad, G * 16, cudaMemcpyDeviceToHost, h->stream));
    if (lik) CU(cudaMemcpyAsync(lik, h->d_out_lik, G * 32, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return LVC_OK;
}

// ------------------------------------------------------------------------------------------------
// consensus + coverage statistics
// ------------------------------------------------------------------------------------------------
// the ordered plane list of the consensus and insertion-call passes (the genotype pass keeps its own device copy)
static int upload_consensus_planes(lvc_handle* h) {
    const int np = (int)h->planes.size();
    if (h->cons_planes_uploaded == (size_t)np) return LVC_OK;     // planes are only ever appended: the count identifies the set
    std::vector<uint32_t*> ptrs; std::vector<uint16_t> keys; int grp_begin[5];
    ordered_planes(h, ptrs, keys, grp_begin);
    int rc = ensure(h, h->c_order_ptrs, ptrs.size() * sizeof(uint32_t*));
    if (rc) return rc;
    CU(cudaMemcpyAsync(h->c_order_ptrs.p, ptrs.data(), ptrs.size() * sizeof(uint32_t*), cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));             // `ptrs` goes out of scope
    memcpy(h->cons_grp_begin, grp_begin, sizeof grp_begin);
    h->cons_planes_uploaded = (size_t)np;
    return LVC_OK;
}

int lvc_consensus(lvc_handle* h, int64_t p0, int64_t p1, uint64_t min_depth, double threshold,
                  const uint32_t* depth_thresholds, int n_thresholds, uint8_t* seq_out, lvc_consensus_stats* stats_out) {
    NvtxRange nvtx_range("lvc_consensus");
    if (!h) return LVC_EINVAL;
    if (!(threshold >= 0.0 && threshold <= 1.0))
        return fail(h, LVC_EINVAL, "consensus threshold %g outside [0, 1]", threshold);
    if (n_thresholds < 0 || n_thresholds > kConsMaxThr || (n_thresholds > 0 && !depth_thresholds))
        return fail(h, LVC_EINVAL, "consensus: %d depth thresholds (0..%d)", n_thresholds, kConsMaxThr);
    if (p1 < 0) { p0 = 0; p1 = h->G; }
    if (p0 < 0 || p1 > h->G || p0 > p1)
        return fail(h, LVC_EINVAL, "consensus range [%lld, %lld) outside [0, %lld)", (long long)p0, (long long)p1,
                    (long long)h->G);
    CU(cudaSetDevice(h->device));
    int rc = upload_consensus_planes(h);
    if (rc) return rc;
    const int64_t n = p1 - p0;
    rc = ensure(h, h->c_seq, (size_t)std::max<int64_t>(n, 1));
    if (rc) return rc;
    rc = ensure(h, h->c_stats, CS_WORDS * sizeof(uint64_t));
    if (rc) return rc;
    CU(cudaMemsetAsync(h->c_stats.p, 0, CS_WORDS * sizeof(uint64_t), h->stream));
    if (n > 0) {
        ConsParams cp;
        cp.p0 = p0; cp.p1 = p1; cp.min_depth = min_depth; cp.threshold = threshold;
        for (int g = 0; g < 5; ++g) cp.grp_begin[g] = h->cons_grp_begin[g];
        cp.n_thr = n_thresholds;
        for (int i = 0; i < kConsMaxThr; ++i) cp.thr[i] = i < n_thresholds ? depth_thresholds[i] : 0u;
        // a grid-stride loop over the range: a few blocks per SM keep enough rows in flight, and the block totals end in
        // one atomic per counter per block
        const unsigned blocks = (unsigned)std::min<int64_t>((n + kConsThreads - 1) / kConsThreads, (int64_t)h->sm_count * 16);
        // launched without programmatic serialization: it starts after every earlier kernel of the stream has finished
        KernelTimer t(h, 3);
        CU(launch_kernel(h, k_consensus, dim3(blocks), dim3(kConsThreads), 0, false, cp, (const uint32_t* const*)h->c_order_ptrs.p,
                         h->d_dels, h->d_ref, (uint8_t*)h->c_seq.p, (unsigned long long*)h->c_stats.p));
        CU(cudaGetLastError());
    }
    if (seq_out && n > 0) CU(cudaMemcpyAsync(seq_out, h->c_seq.p, (size_t)n, cudaMemcpyDeviceToHost, h->stream));
    uint64_t st[CS_WORDS];
    CU(cudaMemcpyAsync(st, h->c_stats.p, sizeof st, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    if (stats_out) {
        lvc_consensus_stats s;
        memset(&s, 0, sizeof s);
        s.n_positions = st[CS_POSITIONS]; s.depth_sum = st[CS_DEPTH_SUM]; s.depth_max = st[CS_DEPTH_MAX];
        s.n_low_depth = st[CS_LOW_DEPTH]; s.n_N = st[CS_N]; s.n_deleted = st[CS_DELETED];
        s.n_ambiguous = st[CS_AMBIGUOUS]; s.n_mismatch = st[CS_MISMATCH];
        for (int i = 0; i < n_thresholds; ++i) s.depth_ge[i] = st[CS_GE + i];
        *stats_out = s;
    }
    return LVC_OK;
}

// ------------------------------------------------------------------------------------------------
// insertions in the consensus
// ------------------------------------------------------------------------------------------------
static_assert(sizeof(lvc_insertion) == sizeof(InsEntry) && sizeof(lvc_insertion) == 24, "lvc_insertion layout");

int lvc_enable_insertions(lvc_handle* h, uint32_t max_keys) {
    if (!h) return LVC_EINVAL;
    if (max_keys == 0 || max_keys > (1u << 30))
        return fail(h, LVC_EINVAL, "lvc_enable_insertions: max_keys %u outside 1..2^30", max_keys);
    if (h->G > 0x7FFFFFFF) return fail(h, LVC_EINVAL, "lvc_enable_insertions: contig longer than 2^31 - 1");
    if (h->peer_ranks > 1) return fail(h, LVC_EINVAL, "lvc_enable_insertions: refused on a handle with peer tables attached");
    if (h->tables_touched)
        return fail(h, LVC_EINVAL, "lvc_enable_insertions: the tables already hold counts; call it after lvc_create or lvc_reset");
    CU(cudaSetDevice(h->device));
    size_t slots = 1;
    while (slots < 2 * (size_t)max_keys) slots <<= 1;
    CU(cudaStreamSynchronize(h->stream));
    cudaFree(h->ins.keys); cudaFree(h->ins.counts); cudaFree(h->ins.dropped);
    h->ins = InsTable{nullptr, nullptr, nullptr, 0};
    InsTable t = {nullptr, nullptr, nullptr, (uint32_t)(slots - 1)};
    if (cudaMalloc(&t.keys, slots * sizeof(ulonglong2)) != cudaSuccess || cudaMalloc(&t.counts, slots * sizeof(uint32_t)) != cudaSuccess ||
        cudaMalloc(&t.dropped, sizeof(uint32_t)) != cudaSuccess) {
        cudaGetLastError();
        cudaFree(t.keys); cudaFree(t.counts);
        return fail(h, LVC_ENOMEM, "lvc_enable_insertions: no device memory for %zu slots", slots);
    }
    h->ins = t;
    CU(cudaMemsetAsync(t.keys, 0, slots * sizeof(ulonglong2), h->stream));
    CU(cudaMemsetAsync(t.counts, 0, slots * sizeof(uint32_t), h->stream));
    CU(cudaMemsetAsync(t.dropped, 0, sizeof(uint32_t), h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return LVC_OK;
}

// the conditions both queries share: counting on, tables covered by the counts, nothing dropped
static int insertions_queryable(lvc_handle* h) {
    if (!h->ins.keys) return fail(h, LVC_EINVAL, "insertion counting is off (lvc_enable_insertions)");
    if (h->ins_uncovered)
        return fail(h, LVC_EINVAL, "the tables hold imported or reduced counts that the insertion counts do not cover; "
                    "lvc_reset starts over");
    CU(cudaMemcpyAsync(h->h_status, h->ins.dropped, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    const uint32_t dropped = h->h_status[0];
    if (dropped)
        return fail(h, LVC_ENOMEM, "%u insertion(s) found no free slot in the insertion table (%u slots); enable counting with "
                    "a larger max_keys", dropped, h->ins.mask + 1);
    return LVC_OK;
}

static bool insertion_before(const lvc_insertion& a, const lvc_insertion& b) {
    if (a.pos != b.pos) return a.pos < b.pos;
    if (a.len != b.len) return a.len < b.len;
    return a.seq < b.seq;
}

// n entries of the device list -> sorted, the first min(n, cap) into out
static int copy_sorted(lvc_handle* h, uint32_t n, lvc_insertion* out, uint32_t cap) {
    std::vector<lvc_insertion> v(n);
    if (n) CU(cudaMemcpyAsync(v.data(), h->i_list.p, (size_t)n * sizeof(lvc_insertion), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    std::sort(v.begin(), v.end(), insertion_before);
    if (out) std::copy(v.begin(), v.begin() + std::min(n, cap), out);
    return LVC_OK;
}

int lvc_copy_insertions(lvc_handle* h, lvc_insertion* out, uint32_t cap, uint32_t* n_out) {
    NvtxRange nvtx_range("lvc_copy_insertions");
    if (!h || !n_out || (cap && !out)) return LVC_EINVAL;
    CU(cudaSetDevice(h->device));
    int rc = insertions_queryable(h);
    if (rc) return rc;
    const size_t slots = (size_t)h->ins.mask + 1;
    rc = ensure(h, h->i_list, slots * sizeof(lvc_insertion) + sizeof(uint32_t));
    if (rc) return rc;
    uint32_t* d_n = (uint32_t*)((uint8_t*)h->i_list.p + slots * sizeof(lvc_insertion));
    CU(cudaMemsetAsync(d_n, 0, sizeof(uint32_t), h->stream));
    CU(launch_kernel(h, k_insertion_list, dim3((unsigned)((slots + kInsScanThreads - 1) / kInsScanThreads)), dim3(kInsScanThreads),
                     0, false, h->ins, (InsEntry*)h->i_list.p, (uint32_t)slots, d_n));
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(h->h_status, d_n, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    *n_out = h->h_status[0];
    return copy_sorted(h, *n_out, out, cap);
}

int lvc_insertion_calls(lvc_handle* h, int64_t p0, int64_t p1, uint64_t min_depth, double threshold, lvc_insertion* out,
                        uint32_t cap, uint32_t* n_out) {
    NvtxRange nvtx_range("lvc_insertion_calls");
    if (!h || !n_out || (cap && !out)) return LVC_EINVAL;
    if (!(threshold >= 0.0 && threshold <= 1.0))
        return fail(h, LVC_EINVAL, "insertion calls: threshold %g outside [0, 1]", threshold);
    if (p1 < 0) { p0 = 0; p1 = h->G; }
    if (p0 < 0 || p1 > h->G || p0 > p1)
        return fail(h, LVC_EINVAL, "insertion calls: range [%lld, %lld) outside [0, %lld)", (long long)p0, (long long)p1,
                    (long long)h->G);
    CU(cudaSetDevice(h->device));
    int rc = insertions_queryable(h);
    if (rc) return rc;
    rc = upload_consensus_planes(h);
    if (rc) return rc;
    const size_t slots = (size_t)h->ins.mask + 1;
    const size_t n = (size_t)(p1 - p0);
    // per-position scratch: total, unresolved, best, number of keys at the best
    rc = ensure(h, h->i_scratch, std::max<size_t>(n, 1) * 4 * sizeof(uint32_t));
    if (rc) return rc;
    rc = ensure(h, h->i_list, slots * sizeof(lvc_insertion) + sizeof(uint32_t));
    if (rc) return rc;
    uint32_t* sc = (uint32_t*)h->i_scratch.p;
    uint32_t* d_n = (uint32_t*)((uint8_t*)h->i_list.p + slots * sizeof(lvc_insertion));
    CU(cudaMemsetAsync(sc, 0, std::max<size_t>(n, 1) * 4 * sizeof(uint32_t), h->stream));
    CU(cudaMemsetAsync(d_n, 0, sizeof(uint32_t), h->stream));
    if (n > 0) {
        const dim3 grid((unsigned)((slots + kInsScanThreads - 1) / kInsScanThreads)), block(kInsScanThreads);
        uint32_t *total = sc, *unres = sc + n, *best = sc + 2 * n, *n_best = sc + 3 * n;
        InsCallParams ip;
        ip.p0 = p0; ip.p1 = p1; ip.min_depth = min_depth; ip.threshold = threshold;
        for (int g = 0; g < 5; ++g) ip.grp_begin[g] = h->cons_grp_begin[g];
        CU(launch_kernel(h, k_insertion_tally, grid, block, 0, false, h->ins, p0, p1, total, unres, best));
        CU(launch_kernel(h, k_insertion_ties, grid, block, 0, false, h->ins, p0, p1, (const uint32_t*)best, n_best));
        CU(launch_kernel(h, k_insertion_call, grid, block, 0, false, h->ins, ip, (const uint32_t* const*)h->c_order_ptrs.p,
                         (const uint32_t*)h->d_dels, (const uint32_t*)total, (const uint32_t*)unres, (const uint32_t*)best,
                         (const uint32_t*)n_best, (InsEntry*)h->i_list.p, d_n));
        CU(cudaGetLastError());
    }
    CU(cudaMemcpyAsync(h->h_status, d_n, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    *n_out = h->h_status[0];
    return copy_sorted(h, *n_out, out, cap);
}

// ------------------------------------------------------------------------------------------------
// table access
// ------------------------------------------------------------------------------------------------
int lvc_num_planes(lvc_handle* h) { return h ? (int)h->planes.size() : LVC_EINVAL; }

int lvc_plane_keys(lvc_handle* h, uint16_t* keys_out) {
    if (!h || !keys_out) return LVC_EINVAL;
    for (size_t i = 0; i < h->plane_key.size(); ++i) keys_out[i] = h->plane_key[i];
    return LVC_OK;
}

int lvc_ensure_plane(lvc_handle* h, uint16_t key) {
    if (!h) return LVC_EINVAL;
    CU(cudaSetDevice(h->device));
    int rc = add_plane(h, key);
    if (rc) return rc;
    CU(cudaStreamSynchronize(h->stream));
    return LVC_OK;
}

__global__ void k_accumulate_u32(uint32_t* __restrict__ dst, const uint32_t* __restrict__ src, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] += src[i];
}

static int import_u32(lvc_handle* h, uint32_t* d_dst, const uint32_t* src, size_t n, int accumulate) {
    if (!accumulate) {
        CU(cudaMemcpyAsync(d_dst, src, n * 4, cudaMemcpyHostToDevice, h->stream));
    } else {
        uint32_t* tmp = nullptr;
        CU(cudaMalloc(&tmp, n * 4));
        CU(cudaMemcpyAsync(tmp, src, n * 4, cudaMemcpyHostToDevice, h->stream));
        CU(launch_kernel(h, k_accumulate_u32, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, false, d_dst, tmp, n));
        CU(cudaStreamSynchronize(h->stream));
        CU(cudaFree(tmp));
    }
    CU(cudaStreamSynchronize(h->stream));
    return LVC_OK;
}

int lvc_copy_plane(lvc_handle* h, uint16_t key, uint32_t* dst) {
    if (!h || !dst || key >= kMaxKeys || h->lut[key] == kNoPlane) return fail(h, LVC_EINVAL, "no plane for key %u", key);
    CU(cudaSetDevice(h->device));
    CU(cudaMemcpyAsync(dst, h->planes[h->lut[key]], (size_t)h->G * 16, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return LVC_OK;
}

int lvc_import_plane(lvc_handle* h, uint16_t key, const uint32_t* src, int accumulate) {
    if (!h || !src) return LVC_EINVAL;
    h->tables_touched = h->ins_uncovered = true;
    CU(cudaSetDevice(h->device));
    int rc = add_plane(h, key);
    if (rc) return rc;
    return import_u32(h, h->planes[h->lut[key]], src, (size_t)h->G * 4, accumulate);
}

int lvc_copy_dels(lvc_handle* h, uint32_t* dst) {
    if (!h || !dst) return LVC_EINVAL;
    CU(cudaSetDevice(h->device));
    CU(cudaMemcpyAsync(dst, h->d_dels, (size_t)h->G * 4, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return LVC_OK;
}
int lvc_import_dels(lvc_handle* h, const uint32_t* src, int accumulate) {
    if (!h || !src) return LVC_EINVAL;
    h->tables_touched = h->ins_uncovered = true;
    CU(cudaSetDevice(h->device));
    return import_u32(h, h->d_dels, src, (size_t)h->G, accumulate);
}
int lvc_copy_covdiff(lvc_handle* h, int32_t* dst) {
    if (!h || !dst) return LVC_EINVAL;
    CU(cudaSetDevice(h->device));
    CU(cudaMemcpyAsync(dst, h->d_covdiff, (size_t)(h->G + 1) * 4, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return LVC_OK;
}
int lvc_import_covdiff(lvc_handle* h, const int32_t* src, int accumulate) {
    if (!h || !src) return LVC_EINVAL;
    h->tables_touched = h->ins_uncovered = true;
    CU(cudaSetDevice(h->device));
    return import_u32(h, (uint32_t*)h->d_covdiff, (const uint32_t*)src, (size_t)h->G + 1, accumulate);
}
int lvc_copy_first(lvc_handle* h, int group, uint32_t* dst) {
    if (!h || !dst || group < 0 || group > 3 || !h->d_first[group]) return LVC_EINVAL;
    CU(cudaSetDevice(h->device));
    CU(cudaMemcpyAsync(dst, h->d_first[group], (size_t)h->G * 16, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return LVC_OK;
}
int lvc_import_first(lvc_handle* h, int group, const uint32_t* src) {
    if (!h || !src || group < 0 || group > 3) return LVC_EINVAL;
    h->tables_touched = h->ins_uncovered = true;
    CU(cudaSetDevice(h->device));
    int rc = ensure_first_table(h, group);
    if (rc) return rc;
    CU(cudaMemsetAsync(h->d_seen, 0, h->seen_words * sizeof(uint32_t), h->stream));      // the hint describes the old table
    CU(cudaMemcpyAsync(h->d_first[group], src, (size_t)h->G * 16, cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return LVC_OK;
}
uint64_t lvc_ordinal(lvc_handle* h) { return h ? h->ordinal : 0; }
int lvc_set_ordinal(lvc_handle* h, uint64_t o) {
    if (!h || o >= 0xFFFFFFFFull) return LVC_EINVAL;
    h->ordinal = o;
    return LVC_OK;
}
void* lvc_plane_devptr(lvc_handle* h, uint16_t key) {
    if (!h || key >= kMaxKeys || h->lut[key] == kNoPlane) return nullptr;
    return h->planes[h->lut[key]];
}
void* lvc_dels_devptr(lvc_handle* h) { return h ? h->d_dels : nullptr; }
void* lvc_covdiff_devptr(lvc_handle* h) { return h ? h->d_covdiff : nullptr; }
void* lvc_first_devptr(lvc_handle* h, int group) {
    if (!h || group < 0 || group > 3) return nullptr;
    h->seen_off = true;       // the caller may write the table (halo exchange clears cells): no first-seen hints any more
    return h->d_first[group];
}
uint64_t lvc_launch_count(lvc_handle* h) { return h ? h->launches : 0; }
uint64_t lvc_h2d_payload_bytes(lvc_handle* h) { return h ? h->h2d_payload_bytes : 0; }

}  // extern "C"

#include "reduce_nccl.hpp"
#include "peer.hpp"
#include "ingest.hpp"
