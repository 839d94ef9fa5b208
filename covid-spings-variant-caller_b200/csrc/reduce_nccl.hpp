// lvc_reduce_tables: the ONE exchange step of the read-chunk sharding (SURVEY 8e): integer SUM of the count tables and
// unsigned MIN of the first-seen ordinals over NCCL (NVLink 5 / NVSwitch), issued as one ncclGroup on the handle's
// stream, directly on the persistent device tables (no staging copy).
//
//   LVC_REDUCE_ALL      all-reduce: every rank ends with the tables of all ranks' reads;
//   LVC_REDUCE_SCATTER  reduce-scatter IN PLACE onto position slices: rank r ends with the complete columns
//                       [r*per, (r+1)*per), per = ceil((G+1)/n) (lvc_position_slice), everything else is cleared, and
//                       the genotype pass is restricted to that slice.  Half the bytes of the all-reduce.
//
// NCCL is bound at run time (dlopen of libnccl.so.2, preferring a copy the process already loaded, e.g. PyTorch's),
// so the library still loads -- for the host-only entry points -- where NCCL is absent.  Included by lvc_api.cu.
#pragma once
#include <dlfcn.h>

namespace lvc_nccl {

struct UniqueId { char internal[128]; };
typedef void* Comm;
enum { kSum = 0, kMax = 2, kMin = 3 };                 // ncclRedOp_t
enum { kUint8 = 1, kInt32 = 2, kUint32 = 3 };          // ncclDataType_t

struct Api {
    void* lib = nullptr;
    int (*GetUniqueId)(UniqueId*) = nullptr;
    int (*CommInitRank)(Comm*, int, UniqueId, int) = nullptr;
    int (*CommDestroy)(Comm) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, Comm, cudaStream_t) = nullptr;
    int (*ReduceScatter)(const void*, void*, size_t, int, int, Comm, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    std::string err;
};

static Api* api() {
    static Api a;
    static std::once_flag once;
    std::call_once(once, [] {
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char* n : names) { a.lib = dlopen(n, RTLD_NOW | RTLD_NOLOAD); if (a.lib) break; }
        if (!a.lib) for (const char* n : names) { a.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if (a.lib) break; }
        if (!a.lib) { a.err = std::string("cannot load libnccl.so.2: ") + (dlerror() ? dlerror() : "?"); return; }
        auto sym = [&](const char* s) { void* p = dlsym(a.lib, s); if (!p && a.err.empty()) a.err = std::string("NCCL symbol missing: ") + s; return p; };
        a.GetUniqueId = (decltype(a.GetUniqueId))sym("ncclGetUniqueId");
        a.CommInitRank = (decltype(a.CommInitRank))sym("ncclCommInitRank");
        a.CommDestroy = (decltype(a.CommDestroy))sym("ncclCommDestroy");
        a.AllReduce = (decltype(a.AllReduce))sym("ncclAllReduce");
        a.ReduceScatter = (decltype(a.ReduceScatter))sym("ncclReduceScatter");
        a.GroupStart = (decltype(a.GroupStart))sym("ncclGroupStart");
        a.GroupEnd = (decltype(a.GroupEnd))sym("ncclGroupEnd");
        a.GetErrorString = (decltype(a.GetErrorString))sym("ncclGetErrorString");
    });
    return &a;
}

}  // namespace lvc_nccl

#define NC(call)                                                                                                    \
    do {                                                                                                            \
        const int r_ = (call);                                                                                      \
        if (r_ != 0) return fail(h, LVC_ECUDA, "%s failed: %s", #call, A->GetErrorString ? A->GetErrorString(r_) : "?"); \
    } while (0)

extern "C" {

int lvc_nccl_unique_id(uint8_t id_out[128]) {
    lvc_nccl::Api* A = lvc_nccl::api();
    if (!id_out) return LVC_EINVAL;
    if (!A->err.empty()) { g_create_error = A->err; return LVC_EIO; }
    lvc_nccl::UniqueId id;
    if (A->GetUniqueId(&id) != 0) { g_create_error = "ncclGetUniqueId failed"; return LVC_ECUDA; }
    memcpy(id_out, id.internal, 128);
    return LVC_OK;
}

int lvc_nccl_comm_create(void** comm_out, int device, int n_ranks, int rank, const uint8_t id[128]) {
    lvc_nccl::Api* A = lvc_nccl::api();
    if (!comm_out || !id || n_ranks < 1 || rank < 0 || rank >= n_ranks) return LVC_EINVAL;
    if (!A->err.empty()) { g_create_error = A->err; return LVC_EIO; }
    if (cudaSetDevice(device) != cudaSuccess) { g_create_error = "cudaSetDevice failed"; return LVC_ECUDA; }
    lvc_nccl::UniqueId uid;
    memcpy(uid.internal, id, 128);
    lvc_nccl::Comm c = nullptr;
    const int r = A->CommInitRank(&c, n_ranks, uid, rank);
    if (r != 0) { g_create_error = std::string("ncclCommInitRank failed: ") + (A->GetErrorString ? A->GetErrorString(r) : "?"); return LVC_ECUDA; }
    *comm_out = c;
    return LVC_OK;
}

void lvc_nccl_comm_destroy(void* comm) {
    lvc_nccl::Api* A = lvc_nccl::api();
    if (comm && A->err.empty()) A->CommDestroy(comm);
}

int lvc_position_slice(const lvc_handle* h, int n_ranks, int rank, int64_t* p0, int64_t* p1) {
    if (!h || n_ranks < 1 || rank < 0 || rank >= n_ranks || !p0 || !p1) return LVC_EINVAL;
    const int64_t per = (h->G + 1 + n_ranks - 1) / n_ranks;
    *p0 = std::min<int64_t>((int64_t)rank * per, h->G);
    *p1 = std::min<int64_t>((int64_t)(rank + 1) * per, h->G);
    return LVC_OK;
}

int lvc_reduce_tables(lvc_handle* h, void* nccl_comm, int n_ranks, int rank, int mode) {
    NvtxRange nvtx_range("lvc_reduce_tables");
    if (!h || !nccl_comm || n_ranks < 1 || rank < 0 || rank >= n_ranks || (mode != LVC_REDUCE_ALL && mode != LVC_REDUCE_SCATTER))
        return LVC_EINVAL;
    if (n_ranks > kRowSlack - 2) return fail(h, LVC_EINVAL, "lvc_reduce_tables: at most %d ranks", kRowSlack - 2);
    lvc_nccl::Api* A = lvc_nccl::api();
    if (!A->err.empty()) return fail(h, LVC_EIO, "%s", A->err.c_str());
    CU(cudaSetDevice(h->device));
    h->last_exchange_bytes = 0;
    if (n_ranks == 1) return LVC_OK;
    h->tables_touched = h->ins_uncovered = true;      // the other ranks' counts arrive without their insertions
    // ---- (1) agree on the set of (allele group, quality) planes: byte-wise MAX of the 1024-key presence map
    if (!h->d_keymap) CU(cudaMalloc(&h->d_keymap, kMaxKeys));
    std::vector<uint8_t> present(kMaxKeys);
    for (int k = 0; k < kMaxKeys; ++k) present[k] = h->lut[k] != kNoPlane;
    CU(cudaMemcpyAsync(h->d_keymap, present.data(), kMaxKeys, cudaMemcpyHostToDevice, h->stream));
    NC(A->AllReduce(h->d_keymap, h->d_keymap, kMaxKeys, lvc_nccl::kUint8, lvc_nccl::kMax, nccl_comm, h->stream));
    CU(cudaMemcpyAsync(present.data(), h->d_keymap, kMaxKeys, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    for (int k = 0; k < kMaxKeys; ++k)
        if (present[k]) { const int rc = add_plane(h, (uint16_t)k); if (rc) return rc; }
    // ---- (2) one group of collectives over every table, the same order on every rank (ascending key)
    const size_t G = (size_t)h->G;
    const size_t per = (G + 1 + (size_t)n_ranks - 1) / (size_t)n_ranks;          // rows per rank
    struct Tab { void* p; size_t width; int dtype, op; int fill; };
    std::vector<Tab> tabs;
    for (int k = 0; k < kMaxKeys; ++k)
        if (h->lut[k] != kNoPlane) tabs.push_back({h->planes[h->lut[k]], 4, lvc_nccl::kUint32, lvc_nccl::kSum, 0});
    tabs.push_back({h->d_dels, 1, lvc_nccl::kUint32, lvc_nccl::kSum, 0});
    tabs.push_back({h->d_covdiff, 1, lvc_nccl::kInt32, lvc_nccl::kSum, 0});
    for (int g = 0; g < 4; ++g)
        if (h->d_first[g]) tabs.push_back({h->d_first[g], 4, lvc_nccl::kUint32, lvc_nccl::kMin, 0xFF});
    NC(A->GroupStart());
    for (const Tab& t : tabs) {
        if (mode == LVC_REDUCE_ALL) {
            const size_t cnt = (t.p == (void*)h->d_covdiff ? G + 1 : G) * t.width;
            NC(A->AllReduce(t.p, t.p, cnt, t.dtype, t.op, nccl_comm, h->stream));
            h->last_exchange_bytes += cnt * 4;
        } else {
            const size_t cnt = per * t.width;
            NC(A->ReduceScatter(t.p, (uint8_t*)t.p + (size_t)rank * cnt * 4, cnt, t.dtype, t.op, nccl_comm, h->stream));
            h->last_exchange_bytes += cnt * 4 * (size_t)n_ranks;
        }
    }
    NC(A->GroupEnd());
    h->launches++;
    if (mode == LVC_REDUCE_SCATTER) {
        CU(cudaMemsetAsync(h->d_seen, 0, h->seen_words * sizeof(uint32_t), h->stream));   // first-seen cells outside the slice are cleared below
        // ---- (3) only the rank's own slice is complete: clear the rest (the next batch's deposits start from zero there)
        for (const Tab& t : tabs) {
            const size_t row_b = t.width * 4, lo = (size_t)rank * per, hi = (size_t)(rank + 1) * per;
            const size_t rows = (size_t)n_ranks * per;                             // <= G + kRowSlack
            if (lo) CU(cudaMemsetAsync(t.p, t.fill, lo * row_b, h->stream));
            if (hi < rows) CU(cudaMemsetAsync((uint8_t*)t.p + hi * row_b, t.fill, (rows - hi) * row_b, h->stream));
        }
        h->geno_p0 = std::min<int64_t>((int64_t)rank * (int64_t)per, h->G);
        h->geno_p1 = std::min<int64_t>((int64_t)(rank + 1) * (int64_t)per, h->G);
        if (h->geno_p1 < 0) h->geno_p1 = 0;
    }
    return LVC_OK;
}

uint64_t lvc_last_exchange_bytes(lvc_handle* h) { return h ? h->last_exchange_bytes : 0; }

}  // extern "C"
#undef NC
