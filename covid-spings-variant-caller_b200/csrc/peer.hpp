// Position ownership over NVLink peer memory (SURVEY 8e row 2 without an exchange step).
//
//   lvc_peer_export  serialises CUDA IPC handles of this handle's tables (every plane, dels, covdiff, first-seen);
//   lvc_peer_attach  opens the other ranks' handles (cudaIpcOpenMemHandle, peer access over NVLink / NVSwitch) and builds
//                    the device-side PeerView: from then on the deposit kernels reduce a base of column c straight into
//                    the tables of the rank that owns c (lvc_common.cuh: plane_row / first_row / dels_cell /
//                    covdiff_cell) -- remote REDs are resolved in the owner's L2, so after a stream-ordered barrier
//                    (lvc_stream_barrier) every rank genotypes its own slice of complete columns;
//   lvc_peer_detach  closes the mappings.
// One process per GPU; the blobs travel over whatever the caller has (torch.distributed all_gather_object in dist.py).
// The plane set must be the same on every rank when the blobs are made (ensure_plane on the union of the keys), and
// a plane added later needs a new export / attach round.  Included by lvc_api.cu.
#pragma once

namespace lvc_peer {

constexpr uint32_t kMagic = 0x4C565031u;   // "LVP1"
struct BlobHeader {
    uint32_t magic, n_planes;
    int64_t G;
    uint8_t has_first[4];
    uint32_t pad;
};

// planes in ascending key order: the same order on every rank
static std::vector<int> planes_by_key(const lvc_handle* h) {
    std::vector<int> order(h->planes.size());
    for (size_t i = 0; i < order.size(); ++i) order[i] = (int)i;
    std::sort(order.begin(), order.end(), [&](int a, int b) { return h->plane_key[a] < h->plane_key[b]; });
    return order;
}

}  // namespace lvc_peer

#define NC(call)                                                                                                    \
    do {                                                                                                            \
        const int r_ = (call);                                                                                      \
        if (r_ != 0) return fail(h, LVC_ECUDA, "%s failed: %s", #call, A->GetErrorString ? A->GetErrorString(r_) : "?"); \
    } while (0)

extern "C" {

int lvc_peer_export(lvc_handle* h, void* blob, size_t cap, size_t* len) {
    if (!h || !len) return LVC_EINVAL;
    CU(cudaSetDevice(h->device));
    const std::vector<int> order = lvc_peer::planes_by_key(h);
    const size_t np = order.size();
    const size_t need = sizeof(lvc_peer::BlobHeader) + ((np * 2 + 7) & ~(size_t)7) + (np + 2 + 4) * sizeof(cudaIpcMemHandle_t);
    *len = need;
    if (!blob) return LVC_OK;                      // size query
    if (cap < need) return fail(h, LVC_EINVAL, "lvc_peer_export: buffer of %zu bytes, %zu needed", cap, need);
    uint8_t* p = (uint8_t*)blob;
    memset(p, 0, need);
    lvc_peer::BlobHeader hd = {};
    hd.magic = lvc_peer::kMagic; hd.n_planes = (uint32_t)np; hd.G = h->G;
    for (int g = 0; g < 4; ++g) hd.has_first[g] = h->d_first[g] != nullptr;
    memcpy(p, &hd, sizeof(hd));
    p += sizeof(hd);
    for (size_t k = 0; k < np; ++k) { const uint16_t key = h->plane_key[order[k]]; memcpy(p + 2 * k, &key, 2); }
    p += (np * 2 + 7) & ~(size_t)7;
    auto put = [&](void* dev) -> int {
        cudaIpcMemHandle_t mh;
        memset(&mh, 0, sizeof(mh));
        if (dev) CU(cudaIpcGetMemHandle(&mh, dev));
        memcpy(p, &mh, sizeof(mh));
        p += sizeof(mh);
        return LVC_OK;
    };
    CU(cudaStreamSynchronize(h->stream));          // the tables exist and are initialised before anyone maps them
    for (size_t k = 0; k < np; ++k) { const int rc = put(h->planes[order[k]]); if (rc) return rc; }
    int rc = put(h->d_dels); if (rc) return rc;
    rc = put(h->d_covdiff); if (rc) return rc;
    for (int g = 0; g < 4; ++g) { rc = put(h->d_first[g]); if (rc) return rc; }
    return LVC_OK;
}

int lvc_peer_detach(lvc_handle* h) {
    if (!h) return LVC_EINVAL;
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    for (void* p : h->peer_opened) cudaIpcCloseMemHandle(p);
    h->peer_opened.clear();
    h->peer_ranks = 0;
    return LVC_OK;
}

int lvc_peer_attach(lvc_handle* h, int rank, int n_ranks, const void* const* blobs, const size_t* lens) {
    if (!h || !blobs || !lens || n_ranks < 1 || n_ranks > kMaxPeers || rank < 0 || rank >= n_ranks) return LVC_EINVAL;
    if (h->ins.keys) return fail(h, LVC_EINVAL, "lvc_peer_attach: refused on a handle that counts insertions");
    int rc = lvc_peer_detach(h);
    if (rc) return rc;
    if (n_ranks == 1) return LVC_OK;
    const std::vector<int> order = lvc_peer::planes_by_key(h);
    const size_t np = order.size();
    PeerView pv;
    memset(&pv, 0, sizeof(pv));
    pv.n_ranks = n_ranks; pv.rank = rank;
    pv.per = (h->G + 1 + n_ranks - 1) / n_ranks;                                   // lvc_position_slice
    pv.lo = std::min<int64_t>((int64_t)rank * pv.per, h->G);
    pv.hi = std::min<int64_t>((int64_t)(rank + 1) * pv.per, h->G);
    // [rank][local plane id] -> that rank's plane with the same key
    std::vector<uint32_t*> ptab((size_t)n_ranks * kMaxKeys, nullptr);
    for (int r = 0; r < n_ranks; ++r) {
        if (r == rank) {
            for (size_t k = 0; k < h->planes.size(); ++k) ptab[(size_t)r * kMaxKeys + k] = h->planes[k];
            pv.dels[r] = h->d_dels; pv.covdiff[r] = h->d_covdiff;
            for (int g = 0; g < 4; ++g) pv.first[r][g] = h->d_first[g];
            continue;
        }
        const uint8_t* p = (const uint8_t*)blobs[r];
        lvc_peer::BlobHeader hd;
        if (!p || lens[r] < sizeof(hd)) return fail(h, LVC_EINVAL, "lvc_peer_attach: blob of rank %d is too short", r);
        memcpy(&hd, p, sizeof(hd));
        const size_t need = sizeof(hd) + (((size_t)hd.n_planes * 2 + 7) & ~(size_t)7) + ((size_t)hd.n_planes + 6) * sizeof(cudaIpcMemHandle_t);
        if (hd.magic != lvc_peer::kMagic || hd.G != h->G || hd.n_planes != np || lens[r] < need)
            return fail(h, LVC_EINVAL, "lvc_peer_attach: rank %d has another contig or plane set (%u planes, G %lld)", r,
                        hd.n_planes, (long long)hd.G);
        p += sizeof(hd);
        for (size_t k = 0; k < np; ++k) {
            uint16_t key;
            memcpy(&key, p + 2 * k, 2);
            if (key != h->plane_key[order[k]]) return fail(h, LVC_EINVAL, "lvc_peer_attach: rank %d has another plane set", r);
        }
        p += (np * 2 + 7) & ~(size_t)7;
        auto get = [&](bool present, void** out) -> int {
            cudaIpcMemHandle_t mh;
            memcpy(&mh, p, sizeof(mh));
            p += sizeof(mh);
            *out = nullptr;
            if (!present) return LVC_OK;
            CU(cudaIpcOpenMemHandle(out, mh, cudaIpcMemLazyEnablePeerAccess));
            h->peer_opened.push_back(*out);
            return LVC_OK;
        };
        for (size_t k = 0; k < np; ++k) {
            void* q = nullptr;
            rc = get(true, &q); if (rc) return rc;
            ptab[(size_t)r * kMaxKeys + (size_t)order[k]] = (uint32_t*)q;
        }
        void* q = nullptr;
        rc = get(true, &q); if (rc) return rc; pv.dels[r] = (uint32_t*)q;
        rc = get(true, &q); if (rc) return rc; pv.covdiff[r] = (int32_t*)q;
        for (int g = 0; g < 4; ++g) {
            if ((hd.has_first[g] != 0) != (h->d_first[g] != nullptr)) return fail(h, LVC_EINVAL, "lvc_peer_attach: rank %d has another plane set", r);
            rc = get(hd.has_first[g] != 0, &q); if (rc) return rc; pv.first[r][g] = (uint32_t*)q;
        }
    }
    if (!h->d_peer_planes) CU(cudaMalloc(&h->d_peer_planes, (size_t)kMaxPeers * kMaxKeys * sizeof(uint32_t*)));
    if (!h->d_peer) CU(cudaMalloc(&h->d_peer, sizeof(PeerView)));
    for (int r = 0; r < n_ranks; ++r) pv.planes[r] = h->d_peer_planes + (size_t)r * kMaxKeys;
    CU(cudaMemcpyAsync(h->d_peer_planes, ptab.data(), ptab.size() * sizeof(uint32_t*), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_peer, &pv, sizeof(pv), cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    h->peer_ranks = n_ranks;
    h->peer_planes_at_attach = np;
    h->seen_off = true;                               // other ranks write this rank's first-seen cells: no hints
    h->geno_p0 = pv.lo; h->geno_p1 = pv.hi;           // this rank genotypes the columns it owns
    return LVC_OK;
}

// Stream-ordered barrier over the ranks of `nccl_comm` (a 4-byte all-reduce on the handle's stream): every rank's earlier
// work on its stream -- the deposit kernel with its remote reductions -- is complete before any rank's later work starts.
int lvc_stream_barrier(lvc_handle* h, void* nccl_comm) {
    if (!h || !nccl_comm) return LVC_EINVAL;
    lvc_nccl::Api* A = lvc_nccl::api();
    if (!A->err.empty()) return fail(h, LVC_EIO, "%s", A->err.c_str());
    CU(cudaSetDevice(h->device));
    if (!h->d_keymap) CU(cudaMalloc(&h->d_keymap, kMaxKeys));
    NC(A->AllReduce(h->d_keymap, h->d_keymap, 1, lvc_nccl::kInt32, lvc_nccl::kMax, nccl_comm, h->stream));
    h->launches++;
    return LVC_OK;
}

}  // extern "C"
#undef NC
