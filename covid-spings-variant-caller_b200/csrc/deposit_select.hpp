// Which deposit kernel a batch runs on: a pure function of the batch's shape and the handle's state, host only (no CUDA
// headers) so that the rule is checked on the CPU (tests/test_deposit_select_cpu.py).
#pragma once
#include <cstdint>

namespace lvc {

enum class DepositKernel { general, warp, ont, tile3, tile4, tile5 };
enum class DepositError { none, planes_after_attach, qc_impl };

struct DepositInputs {
    int impl;                         // lvc_set_impl: 0 auto, 1 general, 2 tile3, 3 warp, 4 tile4, 5 tile5, 6 ONT
    uint64_t n_reads, n_cigar_ops;    // n_reads > 0
    bool replay;                      // second pass over the batch for the keys that had no plane
    bool small_contig;                // G < 2^30: the ONT kernel's cell indices are 32-bit
    bool peer, planes_changed;        // lvc_peer_attach is active; a plane was added since
    bool tile_ok;                     // primary quality < 128 with a plane, threshold <= 128: the tiled kernels' byte arithmetic
    bool qc, qc_prim_coded;           // 2-bit quality codes; the primary quality is one of the batch's four codes
    bool base_codes;                  // 2-bit base codes
};

struct DepositChoice {
    DepositError error;
    DepositKernel kernel;
    int t5_form;                      // payload form, the tile5 instantiation: 0 phred bytes, 1 quality codes, 2 quality + base codes
};

inline DepositChoice select_deposit(const DepositInputs& in) {
    // auto: long reads (ONT) take the CTA-cooperative kernel while their ops fit its tables (<= 40 per read on average),
    // else one warp per read; short reads take the generation-5 tiled kernel
    const bool long_reads = in.n_cigar_ops > 4ull * in.n_reads;
    const bool ont_ok = !in.replay && in.small_contig;
    int impl = in.impl;
    if (impl == 0) impl = !long_reads ? 5 : (in.n_cigar_ops <= 40ull * in.n_reads && ont_ok) ? 6 : 3;
    if (in.peer) {
        // peer tables: only the generation-5 tiled kernel and the any-record kernels route their reductions
        if (in.planes_changed) return {DepositError::planes_after_attach, DepositKernel::general, 0};
        if (impl != 5) impl = long_reads ? 3 : 1;
    }
    bool tile_ok = in.tile_ok;
    if (in.qc) {
        // quality-code batches: the generation-5 tiled kernel, or the any-record kernel
        if (in.impl != 0 && in.impl != 1 && in.impl != 5) return {DepositError::qc_impl, DepositKernel::general, 0};
        tile_ok = tile_ok && in.qc_prim_coded;
        impl = (impl == 1 || in.replay || !tile_ok) ? 1 : 5;
    }
    DepositKernel k = DepositKernel::tile5;
    if (impl == 6 && ont_ok) k = DepositKernel::ont;
    else if (impl == 3 || impl == 6) k = DepositKernel::warp;
    else if (impl == 1) k = DepositKernel::general;
    else if (in.replay || !tile_ok) k = long_reads ? DepositKernel::warp : DepositKernel::general;
    else if (impl == 2) k = DepositKernel::tile3;
    else if (impl == 4) k = DepositKernel::tile4;
    return {DepositError::none, k, in.qc ? (in.base_codes ? 2 : 1) : 0};
}

}  // namespace lvc
