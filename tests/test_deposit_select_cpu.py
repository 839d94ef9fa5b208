"""The deposit kernel selection rule (csrc/deposit_select.hpp) compiled on its own with g++ and checked on the CPU: every
combination of its inputs must pick the same kernel, tile5 instantiation or error as the branch chain that launch_deposit
carried before the rule was a function of its own, kept below as the reference."""
import os
import subprocess

from helpers import ROOT

CSRC = os.path.join(ROOT, "covid-spings-variant-caller_b200", "csrc")

HARNESS = r"""
#include "deposit_select.hpp"
#include <cstdio>
#include <initializer_list>
using namespace lvc;

// launch_deposit's branch chain as it was, with each launch replaced by the kernel it launched; tile_impl and long_impl
// are the defaults the environment switches LVC_TILE_IMPL and LVC_LONG_IMPL could once override
static DepositChoice reference(const DepositInputs& in) {
    const int h_impl = in.impl, h_long_impl = 6, h_tile_impl = 5;
    const uint64_t n = in.n_reads, n_cigar_ops = in.n_cigar_ops;
    const int replay = in.replay;
    const bool small_G = in.small_contig;                      // h->G < (1ll << 30)
    const bool peer = in.peer;                                 // h->peer_ranks > 1
    const bool qc = in.qc;                                     // bv.qbits == 2u
    const bool sbits2 = in.base_codes;                         // bv.sbits == 2u
    const DepositChoice general{DepositError::none, DepositKernel::general, 0}, warp{DepositError::none, DepositKernel::warp, 0},
        ont{DepositError::none, DepositKernel::ont, 0};
    const bool long_reads = n_cigar_ops > 4ull * n;
    const int long_impl = (n_cigar_ops <= 40ull * n && !replay && h_long_impl == 6 && small_G) ? 6 : 3;
    int impl = h_impl == 0 ? (long_reads ? long_impl : h_tile_impl) : h_impl;
    if (peer) {
        if (in.planes_changed)                                 // h->planes.size() != h->peer_planes_at_attach
            return {DepositError::planes_after_attach, DepositKernel::general, 0};
        impl = (impl == 5 || (h_impl == 0 && !long_reads)) ? 5 : (long_reads ? 3 : 1);
    }
    bool tile_ok = in.tile_ok;
    if (qc) {
        if (h_impl != 0 && h_impl != 1 && h_impl != 5) return {DepositError::qc_impl, DepositKernel::general, 0};
        tile_ok = tile_ok && in.qc_prim_coded;                 // qc_pcode < 4
        impl = (impl == 1 || replay || !tile_ok) ? 1 : 5;
    }
    if (qc && impl == 1) {
        return general;
    } else if (impl == 6 && !replay && small_G) {
        return ont;
    } else if (impl == 3 || impl == 6 || ((replay || !tile_ok) && impl != 1 && long_reads)) {
        return warp;
    } else if (impl == 1 || replay || !tile_ok) {
        return general;
    } else {
        if (impl == 4 || impl == 5) {
            if (impl == 5) {
                if (qc && sbits2) return {DepositError::none, DepositKernel::tile5, 2};
                else
                return {DepositError::none, DepositKernel::tile5, qc ? 1 : 0};
            } else return {DepositError::none, DepositKernel::tile4, 0};
        } else
            return {DepositError::none, DepositKernel::tile3, 0};
    }
}

int main() {
    long cases = 0, mismatches = 0, seen[3][6][3] = {};
    for (int impl = 0; impl <= 6; ++impl)
        for (uint64_t n : {uint64_t{1}, uint64_t{3}, uint64_t{1000}})
            // CIGAR ops per read: <= 4, in (4, 40], > 40, at and next to both boundaries
            for (uint64_t ops : {uint64_t{0}, 4 * n, 4 * n + 1, 17 * n, 40 * n, 40 * n + 1, 100 * n})
                for (int bits = 0; bits < 256; ++bits) {
                    DepositInputs in;
                    in.impl = impl; in.n_reads = n; in.n_cigar_ops = ops;
                    in.replay = bits & 1; in.small_contig = bits & 2; in.peer = bits & 4; in.planes_changed = bits & 8;
                    in.tile_ok = bits & 16; in.qc = bits & 32; in.qc_prim_coded = bits & 64; in.base_codes = bits & 128;
                    const DepositChoice a = select_deposit(in), b = reference(in);
                    ++cases;
                    const bool same = a.error == b.error && (a.error != DepositError::none ||
                                      (a.kernel == b.kernel && (a.kernel != DepositKernel::tile5 || a.t5_form == b.t5_form)));
                    if (!same) {
                        if (++mismatches < 8)
                            printf("impl %d n %llu ops %llu bits %d: select %d/%d/%d reference %d/%d/%d\n", impl,
                                   (unsigned long long)n, (unsigned long long)in.n_cigar_ops, bits, (int)a.error,
                                   (int)a.kernel, a.t5_form, (int)b.error, (int)b.kernel, b.t5_form);
                    }
                    ++seen[(int)b.error][(int)b.kernel][b.t5_form];
                }
    printf("cases %ld mismatches %ld\n", cases, mismatches);
    printf("errors %ld %ld\n", seen[1][0][0], seen[2][0][0]);
    for (int k = 0; k < 6; ++k) printf("kernel %d %ld %ld %ld\n", k, seen[0][k][0], seen[0][k][1], seen[0][k][2]);
    return mismatches == 0 ? 0 : 1;
}
"""


def test_select_matches_reference(tmp_path):
    src, exe = os.path.join(tmp_path, "h.cpp"), os.path.join(tmp_path, "h")
    with open(src, "w") as fh:
        fh.write(HARNESS)
    subprocess.run(["g++", "-O1", "-std=c++17", "-fsanitize=address,undefined",
                    "-fno-sanitize-recover=undefined", "-I", CSRC, "-o", exe, src], check=True)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300, env=dict(os.environ, ASAN_OPTIONS="detect_leaks=0"))
    assert r.returncode == 0, r.stdout + r.stderr
    lines = r.stdout.splitlines()
    assert lines[0].startswith("cases ") and lines[0].endswith(" mismatches 0"), r.stdout
    # the enumeration reaches both errors, every kernel and every tile5 instantiation
    errors = [int(x) for x in lines[1].split()[1:]]
    assert all(errors), r.stdout
    counts = {int(f[1]): [int(x) for x in f[2:]] for f in (ln.split() for ln in lines[2:])}
    assert all(counts[k][0] for k in range(6)), r.stdout
    assert counts[5][1] and counts[5][2], r.stdout
