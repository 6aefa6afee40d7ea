// K5 — exact correction for read pairs that overlap at two or more loci.
//
// The reference scores a read pair once, with the log-likelihood of its WHOLE overlap (x_s, x_d)
// (similarity_matrix.cpp:221-241), which is not additive over loci. The first-order planes S, D
// count each shared locus separately; this kernel finds the pairs with x_s + x_d >= 2, accounts
// each at the first locus the two reads share, and records its overlap class:
//     x_s + x_d == 2  -> int32 planes H2[(2,0),(1,1),(0,2)]
//     x_s + x_d == 3  -> int32 planes H3[(3,0),(2,1),(1,2),(0,3)]
//     x_s + x_d >= 4  -> fp64 spill plane, += G(x_s, x_d) (rare; allocated on demand)
// plus a global class histogram. The epilogue then adds G(s,d) = F(s,d) - s F(1,0) - d F(0,1) per
// recorded pair, which together with F(1,0) S + F(0,1) D gives exactly sum_pairs F(x_s, x_d).
//
// Only entries of reads that keep >= 2 loci take part, and read linking (reads.cu) already lists
// them: they are among the "special" entries, numbered in entry order (hence grouped by locus). Each
// thread pairs one of them with the later ones of the same locus, merging the two reads' stored
// (locus, base) lists.
#include "common.cuh"

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <vector>

namespace {

constexpr int TB = 256;

struct MultiArgs {
    uint64_t n_special;       // upper bound of the number of candidates (launch size)
    const uint64_t *n_me;     // device: number of candidates
    const uint32_t *me_code;  // cell << 4 | base << 2 | tail << 1 | 1
    const uint32_t *me_locus;
    const uint32_t *me_pos;   // element of the read's stored list that belongs to this locus
    const uint32_t *me_beg;   // stored list [me_beg, me_end) in g_list / g_base
    const uint32_t *me_end;
    const uint32_t *g_list;   // stored loci, ascending
    const uint8_t *g_base;    // stored bases
    int32_t *H2;              // 3 planes
    int32_t *H3;              // 4 planes
    double *spill;            // may be null
    const double *G;          // device table SGPU_MAX_CLASS^2 (only read when spill != null)
    unsigned long long *hist; // SGPU_MAX_CLASS^2
    uint32_t n_cells;
    uint64_t nn;
    uint32_t L;
    uint32_t tbl_len;         // logprob_table_len(L): classes with x_s + x_d >= tbl_len have no log-likelihood
    int spill_only;           // second pass: record only the classes with x_s + x_d >= 4
    uint32_t min_order;       // 2: every multi-locus pair is enumerated here; 3: the pairs of order 2 come from
                              // the second-order GEMM, which counts every pair of order >= 3 C(x_s,2) / x_s x_d /
                              // C(x_d,2) times too much in the (2,0) / (1,1) / (0,2) planes: taken back here
    unsigned int *max_order;
    unsigned long long *n_pairs;
    int *err;
    const uint8_t *owned;     // ranged accumulation: a pair is recorded by the piece that owns its first common locus (null = all)
};

__global__ void __launch_bounds__(TB) multilocus_kernel(MultiArgs a) {
    // the class histogram has a handful of hot bins: count per block, flush once
    __shared__ uint32_t s_hist[SGPU_MAX_CLASS * SGPU_MAX_CLASS];
    __shared__ unsigned int s_max_order;
    const uint64_t ia = static_cast<uint64_t>(blockIdx.x) * TB + threadIdx.x;
    const uint64_t n_me = *a.n_me;
    if (static_cast<uint64_t>(blockIdx.x) * TB >= n_me) {
        return; // whole block behind the last candidate
    }
    for (uint32_t i = threadIdx.x; i < SGPU_MAX_CLASS * SGPU_MAX_CLASS; i += TB) {
        s_hist[i] = 0;
    }
    if (threadIdx.x == 0) {
        s_max_order = 0;
    }
    __syncthreads();
    unsigned long long local_pairs = 0;
    unsigned int local_max = 0;
    if (ia < n_me && (a.owned == nullptr || a.owned[a.me_locus[ia]])) {
        const uint32_t loc = a.me_locus[ia];
        const uint32_t ca = a.me_code[ia];
        const uint32_t a0 = a.me_beg[ia], ap = a.me_pos[ia], a1 = a.me_end[ia];
        for (uint64_t ib = ia + 1; ib < n_me; ++ib) {
            if (a.me_locus[ib] != loc) {
                break;
            }
            const uint32_t cb = a.me_code[ib];
            if (code_cell(ca) == code_cell(cb) || (ca & cb & 2u)) {
                continue; // same cell, or both reads behind the cutoff K
            }
            const uint32_t b0 = a.me_beg[ib], bp = a.me_pos[ib], b1 = a.me_end[ib];
            // two-pointer merge over the stored loci (similarity_matrix.cpp:221-229), the part behind this
            // locus first: most pairs share nothing there and are single-locus overlaps (first order)
            uint32_t xs = 0, xd = 0;
            for (uint32_t i = ap + 1, j = bp + 1; i < a1 && j < b1;) {
                const uint32_t la = a.g_list[i], lb = a.g_list[j];
                if (la == lb) {
                    a.g_base[i] == a.g_base[j] ? ++xs : ++xd;
                    ++i;
                    ++j;
                } else if (la < lb) {
                    ++i;
                } else {
                    ++j;
                }
            }
            if (xs + xd == 0) {
                continue;
            }
            bool earlier = false; // a common locus before this one: the pair is accounted there
            for (uint32_t i = a0, j = b0; i < ap && j < bp;) {
                const uint32_t la = a.g_list[i], lb = a.g_list[j];
                if (la == lb) {
                    earlier = true;
                    break;
                }
                la < lb ? ++i : ++j;
            }
            if (earlier) {
                continue;
            }
            a.g_base[ap] == a.g_base[bp] ? ++xs : ++xd; // this locus
            if (xs + xd < a.min_order) {
                continue;
            }
            if (xs >= SGPU_MAX_CLASS || xd >= SGPU_MAX_CLASS || xs >= a.L || xd >= a.L || xs + xd >= a.tbl_len) {
                atomicExch(a.err, SGPU_E_CLASS_RANGE);
                continue;
            }
            const uint32_t order = xs + xd;
            const uint32_t lo = min(code_cell(ca), code_cell(cb)), hi = max(code_cell(ca), code_cell(cb));
            const uint64_t ij = static_cast<uint64_t>(lo) * a.n_cells + hi;
            if (!a.spill_only) {
                ++local_pairs;
                if (a.min_order > 2) {
                    const int c20 = static_cast<int>(xs * (xs - 1) / 2), c11 = static_cast<int>(xs * xd), c02 = static_cast<int>(xd * (xd - 1) / 2);
                    if (c20) {
                        atomicAdd(&a.H2[0 * a.nn + ij], -c20);
                        atomicAdd(&a.hist[2 * SGPU_MAX_CLASS + 0], static_cast<unsigned long long>(-static_cast<long long>(c20)));
                    }
                    if (c11) {
                        atomicAdd(&a.H2[1 * a.nn + ij], -c11);
                        atomicAdd(&a.hist[1 * SGPU_MAX_CLASS + 1], static_cast<unsigned long long>(-static_cast<long long>(c11)));
                    }
                    if (c02) {
                        atomicAdd(&a.H2[2 * a.nn + ij], -c02);
                        atomicAdd(&a.hist[0 * SGPU_MAX_CLASS + 2], static_cast<unsigned long long>(-static_cast<long long>(c02)));
                    }
                }
                atomicAdd(&s_hist[xs * SGPU_MAX_CLASS + xd], 1u);
                if (order == 2) {
                    atomicAdd(&a.H2[static_cast<uint64_t>(xd) * a.nn + ij], 1);
                } else if (order == 3) {
                    atomicAdd(&a.H3[static_cast<uint64_t>(xd) * a.nn + ij], 1);
                }
                local_max = max(local_max, order);
            }
            if (order >= 4 && a.spill != nullptr) {
                atomicAdd(&a.spill[ij], a.G[xs * SGPU_MAX_CLASS + xd]);
            }
        }
    }
    if (local_max) {
        atomicMax(&s_max_order, local_max);
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < SGPU_MAX_CLASS * SGPU_MAX_CLASS; i += TB) {
        if (s_hist[i]) {
            atomicAdd(&a.hist[i], static_cast<unsigned long long>(s_hist[i]));
        }
    }
    if (threadIdx.x == 0 && s_max_order) {
        atomicMax(a.max_order, s_max_order);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        local_pairs += __shfl_xor_sync(0xffffffffu, local_pairs, o);
    }
    if ((threadIdx.x & 31) == 0 && local_pairs) {
        atomicAdd(a.n_pairs, local_pairs);
    }
}

// ------------------------------------------------------------------------------------------------
// Second order as a GEMM (SURVEY Appendix D.3). When many reads cover two loci (real data: ~16 % of the
// reads), enumerating the read pairs that share both costs one atomic per pair — hundreds of ms at
// 8 000 cells. The number of read pairs of cells (i, j) that cover a given PAIR of loci with a given base
// pattern is again a sum of outer products, so the first-order machinery (stripe partition, tile staging,
// tcgen05 GEMM) is reused on a derived pileup whose "loci" are locus pairs:
//   run A: 4 pseudo-loci per locus pair (l1, l2), one per base b1 at l1, holding the reads that cover both
//          with that b1, letter = base at l2:        same-letter count S_A = H20 (same at both loci),
//                                                    all-pairs count  T_A = P_s* (same at l1)
//   run B: 1 pseudo-locus per locus pair, letter = base at l2:  S_B = P_*s (same at l2), T_B = P_** (all)
// and with D = T - S of either run
//   N(2,0) += S_A        N(1,1) += D_A + S_B - S_A        N(0,2) += D_B - D_A.
// These are SUBSET counts (every pair of order >= 3 is seen at each of its locus pairs); the enumeration
// kernel, restricted to reads with >= 3 loci, records those pairs and takes the surplus back. Pairs of two
// tail reads are removed by the Z Z^T k-blocks of the GEMM path (pseudo-loci that hold only tail reads).
// ------------------------------------------------------------------------------------------------
struct PairArgs {
    uint64_t n_special;
    const uint32_t *sp_head;
    const uint32_t *sp_rcode; // per head: cell << 4 | tail << 1 | multi
    const uint64_t *g_off;
    const uint32_t *g_list;   // stored loci
    const uint8_t *g_base;
    const uint32_t *g_nst;
    const uint8_t *owned;     // ranged accumulation: the locus pair (l1, l2) belongs to the piece that owns l1 (null = all)
    unsigned long long *occ;  // per locus l1: bit d set = some read covers (l1, l1 + d + 1)
    const uint64_t *pair_base; // per locus: number of locus pairs before it (scan of popc(occ))
    uint64_t n_pairs;         // locus pairs
    // tail pairs: per chromosome the pair ids [z_first[c], z_first[c] + z_count[c]) get tail-only pseudo-loci z_off[c] ...
    const uint8_t *lchr;
    const uint64_t *z_first, *z_off;
    const uint32_t *z_count;
    uint64_t n_z;
    uint32_t *cntA, *cntB;     // entries per pseudo-locus
    const uint64_t *rowA, *rowB;
    uint32_t *gbA, *gbB;       // cell << 2 | letter
    int *err;
};

__device__ __forceinline__ bool pair_head(const PairArgs &a, uint64_t h) {
    return h < a.n_special && a.sp_head[h] == h && a.g_nst[h] >= 2;
}

__global__ void __launch_bounds__(TB) pair_occ_kernel(PairArgs a) {
    const uint64_t h = static_cast<uint64_t>(blockIdx.x) * TB + threadIdx.x;
    if (!pair_head(a, h)) {
        return;
    }
    const uint64_t o = a.g_off[h];
    const uint32_t n = a.g_nst[h];
    for (uint32_t p = 0; p + 1 < n; ++p) {
        if (a.owned && !a.owned[a.g_list[o + p]]) {
            continue;
        }
        for (uint32_t q = p + 1; q < n; ++q) {
            const uint32_t d = a.g_list[o + q] - a.g_list[o + p] - 1;
            if (d >= 64) {
                atomicExch(a.err, 1); // loci of one read more than 64 apart: the caller falls back to enumeration
                return;
            }
            atomicOr(&a.occ[a.g_list[o + p]], 1ull << d);
        }
    }
}

__global__ void __launch_bounds__(TB) pair_popc_kernel(const unsigned long long *__restrict__ occ, uint64_t n_loci,
                                                       uint32_t *__restrict__ pc) {
    const uint64_t l = static_cast<uint64_t>(blockIdx.x) * TB + threadIdx.x;
    if (l < n_loci) {
        pc[l] = __popcll(occ[l]);
    }
}

// FILL = false: count the entries of every pseudo-locus; FILL = true: write them
template <bool FILL>
__global__ void __launch_bounds__(TB) pair_emit_kernel(PairArgs a) {
    const uint64_t h = static_cast<uint64_t>(blockIdx.x) * TB + threadIdx.x;
    if (!pair_head(a, h) || a.g_nst[h] == 2) { // reads with two loci: pair_emit2_kernel
        return;
    }
    const uint64_t o = a.g_off[h];
    const uint32_t n = a.g_nst[h];
    const uint32_t rc = a.sp_rcode[h];
    const uint32_t cell = rc >> 4;
    const bool tail = (rc >> 1) & 1u;
    for (uint32_t p = 0; p + 1 < n; ++p) {
        const uint32_t l1 = a.g_list[o + p], b1 = a.g_base[o + p];
        if (a.owned && !a.owned[l1]) {
            continue;
        }
        const unsigned long long occ = a.occ[l1];
        for (uint32_t q = p + 1; q < n; ++q) {
            const uint32_t d = a.g_list[o + q] - l1 - 1, b2 = a.g_base[o + q];
            const uint64_t pid = a.pair_base[l1] + __popcll(occ & ((1ull << d) - 1ull));
            uint64_t plA[2] = { pid * 4 + b1, 0 }, plB[2] = { pid, 0 };
            int n_out = 1;
            if (tail) { // a tail read: all its loci lie behind the cutoff of its chromosome
                const uint32_t c = a.lchr[l1];
                const uint64_t z = a.z_off[c] + (pid - a.z_first[c]);
                plA[1] = a.n_pairs * 4 + z * 4 + b1;
                plB[1] = a.n_pairs + z;
                n_out = 2;
            }
            for (int k = 0; k < n_out; ++k) {
                const uint32_t ka = atomicAdd(&a.cntA[plA[k]], 1u), kb = atomicAdd(&a.cntB[plB[k]], 1u);
                if (FILL) {
                    a.gbA[a.rowA[plA[k]] + ka] = (cell << 2) | b2;
                    a.gbB[a.rowB[plB[k]] + kb] = (cell << 2) | b2;
                }
            }
        }
    }
}

// The same for the reads that keep exactly two loci (nearly all multi-locus reads): one thread per read,
// no loops, and the lanes of a warp that hit the same pseudo-locus (reads are ordered by first locus, so
// most of a warp does) share one atomic.
template <bool FILL>
__global__ void __launch_bounds__(TB) pair_emit2_kernel(PairArgs a) {
    const uint64_t h = static_cast<uint64_t>(blockIdx.x) * TB + threadIdx.x;
    const uint32_t lane = threadIdx.x & 31;
    const bool on = pair_head(a, h) && a.g_nst[h] == 2 && (a.owned == nullptr || a.owned[a.g_list[a.g_off[h]]]);
    uint64_t plA = ~0ull, plB = ~0ull, zA = ~0ull, zB = ~0ull;
    uint32_t val = 0;
    if (on) {
        const uint64_t o = a.g_off[h];
        const uint32_t rc = a.sp_rcode[h];
        const uint32_t l1 = a.g_list[o], b1 = a.g_base[o], d = a.g_list[o + 1] - l1 - 1, b2 = a.g_base[o + 1];
        const uint64_t pid = a.pair_base[l1] + __popcll(a.occ[l1] & ((1ull << d) - 1ull));
        plA = pid * 4 + b1;
        plB = pid;
        val = ((rc >> 4) << 2) | b2;
        if ((rc >> 1) & 1u) { // tail read
            const uint32_t c = a.lchr[l1];
            const uint64_t z = a.z_off[c] + (pid - a.z_first[c]);
            zA = a.n_pairs * 4 + z * 4 + b1;
            zB = a.n_pairs + z;
        }
    }
    // one aggregated atomic per distinct key in the warp; returns this lane's position
    auto reserve = [&](uint32_t *cnt, uint64_t key) -> uint32_t {
        const uint32_t m = __match_any_sync(0xffffffffu, key);
        const int leader = __ffs(m) - 1;
        uint32_t base = 0;
        if (key != ~0ull && static_cast<int>(lane) == leader) {
            base = atomicAdd(&cnt[key], static_cast<uint32_t>(__popc(m)));
        }
        base = __shfl_sync(0xffffffffu, base, leader);
        return base + __popc(m & ((1u << lane) - 1u));
    };
    const uint32_t ka = reserve(a.cntA, plA), kb = reserve(a.cntB, plB);
    const uint32_t kza = reserve(a.cntA, zA), kzb = reserve(a.cntB, zB);
    if (FILL && on) {
        a.gbA[a.rowA[plA] + ka] = val;
        a.gbB[a.rowB[plB] + kb] = val;
        if (zA != ~0ull) {
            a.gbA[a.rowA[zA] + kza] = val;
            a.gbB[a.rowB[zB] + kzb] = val;
        }
    }
}

// one of the two combinations above, elementwise over the upper triangle; sums of the increments per plane
// go to the class histogram (the classes of order 2 are not enumerated on this path)
__global__ void __launch_bounds__(TB) pair_combine_kernel(const int32_t *__restrict__ S, const int32_t *__restrict__ D,
                                                          int32_t *__restrict__ H2, uint32_t n, uint64_t nn, int run_b,
                                                          unsigned long long *__restrict__ hist) {
    const uint64_t idx = static_cast<uint64_t>(blockIdx.x) * TB + threadIdx.x;
    long long d20 = 0, d11 = 0, d02 = 0;
    if (idx < nn) {
        const uint32_t i = static_cast<uint32_t>(idx / n), j = static_cast<uint32_t>(idx - static_cast<uint64_t>(i) * n);
        if (i < j) {
            const int32_t s = S[idx], d = D[idx];
            if (!run_b) {
                d20 = s;
                d11 = d - s;
                d02 = -d;
            } else {
                d11 = s;
                d02 = d;
            }
            if (d20) {
                H2[0 * nn + idx] += static_cast<int32_t>(d20);
            }
            if (d11) {
                H2[1 * nn + idx] += static_cast<int32_t>(d11);
            }
            if (d02) {
                H2[2 * nn + idx] += static_cast<int32_t>(d02);
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        d20 += __shfl_xor_sync(0xffffffffu, d20, o);
        d11 += __shfl_xor_sync(0xffffffffu, d11, o);
        d02 += __shfl_xor_sync(0xffffffffu, d02, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (d20) {
            atomicAdd(&hist[2 * SGPU_MAX_CLASS + 0], static_cast<unsigned long long>(d20));
        }
        if (d11) {
            atomicAdd(&hist[1 * SGPU_MAX_CLASS + 1], static_cast<unsigned long long>(d11));
        }
        if (d02) {
            atomicAdd(&hist[0 * SGPU_MAX_CLASS + 2], static_cast<unsigned long long>(d02));
        }
    }
}

__global__ void __launch_bounds__(TB) iota_u32_kernel(uint32_t *__restrict__ a, uint32_t n, uint32_t first) {
    const uint32_t i = blockIdx.x * TB + threadIdx.x;
    if (i < n) {
        a[i] = first + i;
    }
}

unsigned blocks_for(uint64_t n) { return static_cast<unsigned>(ceil_div_u64(n ? n : 1, TB)); }

} // namespace

// second order through the GEMM path; returns 1 if the input does not fit the scheme (fall back to enumeration)
static int second_order_gemm(sgpu_ctx *ctx, const sgpu_pileup *p, LinkResult &lr, sgpu_counts *c, long long *class2_pairs) {
    cudaStream_t st = ctx->stream;
    const uint64_t NS = lr.n_special, P = p->n_loci, nn = c->nn;
    const uint32_t N = c->n, n_chr = p->n_chr;
    *class2_pairs = 0;
    DevBuf<unsigned long long> occ;
    DevBuf<uint32_t> pc;
    DevBuf<uint64_t> pair_base;
    DevBuf<int> d_err;
    SGPU_CUDA(ctx, occ.alloc(P, ctx));
    SGPU_CUDA(ctx, pc.alloc(P, ctx));
    SGPU_CUDA(ctx, pair_base.alloc(P + 1, ctx));
    SGPU_CUDA(ctx, d_err.alloc(1, ctx));
    SGPU_CUDA(ctx, cudaMemsetAsync(occ.p, 0, P * sizeof(unsigned long long), st));
    SGPU_CUDA(ctx, cudaMemsetAsync(d_err.p, 0, sizeof(int), st));
    PairArgs a;
    memset(&a, 0, sizeof(a));
    a.n_special = NS;
    a.sp_head = lr.sp_head.p;
    a.sp_rcode = lr.sp_rcode.p;
    a.g_off = lr.g_off.p;
    a.g_list = lr.g_list.p;
    a.g_base = lr.g_base.p;
    a.g_nst = lr.g_nst.p;
    a.owned = lr.ranged ? lr.owned.p : nullptr;
    a.occ = occ.p;
    a.lchr = lr.lchr.p;
    a.err = d_err.p;
    SGPU_TRACE(ctx, "pairs: enter");
    SGPU_LAUNCH(ctx, (pair_occ_kernel<<<blocks_for(NS), TB, 0, st>>>(a)));
    SGPU_LAUNCH(ctx, (pair_popc_kernel<<<blocks_for(P), TB, 0, st>>>(occ.p, P, pc.p)));
    SGPU_TRY(sgpu_scan_u32_u64(ctx, pc.p, pair_base.p, P));
    // locus pairs in total and in front of the cutoff locus / the end of every chromosome
    std::vector<uint64_t> h_first(n_chr), h_last(n_chr), h_zoff(n_chr + 1, 0);
    std::vector<uint32_t> h_zcnt(n_chr);
    SGPU_CUDA(ctx, cudaMemcpyAsync(&ctx->h_scratch[0], pair_base.p + P, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    SGPU_CUDA(ctx, cudaMemcpyAsync(&ctx->h_scratch[1], d_err.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    for (uint32_t ch = 0; ch < n_chr; ++ch) {
        SGPU_CUDA(ctx, cudaMemcpyAsync(&h_first[ch], pair_base.p + lr.h_tail_locus[ch], sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        SGPU_CUDA(ctx, cudaMemcpyAsync(&h_last[ch], pair_base.p + p->h_chr_ptr[ch + 1], sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    }
    SGPU_CUDA(ctx, cudaStreamSynchronize(st));
    if (static_cast<int>(ctx->h_scratch[1] & 0xFFFFFFFFu) != 0) {
        return 1;
    }
    SGPU_TRACE(ctx, "pairs: occupancy + numbering");
    const uint64_t NP = ctx->h_scratch[0];
    if (NP == 0) {
        return SGPU_OK;
    }
    for (uint32_t ch = 0; ch < n_chr; ++ch) {
        h_zcnt[ch] = static_cast<uint32_t>(h_last[ch] - h_first[ch]);
        h_zoff[ch + 1] = h_zoff[ch] + h_zcnt[ch];
    }
    const uint64_t NZ = h_zoff[n_chr];
    const uint64_t RA = 4 * (NP + NZ), RB = NP + NZ;
    if (RA >= 0x7FFFFFF0ull) {
        return 1;
    }
    DevBuf<uint64_t> z_first, z_off, rowA, rowB;
    DevBuf<uint32_t> z_count, cntA, cntB;
    SGPU_CUDA(ctx, z_first.alloc(n_chr, ctx));
    SGPU_CUDA(ctx, z_off.alloc(n_chr + 1, ctx));
    SGPU_CUDA(ctx, z_count.alloc(n_chr, ctx));
    SGPU_CUDA(ctx, cntA.alloc(RA, ctx));
    SGPU_CUDA(ctx, cntB.alloc(RB, ctx));
    SGPU_CUDA(ctx, rowA.alloc(RA + 1, ctx));
    SGPU_CUDA(ctx, rowB.alloc(RB + 1, ctx));
    SGPU_CUDA(ctx, cudaMemcpyAsync(z_first.p, h_first.data(), n_chr * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    SGPU_CUDA(ctx, cudaMemcpyAsync(z_off.p, h_zoff.data(), (n_chr + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    SGPU_CUDA(ctx, cudaMemcpyAsync(z_count.p, h_zcnt.data(), n_chr * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    SGPU_CUDA(ctx, cudaMemsetAsync(cntA.p, 0, RA * sizeof(uint32_t), st));
    SGPU_CUDA(ctx, cudaMemsetAsync(cntB.p, 0, RB * sizeof(uint32_t), st));
    a.pair_base = pair_base.p;
    a.n_pairs = NP;
    a.z_first = z_first.p;
    a.z_off = z_off.p;
    a.z_count = z_count.p;
    a.n_z = NZ;
    a.cntA = cntA.p;
    a.cntB = cntB.p;
    SGPU_LAUNCH(ctx, (pair_emit2_kernel<false><<<blocks_for(NS), TB, 0, st>>>(a)));
    SGPU_LAUNCH(ctx, (pair_emit_kernel<false><<<blocks_for(NS), TB, 0, st>>>(a)));
    SGPU_TRY(sgpu_scan_u32_u64(ctx, cntA.p, rowA.p, RA));
    SGPU_TRY(sgpu_scan_u32_u64(ctx, cntB.p, rowB.p, RB));
    SGPU_CUDA(ctx, cudaMemcpyAsync(&ctx->h_scratch[0], rowA.p + RA, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    SGPU_CUDA(ctx, cudaStreamSynchronize(st)); // also: the host vectors above have been copied
    SGPU_TRACE(ctx, "pairs: count entries");
    const uint64_t EA = ctx->h_scratch[0]; // = entries of run B as well
    if (EA >= 0x7FFFFFF0ull) {
        return 1;
    }
    DevBuf<uint32_t> gbA, gbB;
    DevBuf<uint32_t> zero_bits, zero_start, ident, tailA, tailB;
    DevBuf<int32_t> tmp;
    SGPU_CUDA(ctx, gbA.alloc(EA + 8, ctx));
    SGPU_CUDA(ctx, gbB.alloc(EA + 8, ctx));
    SGPU_CUDA(ctx, zero_bits.alloc(EA / 32 + 2, ctx));
    SGPU_CUDA(ctx, zero_start.alloc(RA + 2, ctx));
    SGPU_CUDA(ctx, ident.alloc(N, ctx));
    SGPU_CUDA(ctx, tailA.alloc(4 * NZ + 1, ctx));
    SGPU_CUDA(ctx, tailB.alloc(NZ + 1, ctx));
    SGPU_CUDA(ctx, tmp.alloc(2 * nn, ctx));
    SGPU_CUDA(ctx, cudaMemsetAsync(cntA.p, 0, RA * sizeof(uint32_t), st));
    SGPU_CUDA(ctx, cudaMemsetAsync(cntB.p, 0, RB * sizeof(uint32_t), st));
    SGPU_CUDA(ctx, cudaMemsetAsync(zero_bits.p, 0, (EA / 32 + 2) * sizeof(uint32_t), st));
    SGPU_CUDA(ctx, cudaMemsetAsync(zero_start.p, 0, (RA + 2) * sizeof(uint32_t), st));
    a.rowA = rowA.p;
    a.rowB = rowB.p;
    a.gbA = gbA.p;
    a.gbB = gbB.p;
    SGPU_LAUNCH(ctx, (pair_emit2_kernel<true><<<blocks_for(NS), TB, 0, st>>>(a)));
    SGPU_LAUNCH(ctx, (pair_emit_kernel<true><<<blocks_for(NS), TB, 0, st>>>(a)));
    SGPU_LAUNCH(ctx, (iota_u32_kernel<<<blocks_for(N), TB, 0, st>>>(ident.p, N, 0)));
    if (NZ) {
        SGPU_LAUNCH(ctx, (iota_u32_kernel<<<blocks_for(4 * NZ), TB, 0, st>>>(tailA.p, static_cast<uint32_t>(4 * NZ), static_cast<uint32_t>(4 * NP))));
        SGPU_LAUNCH(ctx, (iota_u32_kernel<<<blocks_for(NZ), TB, 0, st>>>(tailB.p, static_cast<uint32_t>(NZ), static_cast<uint32_t>(NP))));
    }
    SGPU_CUDA(ctx, cudaGetLastError());
    SGPU_TRACE(ctx, "pairs: fill");
    for (int run = 0; run < 2; ++run) {
        GemmInput in;
        in.row_ptr = run ? rowB.p : rowA.p;
        in.gid_base = nullptr;
        in.gid_base32 = run ? gbB.p : gbA.p;
        in.n_loci = run ? RB : RA;
        in.n_main = run ? NP : 4 * NP;
        in.main_loci = nullptr;
        in.n_entries = EA;
        in.sp_bits = zero_bits.p;
        in.gmap = ident.p;
        in.n_groups = N;
        in.sp_code = nullptr;
        in.sp_locus = nullptr;
        in.sp_start = zero_start.p;
        in.n_special = 0;
        in.tail_loci = run ? tailB.p : tailA.p;
        in.n_tail_loci = run ? NZ : 4 * NZ;
        SGPU_CUDA(ctx, cudaMemsetAsync(tmp.p, 0, 2 * nn * sizeof(int32_t), st));
        bool fresh = true;
        SGPU_TRY(sgpu_gemm_run(ctx, in, N, tmp.p, tmp.p + nn, &fresh));
        SGPU_LAUNCH(ctx, (pair_combine_kernel<<<blocks_for(nn), TB, 0, st>>>(tmp.p, tmp.p + nn, c->i32 + PLANE_H2 * nn, N, nn, run,
                                                                          reinterpret_cast<unsigned long long *>(c->hist))));
        SGPU_CUDA(ctx, cudaGetLastError());
    }
    SGPU_CUDA(ctx, cudaStreamSynchronize(st));
    SGPU_TRACE(ctx, "pairs: GEMM runs + combine");
    (void)class2_pairs;
    return SGPU_OK;
}

int sgpu_multilocus(sgpu_ctx *ctx, const sgpu_pileup *p, LinkResult &lr, sgpu_counts *c,
                    uint32_t L, uint64_t *n_pairs_multi) {
    cudaStream_t st = ctx->stream;
    if (n_pairs_multi) {
        *n_pairs_multi = 0;
    }
    if (lr.n_multi == 0 || p->n_entries == 0 || lr.n_special == 0) {
        return SGPU_OK;
    }
    const uint64_t NS = lr.n_special;
    // Pairs of order 2: enumeration costs m^2 / 2 atomics per locus (m multi-locus reads there; measured
    // 36 ps per pair), the second-order GEMM 5 pseudo-loci per locus pair whatever m is (measured 0.9 us per
    // locus pair at 8 192 padded cells, ~ N^2): the GEMM wins from m ~ 224 N_pad / 8192 reads per locus.
    // SECEDO_B200_SECOND_ORDER=gemm|enum overrides (tests).
    const char *env = getenv("SECEDO_B200_SECOND_ORDER");
    const double n_pad = (c->n + 255) / 256 * 256.0;
    bool use_gemm = env ? env[0] == 'g'
                        : (c->n >= 512 && static_cast<double>(lr.n_multi) > 224.0 * n_pad / 8192.0 * static_cast<double>(p->n_loci));
    if (logprob_table_len(L) <= 2) {
        use_gemm = false; // no class of order 2 has a log-likelihood: the enumeration must see (and refuse) every such pair
    }
    uint64_t hist2_before[3] = { 0, 0, 0 };
    if (use_gemm) {
        // the order-2 classes are not enumerated: their number is read off the class histogram afterwards
        const size_t off[3] = { 2 * SGPU_MAX_CLASS + 0, 1 * SGPU_MAX_CLASS + 1, 0 * SGPU_MAX_CLASS + 2 };
        for (int k = 0; k < 3; ++k) {
            SGPU_CUDA(ctx, cudaMemcpyAsync(&hist2_before[k], c->hist + off[k], sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        }
        SGPU_CUDA(ctx, cudaStreamSynchronize(st));
        long long unused = 0;
        const int rc = second_order_gemm(ctx, p, lr, c, &unused);
        if (rc == 1) {
            use_gemm = false; // loci of one read too far apart for the pair numbering
        } else if (rc != SGPU_OK) {
            return rc;
        } else {
            c->planes_used = std::max(c->planes_used, static_cast<int>(PLANE_H3));
            SGPU_TRY(sgpu_link_candidates(ctx, &lr, 3)); // only reads with >= 3 loci can form pairs of order >= 3
        }
    }
    DevBuf<unsigned long long> d_np;
    DevBuf<unsigned int> d_max;
    DevBuf<int> d_err;
    DevBuf<double> d_G;
    SGPU_CUDA(ctx, d_np.alloc(1, ctx));
    SGPU_CUDA(ctx, d_max.alloc(1, ctx));
    SGPU_CUDA(ctx, d_err.alloc(1, ctx));
    SGPU_CUDA(ctx, cudaMemsetAsync(d_np.p, 0, sizeof(unsigned long long), st));
    SGPU_CUDA(ctx, cudaMemsetAsync(d_max.p, 0, sizeof(unsigned int), st));
    SGPU_CUDA(ctx, cudaMemsetAsync(d_err.p, 0, sizeof(int), st));
    if (c->spill != nullptr) {
        SGPU_CUDA(ctx, d_G.alloc(SGPU_MAX_CLASS * SGPU_MAX_CLASS, ctx));
        SGPU_TRY(sgpu_build_gtable(ctx, c->eps, c->h, c->theta, c->L, SGPU_MAX_CLASS, d_G.p, nullptr));
    }
    MultiArgs a;
    a.n_special = NS;
    a.n_me = lr.me_idx.p + NS;
    a.me_code = lr.me_code.p;
    a.me_locus = lr.me_locus.p;
    a.me_pos = lr.me_pos.p;
    a.me_beg = lr.me_beg.p;
    a.me_end = lr.me_end.p;
    a.g_list = lr.g_list.p;
    a.g_base = lr.g_base.p;
    a.H2 = c->i32 + PLANE_H2 * c->nn;
    a.H3 = c->i32 + PLANE_H3 * c->nn;
    a.spill = c->spill;
    a.G = d_G.p;
    a.hist = reinterpret_cast<unsigned long long *>(c->hist);
    a.n_cells = c->n;
    a.nn = c->nn;
    a.L = L;
    a.tbl_len = logprob_table_len(L);
    a.spill_only = 0;
    a.min_order = use_gemm ? 3 : 2;
    a.max_order = d_max.p;
    a.n_pairs = d_np.p;
    a.err = d_err.p;
    a.owned = lr.ranged ? lr.owned.p : nullptr;
    SGPU_TRACE(ctx, "multi: before enumeration");
    SGPU_LAUNCH(ctx, (multilocus_kernel<<<blocks_for(NS), TB, 0, st>>>(a)));
    SGPU_CUDA(ctx, cudaGetLastError());
    SGPU_TRACE(ctx, "multi: enumeration");
    SGPU_CUDA(ctx, cudaMemcpyAsync(&ctx->h_scratch[0], d_np.p, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    SGPU_CUDA(ctx, cudaMemcpyAsync(&ctx->h_scratch[1], d_max.p, sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
    SGPU_CUDA(ctx, cudaMemcpyAsync(&ctx->h_scratch[2], d_err.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    SGPU_CUDA(ctx, cudaStreamSynchronize(st));
    if (static_cast<int>(ctx->h_scratch[2] & 0xFFFFFFFFu) != 0) {
        return sgpu_fail(ctx, SGPU_E_CLASS_RANGE,
                         "a read pair overlaps with x_s or x_d >= %d (or >= max_fragment_length), or x_s + x_d >= %u",
                         SGPU_MAX_CLASS, logprob_table_len(L));
    }
    if (n_pairs_multi) {
        *n_pairs_multi = ctx->h_scratch[0];
    }
    if (use_gemm) { // + the pairs of order 2 (GEMM counts minus what the enumeration took back)
        const size_t off[3] = { 2 * SGPU_MAX_CLASS + 0, 1 * SGPU_MAX_CLASS + 1, 0 * SGPU_MAX_CLASS + 2 };
        uint64_t after[3];
        for (int k = 0; k < 3; ++k) {
            SGPU_CUDA(ctx, cudaMemcpyAsync(&after[k], c->hist + off[k], sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        }
        SGPU_CUDA(ctx, cudaStreamSynchronize(st));
        if (n_pairs_multi) {
            for (int k = 0; k < 3; ++k) {
                *n_pairs_multi += after[k] - hist2_before[k];
            }
        }
    }
    const unsigned int max_order = static_cast<unsigned int>(ctx->h_scratch[1] & 0xFFFFFFFFu);
    // planes that can be non-zero from now on: (2,0) (1,1) (0,2), and (3,0) .. (0,3) once an overlap of
    // three loci was seen (zeroing, the multi-GPU reduction and the epilogue skip the others)
    if (max_order >= 2) {
        c->planes_used = std::max(c->planes_used, max_order >= 3 ? static_cast<int>(N_PLANES) : static_cast<int>(PLANE_H3));
    }
    if (max_order >= 4 && c->spill == nullptr) {
        // first pair of order >= 4 seen by this counts object: create the spill plane and record
        // just those classes in a second pass
        SGPU_CUDA(ctx, cudaMalloc(&c->spill, c->nn * sizeof(double)));
        SGPU_CUDA(ctx, cudaMemsetAsync(c->spill, 0, c->nn * sizeof(double), st));
        SGPU_CUDA(ctx, d_G.alloc(SGPU_MAX_CLASS * SGPU_MAX_CLASS, ctx));
        SGPU_TRY(sgpu_build_gtable(ctx, c->eps, c->h, c->theta, c->L, SGPU_MAX_CLASS, d_G.p, nullptr));
        a.spill = c->spill;
        a.G = d_G.p;
        a.spill_only = 1;
        SGPU_LAUNCH(ctx, (multilocus_kernel<<<blocks_for(NS), TB, 0, st>>>(a)));
        SGPU_CUDA(ctx, cudaGetLastError());
        SGPU_CUDA(ctx, cudaStreamSynchronize(st));
    }
    return SGPU_OK;
}
