// K3 — first-order read-pair counts as a dense int8 GEMM on the 5th-generation tensor cores.
//
// Per locus l and cell i let c_b(i) be the number of surviving reads of cell i showing base b.
// The reference's per-locus contributions are  S_ij = sum_b c_b(i) c_b(j)  (same base) and
// T_ij = c(i) c(j), c = sum_b c_b  (all pairs), D = T - S. With the 4x4 Hadamard matrix H
// (H H^T = 4 I, first row all ones) and u = H c:
//        u_0(i) u_0(j)                       = T_ij
//        u_1(i) u_1(j) + u_2 u_2 + u_3 u_3   = 4 S_ij - T_ij
// so ONE K-dimension of 4 int8 values per (cell, locus) feeds two int32 accumulators — 4 MMA
// K-slices per 32 loci instead of the 5 (four base planes + a total plane) of the direct form.
//
//   partition_kernel     per locus: (cell, base) of the entries that are the only entry of their read, with the
//                        group map and the bitmap of special entries applied, sorted by stripe of cells
//   stage_tile_kernel    per (k-block of 32 loci, stripe): base counts in a shared-memory tile -> Hadamard planes,
//                        written as finished K-major operand rows U[chunk][cell][k-block][plane][32 loci]
//                        (one 128-byte row per cell and k-block); tail k-blocks hold Z and -Z (S = C C^T - Z Z^T)
//   syrk2_kernel         persistent CTA pairs (cluster of 2, tcgen05 cta_group::2, 256 x 256 tiles): warp 0 of both
//                        CTAs = TMA producer (cp.async.bulk.tensor.3d, 128B swizzle, mbarrier ring of 5 stages),
//                        warp 1 of the leader = tcgen05.mma.kind::i8 issuer (M=256, N=256, K=32;
//                        accumulators Q = 4S - T and T in TMEM, 2 x 256 columns per CTA), warps 2-5 = epilogue
//                        (tcgen05.ld, S = (Q+T)/4, D = T - S, vector stores / load-add-store into the int32 planes,
//                        RED.ADD for edge and split tiles, upper triangle only); the pairs start the n-th tile
//                        together (wave counter) so that a wave shares its operand slabs through L2
// Only output tiles that intersect the upper triangle are computed; the K range of a panel is split across CTAs for
// the tiles that do not fill a whole round of the grid.
//
// Scheduling (sgpu_gemm_run, sgpu_tensor_flush / _poll / _join below): the tensor kernel of a first-order accumulation
// runs on the context's tensor stream, and its launch is held back until the NEXT batch's link_window kernel has been
// issued, so that it shares the SMs with that batch's special-entry chain, partition and staging (DESIGN.md 4).
#include "common.cuh"

#include <cuda.h>

#include <algorithm>
#include <cstdlib>
#include <type_traits>
#include <vector>

namespace {

constexpr int BM = 128;            // rows (cells) of an output tile held by one CTA of a pair
constexpr int BN = 256;            // columns (cells) of an output tile = UMMA N
constexpr int KB_BYTES = 128;      // bytes of K per stage and row: 32 loci x 4 planes
constexpr int LOCI_PER_KB = 32;
constexpr int A_BYTES = BM * KB_BYTES;  // 16 KB
constexpr int GEMM_THREADS = 192;  // 6 warps
constexpr uint32_t TMEM_COLS = 512;

// Panel layout. One 128-byte row per (cell, k-block of 32 loci). The rows of CK consecutive k-blocks
// form a chunk [chunk][cell][k-block in chunk]: the ~1 200 loci that are staged concurrently then touch
// a few tens of MB of address space (2 MB pages: a handful of TLB entries) instead of one row in each of
// the 8 192 cell stripes of a [cell][K] matrix, 128 KB apart, which made the staging atomics TLB bound.
// The GEMM reads the same buffer through a 3-D tensor map (bytes in chunk row, cell, chunk).
struct PanelLayout {
    uint32_t ck_shift;    // log2(k-blocks per chunk)
    uint32_t cell_words;  // 32-bit words between consecutive cells of a chunk: an odd number of 128-byte lines
    uint64_t chunk_words; // words per chunk = n_pad * cell_words
    __host__ __device__ uint64_t row(uint32_t cell, uint32_t kb) const { // first word of the row (cell, kb)
        const uint32_t ch = kb >> ck_shift, kbi = kb - (ch << ck_shift);
        return ch * chunk_words + static_cast<uint64_t>(cell) * cell_words + kbi * 32u;
    }
    __host__ __device__ uint64_t word(uint32_t cell, uint32_t col) const { // staged counts of (cell, locus col)
        return row(cell, col >> 5) + (col & 31u);
    }
};

// ------------------------------------------------------------------------------------------------
// staging
//
// One CTA per (k-block of 32 loci, stripe of cells) accumulates the per-(cell, locus) base counts of
// its loci in a shared-memory tile (one word = 4 x u8 base counts, shared-memory atomics), turns the
// tile into Hadamard planes and writes the finished 128-byte operand rows [plane 0..3][32 loci] once,
// coalesced. Every stripe's CTA scans all entries of the 32 loci and keeps the cells of its stripe; the
// repeated reads come from L2. Nothing is zeroed, atomically updated or re-read in HBM: counting in
// global memory was bound by TLB reach and DRAM row activations (one 32-byte sector per atomic, each in
// a different page), not by bytes.
//
// The reference never compares two reads that both lie behind the per-chromosome cutoff K (SURVEY
// F2). Those pairs only exist at the few loci behind the cutoff; they are removed by extra k-blocks at
// the end of the panel that hold ONLY the tail reads, Z as the A operand and -Z as the B operand of
// the same GEMM:  S = C C^T - Z Z^T.
// ------------------------------------------------------------------------------------------------
constexpr int ST_THREADS = 512;
constexpr uint32_t ST_MAX_CELLS = 424;  // 53 KB tile: four CTAs per SM hide each other's phases
constexpr uint32_t ST_MAX_STRIPES = 63;
constexpr uint32_t CB_SKIP = 0xFFFFu;   // cellbase of an entry the dense scan does not count

// cellbase = (cell << 2 | base) of every entry that is the only entry of its read, with the group map and
// the bitmap of special entries applied, and PARTITIONED BY CELL STRIPE inside every locus:
// seg[l * (n_stripes + 1) + s] = first entry (relative to the locus) of stripe s, [.. + n_stripes] = end of
// the last stripe (the special entries, staged from their own list, are left out). A staging CTA then reads
// exactly the entries of its stripe. One CTA per locus: count per stripe, scan, scatter (order inside a
// stripe does not matter).
template <typename GB>
struct PartitionArgs {
    const uint64_t *row_ptr;
    const GB *gid_base;
    const uint32_t *sp_bits;
    const uint32_t *gmap;
    uint32_t n_groups, n_cells;
    uint32_t identity;     // group g is cell g: no table in shared memory (16 KB less per CTA at 8 000 cells: more CTAs per SM,
                           // above all beside the tensor kernel of the previous batch)
    uint64_t n_loci;
    uint32_t n_stripes;
    uint32_t stripe_magic; // cell / cells_per_cta = (cell * magic) >> 32, exact for cells < 65 536
    uint32_t cells_per_cta;
    uint16_t *cellbase;    // (cell - first cell of its stripe) << 2 | base: fits 16 bits for any number of cells
    uint32_t *seg;
    int *err;
};

constexpr uint32_t PART_OUT = 3 * 2048 + 8;               // shared-memory elements of the assembled locus
constexpr int PART_ROUNDS = 3;                            // rounds of 256 threads x 8 entries
constexpr uint32_t PART_CACHE = PART_ROUNDS * 2048 - 8;  // entries of a locus handled in registers + shared memory

// Gathers from the group map and scattered 2-byte stores cost one L1 wavefront per lane when they go to
// global memory; both are done in shared memory here (the map is copied once per CTA, the partitioned
// locus is assembled in shared memory and written out contiguously).
template <typename GB>
__global__ void __launch_bounds__(256) partition_kernel(const PartitionArgs<GB> a) {
    constexpr int PER_VEC = 16 / sizeof(GB); // entries per 16-byte load: 8 (two loads of 4 for wide entries)
    extern __shared__ __align__(16) uint16_t s_dyn[];
    __shared__ uint32_t s_cnt[ST_MAX_STRIPES + 1]; // entries of the stripe seen so far / start of the stripe
    uint16_t *s_out = s_dyn;                       // [PART_OUT] the partitioned locus
    uint16_t *s_map = s_dyn + PART_OUT;            // [n_groups] cell of the group, 0xFFFF = outside the matrix
    const uint32_t ns = a.n_stripes;
    if (!a.identity) {
        for (uint32_t g = threadIdx.x; g < a.n_groups; g += 256) {
            const uint32_t c = a.gmap[g];
            s_map[g] = static_cast<uint16_t>(c < a.n_cells ? c : 0xFFFFu);
        }
    }
    __syncthreads();
    auto cell_of = [&](uint32_t gid) -> uint32_t { return a.identity ? gid : s_map[gid]; }; // gid < n_groups (<= n_cells if identity)
    // stripe << 16 | value of entry e (value = cell inside its stripe << 2 | base); 0xFFFFFFFF = left out
    auto classify = [&](uint64_t e) -> uint32_t {
        uint32_t v = 0xFFFFFFFFu;
        const uint32_t gb = a.gid_base[e];
        if (!((a.sp_bits[e >> 5] >> (e & 31)) & 1u)) {
            const uint32_t gid = gb >> 2;
            uint32_t cell;
            if (gid >= a.n_groups || (cell = cell_of(gid)) == 0xFFFFu) {
                atomicExch(a.err, SGPU_E_CELL_RANGE);
            } else {
                const uint32_t stripe = __umulhi(cell, a.stripe_magic);
                v = (stripe << 16) | ((cell - stripe * a.cells_per_cta) << 2) | (gb & 3u);
            }
        }
        return v;
    };
    for (uint64_t l = blockIdx.x; l < a.n_loci; l += gridDim.x) {
        const uint64_t e0 = a.row_ptr[l];
        const uint32_t n = static_cast<uint32_t>(a.row_ptr[l + 1] - e0);
        uint32_t *sg = a.seg + l * (ns + 1);
        if (n <= PART_CACHE) {
            // one sweep: the shared-memory atomic that counts the stripe also ranks the entry inside it
            // (~20 stripes: the lanes of a warp spread over them, few same-address conflicts). Values and ranks stay
            // in registers between the sweep and the scatter (every thread meets the same entries in both).
            if (threadIdx.x <= ns) {
                s_cnt[threadIdx.x] = 0;
            }
            __syncthreads();
            // eight consecutive entries per thread and round: one 16-byte load and one byte of the bitmap (an aligned
            // window covers the locus; entries outside it are masked)
            const uint64_t e1 = e0 + n, base = e0 & ~7ull;
            const bool vec_ok = (reinterpret_cast<uintptr_t>(a.gid_base) & 15u) == 0;
            uint32_t vr[PART_ROUNDS][8]; // stripe << 24 | value << 13 | rank inside the stripe; 0xFFFFFFFF = left out
#pragma unroll
            for (int it = 0; it < PART_ROUNDS; ++it) {
                const uint64_t v0 = base + 8ull * threadIdx.x + static_cast<uint64_t>(it) * (8 * 256);
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    vr[it][k] = 0xFFFFFFFFu;
                }
                if (v0 < e1) {
                    __align__(16) GB gb[8];
                    if (vec_ok && v0 >= e0 && v0 + 8 <= e1) {
#pragma unroll
                        for (int q = 0; q < 8 / PER_VEC; ++q) {
                            reinterpret_cast<uint4 *>(gb)[q] = reinterpret_cast<const uint4 *>(a.gid_base + v0)[q];
                        }
                    } else {
#pragma unroll
                        for (int k = 0; k < 8; ++k) {
                            gb[k] = (v0 + k >= e0 && v0 + k < e1) ? a.gid_base[v0 + k] : 0;
                        }
                    }
                    const uint32_t special = (a.sp_bits[v0 >> 5] >> (v0 & 31)) & 0xFFu;
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        const uint64_t e = v0 + k;
                        if (e < e0 || e >= e1 || ((special >> k) & 1u)) {
                            continue;
                        }
                        const uint32_t gid = gb[k] >> 2;
                        uint32_t cell;
                        if (gid >= a.n_groups || (cell = cell_of(gid)) == 0xFFFFu) {
                            atomicExch(a.err, SGPU_E_CELL_RANGE);
                        } else {
                            const uint32_t stripe = __umulhi(cell, a.stripe_magic);
                            const uint32_t v = ((cell - stripe * a.cells_per_cta) << 2) | (gb[k] & 3u);
                            vr[it][k] = (stripe << 24) | (v << 13) | atomicAdd(&s_cnt[stripe], 1u);
                        }
                    }
                }
            }
            __syncthreads();
            if (threadIdx.x < 32) { // exclusive scan over the stripes (<= 63): s_cnt[s] becomes the start of stripe s
                uint32_t c0 = threadIdx.x < ns ? s_cnt[threadIdx.x] : 0, c1 = threadIdx.x + 32 < ns ? s_cnt[threadIdx.x + 32] : 0;
                uint32_t i0 = c0, i1 = c1;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t t0 = __shfl_up_sync(0xffffffffu, i0, o), t1 = __shfl_up_sync(0xffffffffu, i1, o);
                    if (static_cast<int>(threadIdx.x) >= o) {
                        i0 += t0;
                        i1 += t1;
                    }
                }
                const uint32_t total0 = __shfl_sync(0xffffffffu, i0, 31);
                i1 += total0;
                if (threadIdx.x < ns) {
                    s_cnt[threadIdx.x] = i0 - c0;
                    sg[threadIdx.x] = i0 - c0;
                }
                if (threadIdx.x + 32 < ns) {
                    s_cnt[threadIdx.x + 32] = i1 - c1;
                    sg[threadIdx.x + 32] = i1 - c1;
                }
                if (threadIdx.x == 31) {
                    sg[ns] = i1; // end of the last stripe
                    s_cnt[ns] = i1;
                }
            }
            __syncthreads();
            // the partitioned locus is assembled in shared memory at the offset (e0 mod 8), so that its 16-byte chunks
            // line up with those of the output array
            const uint32_t shift = static_cast<uint32_t>(e0 & 7u);
#pragma unroll
            for (int it = 0; it < PART_ROUNDS; ++it) {
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const uint32_t x = vr[it][k];
                    if (x != 0xFFFFFFFFu) {
                        s_out[shift + s_cnt[x >> 24] + (x & 0x1FFFu)] = static_cast<uint16_t>((x >> 13) & 0x7FFu);
                    }
                }
            }
            __syncthreads();
            const uint32_t n_out = s_cnt[ns];
            const bool out_vec = (reinterpret_cast<uintptr_t>(a.cellbase) & 15u) == 0;
            // [shift, shift + n_out) of s_out -> cellbase[e0 ...]: whole 16-byte chunks where they are complete
            const uint32_t c_lo = out_vec ? (shift + 7) / 8 : 0, c_hi = out_vec ? (shift + n_out) / 8 : 0; // chunks [c_lo, c_hi)
            if (c_hi > c_lo) {
                for (uint32_t i = shift + threadIdx.x; i < c_lo * 8; i += 256) {
                    a.cellbase[base + i] = s_out[i];
                }
                uint4 *dst = reinterpret_cast<uint4 *>(a.cellbase + base);
                const uint4 *src = reinterpret_cast<const uint4 *>(s_out);
                for (uint32_t c = c_lo + threadIdx.x; c < c_hi; c += 256) {
                    dst[c] = src[c];
                }
                for (uint32_t i = c_hi * 8 + threadIdx.x; i < shift + n_out; i += 256) {
                    a.cellbase[base + i] = s_out[i];
                }
            } else {
                for (uint32_t i = shift + threadIdx.x; i < shift + n_out; i += 256) {
                    a.cellbase[base + i] = s_out[i];
                }
            }
            __syncthreads();
        } else {
            // a locus too large for the shared-memory round: count, scan, then rank with global re-reads
            if (threadIdx.x <= ns) {
                s_cnt[threadIdx.x] = 0;
            }
            __syncthreads();
            for (uint32_t i = threadIdx.x; i < n; i += 256) {
                const uint32_t v = classify(e0 + i);
                if (v != 0xFFFFFFFFu) {
                    atomicAdd(&s_cnt[v >> 16], 1u);
                }
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                uint32_t acc = 0;
                for (uint32_t s = 0; s < ns; ++s) {
                    const uint32_t c = s_cnt[s];
                    sg[s] = acc;
                    s_cnt[s] = acc;
                    acc += c;
                }
                sg[ns] = acc;
            }
            __syncthreads();
            for (uint32_t i = threadIdx.x; i < n; i += 256) {
                const uint32_t v = classify(e0 + i);
                if (v != 0xFFFFFFFFu) {
                    a.cellbase[e0 + atomicAdd(&s_cnt[v >> 16], 1u)] = static_cast<uint16_t>(v & 0xFFFFu);
                }
            }
            __syncthreads();
        }
    }
}

struct StageArgs {
    const uint64_t *row_ptr;
    const uint16_t *cellbase;  // see partition_kernel
    const uint32_t *seg;
    const uint32_t *sp_code;   // special entries, ascending by entry (hence by locus)
    const uint32_t *sp_locus;
    const uint32_t *sp_start;  // per locus: first special entry of the locus (n_loci + 1 values)
    uint32_t n_pad;
    uint32_t l0, nl;           // main k-blocks: loci [l0, l0 + nl) (of main_loci, if given), 32 per k-block
    const uint32_t *main_loci; // ranged accumulation: the owned loci (ascending), or null = all loci
    uint32_t kbs_main;
    const uint32_t *tail_loci; // tail k-blocks: loci tail_loci[0 .. n_tail), ascending
    uint32_t n_tail, kbs_tail; // Z goes to k-block kbs_main + t, -Z to kbs_main + kbs_tail + t
    uint32_t cells_per_cta, n_stripes;
    PanelLayout pl;
    uint32_t *U;
    int *err;
};

// dot product of four unsigned bytes with four signed bytes
__device__ __forceinline__ int dp4a_us(uint32_t a, int b) {
    int d;
    asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(0));
    return d;
}

// One count. Range check without looking at the old value: the CTA compares the number of counts it
// added with the sum of the tile's bytes afterwards (a byte that wrapped past 255 loses 255 or 256),
// and a byte above 127 is seen when the planes are built.
__device__ __forceinline__ void tile_add(uint32_t *tile, uint32_t r, uint32_t j, uint32_t base) {
    atomicAdd(&tile[r * 32 + ((j + r) & 31u)], 1u << (8u * base));
}

__global__ void __launch_bounds__(ST_THREADS, 4) stage_tile_kernel(const StageArgs a) {
    extern __shared__ uint32_t tile[]; // [cell in stripe][32 loci], word of locus j of row r at (j + r) % 32
    __shared__ uint64_t s_e0[32], s_e1[32];
    __shared__ uint32_t s_loc[32];
    __shared__ int s_balance;     // counts added - counts found in the tile
    __shared__ uint32_t s_sp0[32], s_sp1[32];
    // the stripes of one k-block are neighbours in the grid: they run together and share its entries in L2
    const uint32_t kb = blockIdx.x / a.n_stripes;
    const uint32_t stripe = blockIdx.x - kb * a.n_stripes;
    const uint32_t c0 = stripe * a.cells_per_cta;
    const uint32_t nc = min(a.cells_per_cta, a.n_pad - c0);
    const bool tail = kb >= a.kbs_main;
    if (threadIdx.x < 32) {
        const uint32_t j = threadIdx.x;
        uint32_t l = 0xFFFFFFFFu;
        if (!tail) {
            const uint32_t col = kb * LOCI_PER_KB + j;
            if (col < a.nl) {
                l = a.main_loci ? a.main_loci[a.l0 + col] : a.l0 + col;
            }
        } else {
            const uint32_t t = (kb - a.kbs_main) * LOCI_PER_KB + j;
            if (t < a.n_tail) {
                l = a.tail_loci[t];
            }
        }
        s_loc[j] = l;
        // this stripe's segment of the locus
        uint64_t b0 = 0, b1 = 0;
        if (l != 0xFFFFFFFFu) {
            const uint64_t e0 = a.row_ptr[l];
            const uint32_t *sg = a.seg + static_cast<uint64_t>(l) * (a.n_stripes + 1) + stripe;
            b0 = e0 + sg[0];
            b1 = e0 + sg[1];
        }
        s_e0[j] = b0;
        s_e1[j] = b1;
        if (j == 0) {
            s_balance = 0;
        }
        // the special entries of locus l: a contiguous range of the (ascending) list
        s_sp0[j] = l != 0xFFFFFFFFu ? a.sp_start[l] : 0;
        s_sp1[j] = l != 0xFFFFFFFFu ? a.sp_start[l + 1] : 0;
    }
    for (uint32_t i = threadIdx.x; i < nc * 32; i += ST_THREADS) {
        tile[i] = 0;
    }
    __syncthreads();

    // ---- entries that are the only entry of their read (in a tail k-block all of them are tail reads:
    // such a read was created at its own locus, which lies behind the cutoff). Warp j takes locus j.
    uint32_t n_added = 0;
    for (uint32_t j = threadIdx.x >> 5; j < 32; j += ST_THREADS / 32) {
        const uint32_t lane = threadIdx.x & 31;
        const uint64_t b1 = s_e1[j];
        for (uint64_t eb = s_e0[j] + lane; eb < b1; eb += 256) {
            uint32_t cb[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) { // eight loads in flight: a whole locus segment in one round
                cb[u] = eb + 32 * u < b1 ? a.cellbase[eb + 32 * u] : CB_SKIP;
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const uint32_t r = cb[u] >> 2; // cell inside this stripe
                if (cb[u] != CB_SKIP && r < nc) {
                    tile_add(tile, r, j, cb[u] & 3u);
                    ++n_added;
                }
            }
        }
    }
    // ---- surviving entries of reads with several entries
    if (!tail) {
        // consecutive loci: their special entries are one contiguous range of the (ascending) list
        const uint32_t l_first = s_loc[0];
        const uint32_t n_valid = l_first != 0xFFFFFFFFu ? min(32u, a.nl - kb * LOCI_PER_KB) : 0;
        if (n_valid && s_loc[n_valid - 1] - l_first != n_valid - 1) {
            // a list of owned loci with a gap inside this k-block (the border between two chromosomes' ranges): locus by locus
            for (uint32_t j = 0; j < n_valid; ++j) {
                for (uint32_t s = s_sp0[j] + threadIdx.x; s < s_sp1[j]; s += ST_THREADS) {
                    const uint32_t c = a.sp_code[s];
                    const uint32_t r = code_cell(c) - c0;
                    if (c != CODE_DROPPED && r < nc) {
                        tile_add(tile, r, j, code_base(c));
                        ++n_added;
                    }
                }
            }
        } else if (n_valid) {
            const uint32_t sp1 = s_sp1[n_valid - 1];
            for (uint32_t s = s_sp0[0] + threadIdx.x; s < sp1; s += ST_THREADS) {
                const uint32_t c = a.sp_code[s];
                const uint32_t r = code_cell(c) - c0;
                if (c != CODE_DROPPED && r < nc) {
                    tile_add(tile, r, a.sp_locus[s] - l_first, code_base(c));
                    ++n_added;
                }
            }
        }
    } else {
        for (uint32_t j = 0; j < 32; ++j) {
            for (uint32_t s = s_sp0[j] + threadIdx.x; s < s_sp1[j]; s += ST_THREADS) {
                const uint32_t c = a.sp_code[s];
                if (c == CODE_DROPPED || !code_tail(c)) {
                    continue;
                }
                const uint32_t r = code_cell(c) - c0;
                if (r < nc) {
                    tile_add(tile, r, j, code_base(c));
                    ++n_added;
                }
            }
        }
    }
    __syncthreads();

    // ---- Hadamard planes, written as finished operand rows: 8 consecutive lanes own one 128-byte row
    const uint32_t kb_neg = kb + a.kbs_tail;
    bool bad = false;
    int balance = static_cast<int>(n_added);
    for (uint32_t item = threadIdx.x; item < nc * 8; item += ST_THREADS) {
        const uint32_t r = item >> 3, g = item & 7;
        // u_p = H_p . (counts of the four bases), one dp4a per plane and locus; H rows as signed bytes
        uint32_t w[4], wn[4]; // per plane, 4 loci packed (and negated)
        int u[4][4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const uint32_t v = tile[r * 32 + ((4 * g + q + r) & 31u)];
            u[0][q] = dp4a_us(v, 0x01010101);
            u[1][q] = dp4a_us(v, static_cast<int>(0xFF01FF01u)); // + - + -
            u[2][q] = dp4a_us(v, static_cast<int>(0xFFFF0101u)); // + + - -
            u[3][q] = dp4a_us(v, static_cast<int>(0x01FFFF01u)); // + - - +
            balance -= u[0][q];
        }
        bad |= ((u[0][0] | u[0][1] | u[0][2] | u[0][3]) & ~127) != 0;
#pragma unroll
        for (int p = 0; p < 4; ++p) {
            w[p] = __byte_perm(__byte_perm(u[p][0], u[p][1], 0x0040), __byte_perm(u[p][2], u[p][3], 0x0040), 0x5410);
        }
        if (tail) {
#pragma unroll
            for (int p = 0; p < 4; ++p) {
                wn[p] = __byte_perm(__byte_perm(-u[p][0], -u[p][1], 0x0040), __byte_perm(-u[p][2], -u[p][3], 0x0040), 0x5410);
            }
        }
        uint32_t *out = a.U + a.pl.row(c0 + r, kb);
#pragma unroll
        for (int p = 0; p < 4; ++p) {
            out[p * 8 + g] = w[p];
        }
        if (tail) {
            uint32_t *outn = a.U + a.pl.row(c0 + r, kb_neg);
#pragma unroll
            for (int p = 0; p < 4; ++p) {
                outn[p * 8 + g] = wn[p];
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        balance += __shfl_xor_sync(0xffffffffu, balance, o);
    }
    if ((threadIdx.x & 31) == 0 && balance) {
        atomicAdd(&s_balance, balance);
    }
    __syncthreads();
    // > 127 reads of one cell at one locus: outside int8 (a wrapped byte leaves the balance positive)
    if (bad || (threadIdx.x == 0 && s_balance != 0)) {
        atomicExch(a.err, SGPU_E_COUNT_RANGE);
    }
}

// ------------------------------------------------------------------------------------------------
// PTX helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "WAIT_LOOP:\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
            "@p bra WAIT_DONE;\n\t"
            "bra WAIT_LOOP;\n\t"
            "WAIT_DONE:\n\t"
            "}" ::"r"(bar),
            "r"(parity)
            : "memory");
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
            "{\n\t"
            ".reg .pred P;\n\t"
            "elect.sync _|P, 0xffffffff;\n\t"
            "selp.b32 %0, 1, 0, P;\n\t"
            "}"
            : "=r"(pred));
    return pred != 0;
}
// UMMA shared-memory descriptor: K-major, 128B swizzle, 8-row groups 1024 B apart (SBO), LBO = 1
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);      // start address, bits [0,14)
    d |= static_cast<uint64_t>(1) << 16;                      // leading byte offset (unused for SW128 K-major)
    d |= static_cast<uint64_t>(1024 >> 4) << 32;              // stride byte offset
    d |= static_cast<uint64_t>(1) << 46;                      // descriptor version (Blackwell)
    d |= static_cast<uint64_t>(2) << 61;                      // SWIZZLE_128B
    return d;
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
            "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
            : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
              "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
              "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
              "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
            : "r"(taddr));
}

struct WorkItem {
    uint32_t rb, cb;   // row block (x256), column block (x256)
    uint32_t k0, k1;   // k-block range
    uint32_t partial;  // 1: the tile's K range is shared with other CTAs -> atomics only
};

// Work list of one launch: the first n_full items are whole tiles (all k-blocks), n_full a multiple of
// the number of pairs so that every pair owns the same number of them; the remaining tiles are cut into `splits`
// K ranges each, so that the last round keeps every SM busy for 1/splits of a tile instead of leaving
// most of them idle for a whole tile (528 tiles on 74 pairs = 7.13 rounds).
struct WorkList {
    const uint2 *tiles; // (row block, column block), rasterised for L2 reuse
    uint32_t n_full;    // tiles processed whole
    uint32_t n_work;    // n_full + (n_tiles - n_full) * splits
    uint32_t splits;    // K ranges per remaining tile (>= 1)
    uint32_t kbs;       // k-blocks of the panel (main + tail)
    uint32_t per;       // k-blocks per K range of a remaining tile
    uint32_t ck_shift;  // log2(k-blocks per chunk of the panel layout)
    uint32_t kb_neg0;   // k-blocks >= kb_neg0 hold tail reads only: their B operand is k-block kb + kb_negd (-Z)
    uint32_t kb_negd;
    unsigned int *wave_ctr; // pairs that have issued all loads of their n-th work item
};
__device__ __forceinline__ WorkItem work_item(const WorkList &wl, uint32_t w) {
    if (w < wl.n_full) {
        const uint2 t = wl.tiles[w];
        return WorkItem{ t.x, t.y, 0u, wl.kbs, 0u };
    }
    const uint32_t j = w - wl.n_full;
    const uint32_t tile = j / wl.splits, split = j - tile * wl.splits;
    const uint2 t = wl.tiles[wl.n_full + tile];
    const uint32_t k0 = split * wl.per;
    return WorkItem{ t.x, t.y, k0, min(wl.kbs, k0 + wl.per), wl.splits > 1 ? 1u : 0u };
}

// how whole tiles reach the count planes
enum : int {
    EPI_RED = 0,   // atomics, zeros skipped
    EPI_STORE = 1, // the planes are known to be zero: plain vector stores
    EPI_RMW = 2    // vector load + add + store (the tile is owned by one CTA)
};

// ------------------------------------------------------------------------------------------------
// the GEMM on CTA pairs (tcgen05 cta_group::2): a cluster of two CTAs owns a 256 x 256 output tile,
// each CTA 128 of its rows (its own TMEM) and HALF of the B operand (128 of the 256 columns' rows), which
// the tensor cores of both SMs read across the pair. Per CTA and k-block that is 32 KB of operands
// instead of the 48 KB of a single CTA with a 128 x 256 tile (a deeper ring, a third less L2->SM traffic
// and shared-memory bandwidth). Only the leader CTA issues MMAs; both CTAs' TMA loads report to the leader's
// barrier; the leader's commits release the stage / publish the accumulators in both CTAs (multicast).
// ------------------------------------------------------------------------------------------------
constexpr int HALF_B_BYTES = 128 * KB_BYTES;             // 16 KB
constexpr int STAGE_BYTES = A_BYTES + HALF_B_BYTES;      // 32 KB per CTA
// 5 stages (161 KB) leave shared memory to the staging kernels of the next batch that run beside the deferred kernel
// (sgpu_ctx::tensor_jobs); 4 are slower. With the SM to itself (SECEDO_B200_ASYNC_GEMM=0) 6 stages (193 KB) would be
// 2-3 % faster per launch (DESIGN.md 4, K3)
constexpr int STAGES = 5;
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /* alignment slack */ + 256 /* barriers */;
constexpr uint32_t IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((256u >> 3) << 17) | ((256u >> 4) << 24); // M = 256, N = 256

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) { // same offset in CTA `rank` of the cluster
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_remote(uint32_t cluster_addr, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cluster.b64 _, [%0], %1;" ::"r"(cluster_addr), "r"(bytes)
                 : "memory");
}
// TMA load of one CTA of a pair; the completion is reported to a barrier of the LEADER CTA
__device__ __forceinline__ void tma_load_3d_2sm(uint32_t dst, const CUtensorMap *map, uint32_t leader_bar, int32_t c0, int32_t c1,
                                                int32_t c2) {
    asm volatile(
            "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
            "l"(map), "r"(leader_bar), "r"(c0), "r"(c1), "r"(c2)
            : "memory");
}
__device__ __forceinline__ void umma_i8_2sm(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t accumulate) {
    asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t"
            "}" ::"r"(d_tmem),
            "l"(a_desc), "l"(b_desc), "r"(IDESC), "r"(accumulate)
            : "memory");
}
__device__ __forceinline__ void umma_commit_2sm(uint32_t bar) { // arrives on `bar` in BOTH CTAs of the pair
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
                 "h"(static_cast<uint16_t>(3))
                 : "memory");
}

// work item of a pair: tiles are (row block of 256, column block of 256)
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
        syrk2_kernel(const __grid_constant__ CUtensorMap map_u, const WorkList wl, int32_t *__restrict__ S, int32_t *__restrict__ D,
                     uint32_t n_cells, int epi_mode) {
    const uint32_t n_work = wl.n_work;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + STAGES * STAGE_BYTES);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * STAGES + 2);
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + STAGES);
    const uint32_t tmem_full = smem_u32(bars + 2 * STAGES), tmem_empty = smem_u32(bars + 2 * STAGES + 1);
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const uint32_t pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
    const bool leader = rank == 0;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_u) : "memory");
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full0 + 8 * s, 2);  // one arrive.expect_tx per CTA of the pair (only the leader's is used)
            mbar_init(empty0 + 8 * s, 1); // the leader's commit, multicast
        }
        mbar_init(tmem_full, 1);          // the leader's commit, multicast
        mbar_init(tmem_empty, 256);       // the epilogue threads of both CTAs (only the leader's is used)
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    cluster_sync_all(); // barriers and TMEM of both CTAs exist before anything is sent across the pair
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t tmem_Q = tmem_base, tmem_T = tmem_base + BN;

    if (warp == 0) {
        // ===== TMA producer (both CTAs): own 128 rows of A, own half of B =====
        if (elect_one()) {
            uint32_t stage = 0, phase = 0, wave = 0;
            for (uint32_t w = pair; w < n_work; w += n_pairs, ++wave) {
                const WorkItem wi = work_item(wl, w);
                // Wave sync: the pairs start the loads of their n-th tile together. The tiles of a wave share operand
                // slabs through L2, but L2 only holds what was fetched during the last ~30 us; without this the pairs
                // drift apart (diagonal tiles have slower epilogues) and every pair streams its slabs from HBM again.
                // All pairs are resident (grid <= SM count, one CTA per SM), every wave before the last one is full.
                if (leader && wave > 0) {
                    atomicAdd(wl.wave_ctr, 1u);
                    // arrivals so far: n_pairs per earlier wave, and the pairs that have an item in this (maybe last, partial) wave
                    const uint32_t want = (wave - 1) * n_pairs + min(n_pairs, n_work - wave * n_pairs);
                    uint32_t seen;
                    do {
                        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(wl.wave_ctr) : "memory");
                        if (seen < want) {
                            __nanosleep(64);
                        }
                    } while (seen < want);
                }
                for (uint32_t kb = wi.k0; kb < wi.k1; ++kb) {
                    mbar_wait(empty0 + 8 * stage, phase ^ 1);
                    const uint32_t sa = smem_u32(smem + stage * STAGE_BYTES), sb = sa + A_BYTES;
                    const uint32_t bar = mapa_u32(full0 + 8 * stage, 0); // the leader's barrier
                    mbar_expect_tx_remote(bar, STAGE_BYTES);
                    const int32_t ch = static_cast<int32_t>(kb >> wl.ck_shift);
                    const int32_t kx = static_cast<int32_t>((kb - (static_cast<uint32_t>(ch) << wl.ck_shift)) * KB_BYTES);
                    const uint32_t kbb = kb >= wl.kb_neg0 ? kb + wl.kb_negd : kb;
                    const int32_t chb = static_cast<int32_t>(kbb >> wl.ck_shift);
                    const int32_t kxb = static_cast<int32_t>((kbb - (static_cast<uint32_t>(chb) << wl.ck_shift)) * KB_BYTES);
                    tma_load_3d_2sm(sa, &map_u, bar, kx, wi.rb * 256 + rank * 128, ch);
                    tma_load_3d_2sm(sb, &map_u, bar, kxb, wi.cb * 256 + rank * 128, chb);
                    if (++stage == STAGES) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (leader CTA only) =====
        if (leader && elect_one()) {
            uint32_t stage = 0, phase = 0, acc_phase = 0;
            for (uint32_t w = pair; w < n_work; w += n_pairs) {
                const WorkItem wi = work_item(wl, w);
                mbar_wait(tmem_empty, acc_phase ^ 1); // both CTAs' epilogues have drained the accumulators
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                for (uint32_t kb = wi.k0; kb < wi.k1; ++kb) {
                    mbar_wait(full0 + 8 * stage, phase);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t sa = smem_u32(smem + stage * STAGE_BYTES), sb = sa + A_BYTES;
                    const uint32_t first = kb == wi.k0 ? 0u : 1u;
                    umma_i8_2sm(tmem_T, make_desc(sa), make_desc(sb), first);
                    umma_i8_2sm(tmem_Q, make_desc(sa + 32), make_desc(sb + 32), first);
                    umma_i8_2sm(tmem_Q, make_desc(sa + 64), make_desc(sb + 64), 1u);
                    umma_i8_2sm(tmem_Q, make_desc(sa + 96), make_desc(sb + 96), 1u);
                    umma_commit_2sm(empty0 + 8 * stage); // frees the slot in both CTAs once these MMAs retire
                    if (++stage == STAGES) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
                umma_commit_2sm(tmem_full); // accumulators complete, in both CTAs
                acc_phase ^= 1;
            }
        }
    } else {
        // ===== epilogue (both CTAs): warps 2..5, TMEM lanes 32*(warp%4) .. +31 = this CTA's 128 rows =====
        const uint32_t lane_base = 32 * (warp & 3);
        const uint32_t leader_tmem_empty = mapa_u32(tmem_empty, 0);
        uint32_t acc_phase = 0;
        for (uint32_t w = pair; w < n_work; w += n_pairs) {
            const WorkItem wi = work_item(wl, w);
            mbar_wait(tmem_full, acc_phase);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t row0 = wi.rb * 256 + rank * 128;
            const uint32_t row = row0 + lane_base + lane;
            int32_t *Srow = S + static_cast<uint64_t>(row) * n_cells;
            int32_t *Drow = D + static_cast<uint64_t>(row) * n_cells;
            // this CTA's 128 x 256 part lies strictly above the diagonal and inside the matrix
            const bool interior = wi.cb * 256 >= row0 + 128 && wi.cb * 256 + 256 <= n_cells && row0 + 128 <= n_cells;
            const bool vec = interior && !wi.partial && epi_mode != EPI_RED && (n_cells & 3u) == 0;
#pragma unroll 1
            for (uint32_t cc = 0; cc < 256 / 32; ++cc) {
                uint32_t q[32], t[32];
                tmem_ld32(tmem_Q + (lane_base << 16) + cc * 32, q);
                tmem_ld32(tmem_T + (lane_base << 16) + cc * 32, t);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                const uint32_t col0 = wi.cb * 256 + cc * 32;
                if (vec) {
                    int4 *ps = reinterpret_cast<int4 *>(Srow + col0), *pd = reinterpret_cast<int4 *>(Drow + col0);
                    int4 os[8], od[8];
                    if (epi_mode == EPI_RMW) {
#pragma unroll
                        for (int k = 0; k < 8; ++k) {
                            os[k] = ps[k];
                            od[k] = pd[k];
                        }
                    }
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        int32_t sv[4], dv[4];
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const int32_t tv = static_cast<int32_t>(t[4 * k + e]);
                            sv[e] = (static_cast<int32_t>(q[4 * k + e]) + tv) >> 2; // (4S - T + T) / 4
                            dv[e] = tv - sv[e];
                        }
                        int4 vs = make_int4(sv[0], sv[1], sv[2], sv[3]);
                        int4 vd = make_int4(dv[0], dv[1], dv[2], dv[3]);
                        if (epi_mode == EPI_RMW) {
                            vs.x += os[k].x, vs.y += os[k].y, vs.z += os[k].z, vs.w += os[k].w;
                            vd.x += od[k].x, vd.y += od[k].y, vd.z += od[k].z, vd.w += od[k].w;
                        }
                        ps[k] = vs;
                        pd[k] = vd;
                    }
                } else if (row < n_cells && col0 + 31 > row) {
#pragma unroll
                    for (int k = 0; k < 32; ++k) {
                        const uint32_t col = col0 + k;
                        const int32_t tv = static_cast<int32_t>(t[k]);
                        const int32_t sv = (static_cast<int32_t>(q[k]) + tv) >> 2;
                        const int32_t dv = tv - sv;
                        if (col > row && col < n_cells) {
                            if (sv) {
                                atomicAdd(Srow + col, sv);
                            }
                            if (dv) {
                                atomicAdd(Drow + col, dv);
                            }
                        }
                    }
                }
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            mbar_arrive_remote(leader_tmem_empty);
            acc_phase ^= 1;
        }
    }
    __syncthreads();
    cluster_sync_all(); // nobody frees TMEM or exits while the other CTA may still be using the pair
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS));
    }
}

} // namespace

// One launch of the tensor kernel, with everything it needs held by value: the launch may be issued later than the call that
// prepared it (sgpu_ctx::tensor_jobs, late launch).
namespace {
struct TensorLaunch {
    CUtensorMap map;
    WorkList wl;
    int32_t *S = nullptr, *D = nullptr;
    uint32_t N = 0;
    int epi = EPI_RMW;
    unsigned grid = 0;                     // CTA pairs
    sgpu_ctx::TensorJob job;               // events + what the job will own
    cudaEvent_t staged = nullptr;          // on ctx->stream, behind the staging kernel (late launches only)
};

// t0, memset of the wave counter, kernel, t1 on stream gs; the job joins the context's list
int issue_tensor_launch(sgpu_ctx *ctx, cudaStream_t gs, TensorLaunch &tl) {
    ctx->tensor_jobs.push_back(tl.job); // the list owns the events and the panel from here on, whatever happens below
    SGPU_CUDA(ctx, cudaMemsetAsync(tl.wl.wave_ctr, 0, sizeof(unsigned int), gs));
    SGPU_CUDA(ctx, cudaEventRecord(tl.job.t0, gs));
    SGPU_LAUNCH(ctx, (syrk2_kernel<<<2 * tl.grid, GEMM_THREADS, SMEM_BYTES, gs>>>(tl.map, tl.wl, tl.S, tl.D, tl.N, tl.epi)));
    const cudaError_t le = cudaGetLastError();
    SGPU_CUDA(ctx, cudaEventRecord(tl.job.t1, gs));
    SGPU_CUDA(ctx, le);
    return SGPU_OK;
}
} // namespace

// The prepared launch of the last deferred tensor kernel, if it has not been issued yet. It is issued behind the NEXT batch's
// link_window kernel (after_main = true: that kernel needs whole SMs and would otherwise wait for the tensor kernel to end,
// with the stream's other kernels queued behind it; issued in this order the tensor kernel runs beside the special-entry
// chain, the partition and the staging of the next batch instead), or by whoever needs the result or the stream first.
int sgpu_tensor_flush(sgpu_ctx *ctx, bool after_main) {
    TensorLaunch *tl = static_cast<TensorLaunch *>(ctx->pending_gemm);
    if (!tl) {
        return SGPU_OK;
    }
    ctx->pending_gemm = nullptr;
    struct Cleanup {
        sgpu_ctx *ctx;
        TensorLaunch *tl;
        bool issued = false;
        ~Cleanup() {
            ctx->event_pool.push_back(tl->staged);
            if (!issued) { // an error before the launch: the job never reached the list
                ctx->event_pool.push_back(tl->job.t0);
                ctx->event_pool.push_back(tl->job.t1);
                sgpu_dev_free(ctx, tl->job.U);
                sgpu_dev_free(ctx, tl->job.err);
            }
            delete tl;
        }
    } cleanup{ ctx, tl };
    cudaStream_t gs = ctx->tensor_stream;
    if (after_main) {
        SGPU_CUDA(ctx, cudaEventRecord(tl->staged, ctx->stream)); // re-recorded: behind everything queued so far (incl. the staging)
    }
    SGPU_CUDA(ctx, cudaStreamWaitEvent(gs, tl->staged, 0));
    SGPU_TRY(sgpu_cache_preference(ctx, true)); // what is launched from now on may run beside this kernel
    cleanup.issued = true; // from here on the job is in the list (issue_tensor_launch appends it before it reports a launch error)
    return issue_tensor_launch(ctx, gs, *tl);
}

// Upper-triangle 256 x 256 output tiles in an order that keeps the tiles in flight (one per CTA pair) inside a block
// of ~9 row blocks x 8 column blocks, so that a wave touches ~4 400 distinct operand rows instead of
// ~20 000: bands of 8 column blocks, row-block-major inside a band.
static int tile_list(sgpu_ctx *ctx, uint32_t N, uint32_t n_pad, const uint2 **d_tiles, uint32_t *n_tiles) {
    constexpr uint32_t BAND = 8;
    if (ctx->tile_cache && ctx->tile_cache_cells == N) {
        *d_tiles = static_cast<const uint2 *>(ctx->tile_cache);
        *n_tiles = ctx->tile_cache_n;
        return SGPU_OK;
    }
    std::vector<uint2> tiles;
    const uint32_t n_cb = n_pad / BN, n_rb = n_pad / BN;
    for (uint32_t band = 0; band < n_cb; band += BAND) {
        const uint32_t cb_end = std::min(n_cb, band + BAND);
        for (uint32_t rb = 0; rb < n_rb; ++rb) {
            for (uint32_t cb = band; cb < cb_end; ++cb) {
                // the tile intersects the upper triangle: its last column > its first row
                if (cb * BN + BN - 1 > rb * BN && rb * BN < N && cb * BN < N) {
                    tiles.push_back(make_uint2(rb, cb));
                }
            }
        }
    }
    if (ctx->tile_cache) {
        SGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        SGPU_CUDA(ctx, cudaFree(ctx->tile_cache));
        ctx->tile_cache = nullptr;
    }
    SGPU_CUDA(ctx, cudaMalloc(&ctx->tile_cache, std::max<size_t>(1, tiles.size()) * sizeof(uint2)));
    SGPU_CUDA(ctx, cudaMemcpy(ctx->tile_cache, tiles.data(), tiles.size() * sizeof(uint2), cudaMemcpyHostToDevice));
    ctx->tile_cache_cells = N;
    ctx->tile_cache_n = static_cast<uint32_t>(tiles.size());
    *d_tiles = static_cast<const uint2 *>(ctx->tile_cache);
    *n_tiles = ctx->tile_cache_n;
    return SGPU_OK;
}

int sgpu_gemm_counts(sgpu_ctx *ctx, const sgpu_pileup *p, const LinkResult &lr, sgpu_counts *c, uint64_t *n_pairs) {
    if (n_pairs) {
        *n_pairs = 0; // not enumerated on this path
    }
    GemmInput in;
    in.row_ptr = p->d_row_ptr;
    in.gid_base = p->wide ? nullptr : p->d_gid_base;
    in.gid_base32 = p->wide ? p->d_gid_base32 : nullptr;
    in.n_loci = p->n_loci;
    in.n_main = lr.ranged ? lr.n_own : p->n_loci;
    in.main_loci = lr.ranged ? lr.own_loci.p : nullptr;
    in.n_entries = p->n_entries;
    in.sp_bits = lr.sp_bits.p;
    in.gmap = lr.gmap.p;
    in.gmap_identity = lr.gmap_identity;
    in.n_groups = lr.n_groups;
    in.sp_code = lr.sp_code.p;
    in.sp_locus = lr.sp_locus.p;
    in.sp_start = lr.sp_start.p;
    in.n_special = lr.n_special;
    in.tail_loci = lr.tail_loci.p;
    in.n_tail_loci = lr.n_tail_loci;
    in.may_defer = true;
    return sgpu_gemm_run(ctx, in, c->n, c->i32 + PLANE_S * c->nn, c->i32 + PLANE_D * c->nn, &c->fresh, &c->poisoned);
}

// The GEMM path on any CSR of (cell group, letter) entries: loci [0, n_main) are counted, the loci listed
// in tail_loci are subtracted as Z Z^T. Used for the pileup itself and for the derived pileup of locus
// pairs of the second-order correction (multilocus.cu).
int sgpu_gemm_run(sgpu_ctx *ctx, const GemmInput &in, uint32_t N, int32_t *S_plane, int32_t *D_plane, bool *fresh, bool *poisoned) {
    cudaStream_t st = ctx->stream;
    const uint64_t P = in.n_main;
    if (P == 0 || in.n_entries == 0 || N < 2) {
        return SGPU_OK;
    }
    if (N > ST_MAX_STRIPES * (ST_MAX_CELLS & ~3u) - 256) { // stripes of the staging tiles; cells are 16-bit in the partition's group map
        return sgpu_fail(ctx, SGPU_E_ARG, "the GEMM path supports at most %u cells", ST_MAX_STRIPES * (ST_MAX_CELLS & ~3u) - 256);
    }
    const uint32_t n_pad = (N + BN - 1) / BN * BN;
    // the tail k-blocks (Z and -Z) ride along with the first panel
    const uint32_t kbs_tail = static_cast<uint32_t>((in.n_tail_loci + LOCI_PER_KB - 1) / LOCI_PER_KB);
    // panel: at most 3 GB of Hadamard planes (98 304 loci at 8 192 padded cells: a bench sub-batch of ~65 700 significant
    // loci used to spill a few hundred loci into a second panel, i.e. a second read-modify-write pass over the planes)
    uint64_t panel = (3ull << 30) / (4ull * n_pad) / LOCI_PER_KB * LOCI_PER_KB;
    if (const char *env = getenv("SECEDO_B200_PANEL_LOCI")) { // tests: force several panels on small inputs
        panel = std::max(1, atoi(env)) / LOCI_PER_KB * LOCI_PER_KB;
    }
    panel = std::max<uint64_t>(panel, LOCI_PER_KB);
    panel = std::min<uint64_t>(panel, (P + LOCI_PER_KB - 1) / LOCI_PER_KB * LOCI_PER_KB);
    const uint64_t kbs_max = panel / LOCI_PER_KB + 2ull * kbs_tail;
    PanelLayout pl;
    pl.ck_shift = 5; // 32 k-blocks = 1 024 loci per chunk: 4 KB per cell, 33.8 MB per chunk at 8 192 cells
    const uint32_t ck = 1u << pl.ck_shift;
    pl.cell_words = (ck | 1u) * 32u; // odd number of lines: consecutive cells do not alias in the L2 sets
    pl.chunk_words = static_cast<uint64_t>(n_pad) * pl.cell_words;
    const uint64_t n_chunks_max = (kbs_max + ck - 1) / ck;
    SGPU_TRACE(ctx, "gemm: enter");

    // tensor kernels of earlier batches: issue the one still pending, retire the finished ones; never more than two operand
    // panels in flight
    SGPU_TRY(sgpu_tensor_flush(ctx, false));
    SGPU_TRY(sgpu_tensor_poll(ctx, false));
    while (ctx->tensor_jobs.size() >= 2) {
        SGPU_CUDA(ctx, cudaEventSynchronize(ctx->tensor_jobs.front().t1));
        SGPU_TRY(sgpu_tensor_poll(ctx, false));
    }
    DevBuf<uint32_t> U;
    DevBuf<int> d_err;
    SGPU_CUDA(ctx, U.alloc(n_chunks_max * pl.chunk_words, ctx));
    SGPU_CUDA(ctx, d_err.alloc(2, ctx));
    SGPU_CUDA(ctx, cudaMemsetAsync(d_err.p, 0, 2 * sizeof(int), st));
    SGPU_TRACE(ctx, "gemm: alloc");

    // tensor map over U: [chunk][cell][ck x 128 bytes], box = 128 cells x 128 bytes, 128B swizzle
    CUtensorMap map;
    {
        const cuuint64_t gdim[3] = { static_cast<cuuint64_t>(ck) * KB_BYTES, n_pad, n_chunks_max };
        const cuuint64_t gstride[2] = { static_cast<cuuint64_t>(pl.cell_words) * 4, pl.chunk_words * 4 };
        const cuuint32_t box[3] = { KB_BYTES, 128, 1 };
        const cuuint32_t estr[3] = { 1, 1, 1 };
        // resolved through the runtime so that the library does not link libcuda.so (it must load, and
        // fail loudly in sgpu_init, on a machine without a driver)
        typedef CUresult (*encode_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                      const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                      CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        SGPU_CUDA(ctx, cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (fn == nullptr || qres != cudaDriverEntryPointSuccess) {
            return sgpu_fail(ctx, SGPU_E_CUDA, "driver does not provide cuTensorMapEncodeTiled");
        }
        CUresult r = reinterpret_cast<encode_fn>(fn)(&map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, U.p, gdim, gstride, box, estr,
                                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                            CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            return sgpu_fail(ctx, SGPU_E_CUDA, "cuTensorMapEncodeTiled failed (%d)", static_cast<int>(r));
        }
    }
    SGPU_CUDA(ctx, cudaFuncSetAttribute(syrk2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    const uint2 *d_tiles = nullptr;
    uint32_t n_tiles = 0;
    SGPU_TRY(tile_list(ctx, N, n_pad, &d_tiles, &n_tiles));
    SGPU_TRACE(ctx, "gemm: tensor map + tiles");

    // The tensor kernel goes to the context's tensor stream behind an event of its staging kernel and the call returns
    // without waiting for it (in.may_defer: the first-order counts of sgpu_counts_accumulate; callers that read the
    // result right away keep the kernel on ctx->stream). The panel and the error / wave-counter words belong to the job of
    // the LAST panel; an error return before that job exists waits for the kernels already launched.
    const bool defer = in.may_defer && ctx->async_gemm && ctx->tensor_stream != nullptr;
    cudaStream_t gs = defer ? ctx->tensor_stream : st;
    struct PanelOwner {
        sgpu_ctx *ctx;
        cudaStream_t gs;
        void *U;
        int *err;
        bool launched = false;
        ~PanelOwner() {
            if (U || err) {
                if (launched) {
                    cudaStreamSynchronize(gs);
                }
                sgpu_dev_free(ctx, U);
                sgpu_dev_free(ctx, err);
            }
        }
    } owner{ ctx, gs, U.take(), d_err.take() };
    uint32_t *const Up = static_cast<uint32_t *>(owner.U);
    int *const errp = owner.err;
    auto get_event = [&](cudaEvent_t *e) -> cudaError_t {
        if (!ctx->event_pool.empty()) {
            *e = ctx->event_pool.back();
            ctx->event_pool.pop_back();
            return cudaSuccess;
        }
        return cudaEventCreateWithFlags(e, cudaEventDefault);
    };
    // staging time: events on ctx->stream, read after the synchronisation that follows every staging kernel
    cudaEvent_t ev_s0 = nullptr, ev_s1 = nullptr;
    SGPU_CUDA(ctx, get_event(&ev_s0));
    SGPU_CUDA(ctx, get_event(&ev_s1));
    struct EventReturn {
        sgpu_ctx *ctx;
        cudaEvent_t *a, *b;
        ~EventReturn() {
            ctx->event_pool.push_back(*a);
            ctx->event_pool.push_back(*b);
        }
    } event_return{ ctx, &ev_s0, &ev_s1 };
    const uint32_t sms = static_cast<uint32_t>(ctx->sm_count);
    // stripes of cells per staging CTA: as few as the largest tile (ST_MAX_CELLS) allows
    const uint32_t n_stripes = std::min<uint32_t>(ST_MAX_STRIPES, (n_pad + ST_MAX_CELLS - 1) / ST_MAX_CELLS);
    const uint32_t cells_per_cta = ((n_pad + n_stripes - 1) / n_stripes + 3) / 4 * 4;
    const size_t st_smem = static_cast<size_t>(cells_per_cta) * 128;
    SGPU_CUDA(ctx, cudaFuncSetAttribute(stage_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(st_smem)));

    // per-entry (cell, base) with the group map and the special bitmap applied, partitioned by stripe
    // inside every locus, once per call
    DevBuf<uint16_t> cellbase;
    DevBuf<uint32_t> seg;
    const uint64_t E = in.n_entries;
    SGPU_CUDA(ctx, cellbase.alloc(E + 8, ctx));
    SGPU_CUDA(ctx, seg.alloc(in.n_loci * (n_stripes + 1), ctx));
    SGPU_CUDA(ctx, cudaEventRecord(ev_s0, st)); // the partition is folded into the first panel's staging time
    {
        const unsigned grid = static_cast<unsigned>(std::min<uint64_t>(in.n_loci, static_cast<uint64_t>(sms) * 16));
        const size_t psmem = (static_cast<size_t>(PART_OUT) + (in.gmap_identity ? 0 : in.n_groups)) * sizeof(uint16_t);
        if (psmem > 200 * 1024) {
            return sgpu_fail(ctx, SGPU_E_ARG, "too many groups (%u) for the shared-memory group map of the GEMM path", in.n_groups);
        }
        auto run_partition = [&](auto *gid_base) -> int {
            using GB = std::remove_const_t<std::remove_pointer_t<decltype(gid_base)>>;
            PartitionArgs<GB> pa;
            pa.row_ptr = in.row_ptr;
            pa.gid_base = gid_base;
            pa.sp_bits = in.sp_bits;
            pa.gmap = in.gmap;
            pa.n_groups = in.n_groups;
            pa.n_cells = N;
            pa.identity = in.gmap_identity ? 1u : 0u;
            pa.n_loci = in.n_loci;
            pa.n_stripes = n_stripes;
            pa.stripe_magic = static_cast<uint32_t>(((1ull << 32) + cells_per_cta - 1) / cells_per_cta);
            pa.cells_per_cta = cells_per_cta;
            pa.cellbase = cellbase.p;
            pa.seg = seg.p;
            pa.err = errp;
            SGPU_CUDA(ctx, cudaFuncSetAttribute(partition_kernel<GB>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(psmem)));
            SGPU_LAUNCH(ctx, (partition_kernel<GB><<<grid, 256, psmem, st>>>(pa)));
            return SGPU_OK;
        };
        SGPU_TRY(in.gid_base32 ? run_partition(in.gid_base32) : run_partition(in.gid_base));
    }

    bool first = true;
    for (uint64_t l0 = 0; l0 < P; l0 += panel) {
        const uint64_t l1 = std::min<uint64_t>(P, l0 + panel);
        const uint64_t nl = l1 - l0;
        const bool last = l1 == P;
        const uint32_t kbs_main = static_cast<uint32_t>((nl + LOCI_PER_KB - 1) / LOCI_PER_KB);
        const uint32_t kt = first ? kbs_tail : 0;
        if (!first) {
            SGPU_CUDA(ctx, cudaEventRecord(ev_s0, st));
        }
        StageArgs sa;
        sa.row_ptr = in.row_ptr;
        sa.cellbase = cellbase.p;
        sa.seg = seg.p;
        sa.n_pad = n_pad;
        sa.sp_code = in.sp_code;
        sa.sp_locus = in.sp_locus;
        sa.sp_start = in.sp_start;
        sa.l0 = static_cast<uint32_t>(l0);
        sa.nl = static_cast<uint32_t>(nl);
        sa.main_loci = in.main_loci;
        sa.kbs_main = kbs_main;
        sa.tail_loci = in.tail_loci;
        sa.n_tail = kt ? static_cast<uint32_t>(in.n_tail_loci) : 0;
        sa.kbs_tail = kt;
        sa.cells_per_cta = cells_per_cta;
        sa.n_stripes = n_stripes;
        sa.pl = pl;
        sa.U = Up;
        sa.err = errp;
        SGPU_LAUNCH(ctx, (stage_tile_kernel<<<(kbs_main + kt) * n_stripes, ST_THREADS, st_smem, st>>>(sa)));
        SGPU_CUDA(ctx, cudaGetLastError());
        SGPU_CUDA(ctx, cudaEventRecord(ev_s1, st));
        SGPU_TRACE(ctx, "gemm: stage");
        // The range checks of the partition and staging kernels are looked at BEFORE the tensor kernel touches the count
        // planes: an input outside the int8 path (more than 127 reads of one cell at one locus) or with bad group ids
        // leaves the planes as they were (first panel; SGPU_PATH_AUTO then takes the scatter path) or holding the sum of
        // the panels before it. The tensor stream is busy with the previous batch meanwhile.
        SGPU_CUDA(ctx, cudaMemcpyAsync(&ctx->h_scratch[2], errp, sizeof(int), cudaMemcpyDeviceToHost, st));
        SGPU_CUDA(ctx, cudaStreamSynchronize(st));
        {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, ev_s0, ev_s1) == cudaSuccess) {
                ctx->ms_stage += ms;
            }
        }
        const int err = static_cast<int>(ctx->h_scratch[2] & 0xFFFFFFFFu);
        if (err == SGPU_E_CELL_RANGE) {
            return sgpu_fail(ctx, err, "a group id is >= n_groups or maps to a cell >= num_cells (filter the pileup first)");
        }
        if (err != 0) {
            if (first) {
                return sgpu_fail(ctx, SGPU_E_COUNT_RANGE, "more than 127 reads of one cell at one locus: outside the int8 GEMM path, use the "
                                 "scatter path (count planes untouched)");
            }
            if (poisoned) {
                *poisoned = true; // the panels before this one have been added: the planes hold a partial sum
            }
            return sgpu_fail(ctx, SGPU_E_COUNT_RANGE, "more than 127 reads of one cell at one locus: outside the int8 GEMM path, use the scatter "
                             "path (the counts object holds a partial sum: sgpu_counts_zero before using it again)");
        }

        WorkList wl;
        wl.tiles = d_tiles;
        wl.kbs = kbs_main + kt;
        wl.ck_shift = pl.ck_shift;
        wl.kb_neg0 = kbs_main;
        wl.kb_negd = kt;
        wl.wave_ctr = reinterpret_cast<unsigned int *>(errp + 1);
        // whole tiles in full rounds of the grid; the rest (or everything, when there are few tiles) in
        // K ranges so that every SM has work in the last round
        const uint32_t units = sms / 2; // CTA pairs that take work items
        wl.n_full = n_tiles >= 2 * units ? n_tiles / units * units : 0;
        const uint32_t rest = n_tiles - wl.n_full;
        uint32_t splits = 1;
        if (rest) {
            const uint32_t target = wl.n_full ? units : 2 * units;
            splits = static_cast<uint32_t>(std::min<uint64_t>(wl.kbs, std::max<uint32_t>(1, target / rest)));
        }
        wl.per = (wl.kbs + splits - 1) / splits;
        wl.splits = (wl.kbs + wl.per - 1) / wl.per; // no empty range
        wl.n_work = wl.n_full + rest * wl.splits;
        // the planes are zero right after sgpu_counts_zero: the first panel stores, later ones add in place
        const int epi = *fresh ? EPI_STORE : EPI_RMW;
        const unsigned grid = static_cast<unsigned>(std::min<uint64_t>(wl.n_work, units));
        TensorLaunch tl;
        tl.map = map;
        tl.wl = wl;
        tl.S = S_plane;
        tl.D = D_plane;
        tl.N = N;
        tl.epi = epi;
        tl.grid = grid;
        tl.job.planes = S_plane;
        SGPU_CUDA(ctx, get_event(&tl.job.t0));
        SGPU_CUDA(ctx, get_event(&tl.job.t1));
        *fresh = false;
        if (last && defer) {
            // prepared, not issued: sgpu_tensor_flush (behind the next batch's link_window kernel, or at the first join)
            TensorLaunch *pending = new TensorLaunch(tl);
            if (get_event(&pending->staged) != cudaSuccess || cudaEventRecord(pending->staged, st) != cudaSuccess) {
                delete pending;
                return sgpu_fail(ctx, SGPU_E_CUDA, "event for the deferred tensor kernel");
            }
            pending->job.U = owner.U;
            pending->job.err = owner.err;
            owner.U = nullptr;
            owner.err = nullptr;
            ctx->pending_gemm = pending;
        } else {
            if (defer) {
                SGPU_CUDA(ctx, cudaStreamWaitEvent(gs, ev_s1, 0)); // staged (and everything before it on ctx->stream: the zeroed planes)
                SGPU_TRY(sgpu_cache_preference(ctx, true));        // what is launched from now on may run beside this kernel
            }
            if (last) { // the job of the last panel owns the panel
                tl.job.U = owner.U;
                tl.job.err = owner.err;
            }
            owner.launched = true;
            if (last) { // the job list owns them now (also if the launch fails: the job is in the list by then)
                owner.U = nullptr;
                owner.err = nullptr;
            }
            SGPU_TRY(issue_tensor_launch(ctx, gs, tl));
            if (!last && defer) {
                SGPU_CUDA(ctx, cudaStreamWaitEvent(st, ctx->tensor_jobs.back().t1, 0)); // the next panel is staged into the same buffer
            }
        }
        first = false;
        SGPU_TRACE(ctx, "gemm: syrk");
    }
    if (!defer) { // the caller goes on with the result on ctx->stream: nothing stays in flight
        SGPU_CUDA(ctx, cudaStreamSynchronize(st));
        SGPU_TRY(sgpu_tensor_poll(ctx, true));
    }
    return SGPU_OK;
}

// Jobs whose end event has been reached: kernel time into the context's statistics, events back to the pool, operand
// panel back to the cache (whoever gets it next is ordered behind this call on ctx->stream, and the kernel is done).
int sgpu_tensor_poll(sgpu_ctx *ctx, bool wait_all) {
    if (wait_all) {
        SGPU_TRY(sgpu_tensor_flush(ctx, false));
    }
    while (!ctx->tensor_jobs.empty()) {
        sgpu_ctx::TensorJob &j = ctx->tensor_jobs.front();
        cudaError_t q = wait_all ? cudaEventSynchronize(j.t1) : cudaEventQuery(j.t1);
        if (q == cudaErrorNotReady) {
            break; // jobs finish in order
        }
        if (q != cudaSuccess) {
            return sgpu_fail(ctx, SGPU_E_CUDA, "tensor kernel failed: %s", cudaGetErrorString(q));
        }
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, j.t0, j.t1) == cudaSuccess) {
            ctx->ms_syrk += ms;
            ++ctx->n_syrk;
        }
        ctx->event_pool.push_back(j.t0);
        ctx->event_pool.push_back(j.t1);
        sgpu_dev_free(ctx, j.U);
        sgpu_dev_free(ctx, j.err);
        ctx->tensor_jobs.pop_front();
    }
    return SGPU_OK;
}

int sgpu_tensor_join(sgpu_ctx *ctx, const void *planes) {
    const TensorLaunch *pending = static_cast<const TensorLaunch *>(ctx->pending_gemm);
    if (pending && (planes == nullptr || pending->job.planes == planes)) {
        SGPU_TRY(sgpu_tensor_flush(ctx, false));
    }
    for (auto it = ctx->tensor_jobs.rbegin(); it != ctx->tensor_jobs.rend(); ++it) {
        if (planes == nullptr || it->planes == planes) { // jobs finish in order: the last one of these planes covers the earlier ones
            SGPU_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, it->t1, 0));
            break;
        }
    }
    return sgpu_cache_preference(ctx, false); // what the caller launches next runs alone (or at most beside another object's kernel)
}
