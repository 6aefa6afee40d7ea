// Normalised graph Laplacian of the similarity matrix and its leading eigenpairs (SURVEY 8(f) row 3).
//
// Reference: laplacian() spectral_clustering.cpp:33-52 and the arma::eig_sym call in spectral_clustering()
// :127-138. The reference decomposes the whole N x N Laplacian L = I - D^-1/2 A D^-1/2 (LAPACK dsyevd through
// Armadillo) and then uses the eigenvectors of the 3..7 SMALLEST eigenvalues only (:166-171, :218, :236).
// Here the matrix stays in HBM (it is produced there by the epilogue) and only those eigenpairs are computed:
//
//   B  = D^-1/2 A D^-1/2                     the k smallest eigenvalues of L are 1 - (the k largest of B)
//   v0 = sqrt(d) / |sqrt(d)|, B v0 = v0      known in closed form; deflated at once: M = B - v0 v0^T
//   Chebyshev-filtered subspace iteration on M with a block of b vectors: Rayleigh-Ritz, converged Ritz
//   pairs are locked from the top and deflated INTO the matrix (M -= theta x x^T, one pass over M), the filter
//   damps [lower bound (Lanczos), smallest Ritz value of the block].
//
// The only O(N^2) work per step is the block product Y = alpha M X + beta X + gamma W (symm_block_kernel):
// every element of M is read exactly once per product, so the kernel is HBM bound for b <= 16
// (8 N^2 bytes per product) and FP64 bound above. Everything else is O(N b^2) or on b x b matrices
// (host, spectral_host.hpp).
#include "common.cuh"
#include "spectral_host.hpp"

#include <cmath>
#include <cstdlib>
#include <cstring>

namespace {


constexpr int MV_THREADS = 256;
constexpr int MV_PAD = 64; // matrices and blocks are padded to a multiple of this many rows
// rows of X staged per shared-memory chunk (double buffered with cp.async)
__host__ __device__ constexpr int mv_kc(int width) { return width <= 16 ? 64 : 32; }
// rows of the output per thread / rows of M per pipeline stage: narrow blocks are HBM bound (more bytes in
// flight: 2 x 8 rows of 16 bytes per thread), wide ones FP64 bound (4 x 8 register tile, half the shared-memory reads)
constexpr int mv_r(int width) { return width <= 16 ? 2 : 4; }
constexpr int mv_u(int width) { return width <= 16 ? 8 : 2; }

// partial[split][r][0..B) = sum over k in the split of M[k][r] * X[k][0..B)   (M symmetric: column r of M read
// as row segments, so a warp reads 32 * R * 8 contiguous bytes per k). Thread tile R rows x 8 columns in
// registers; U rows of M per pipeline stage, two stages in flight.
template <int B, int R, int U>
__global__ void __launch_bounds__(MV_THREADS, 2)
symm_block_kernel(const double *__restrict__ M, uint32_t ld, const double *__restrict__ X, double *__restrict__ partial,
                  uint32_t k_per_split) {
    constexpr int CG = B / 8;     // column groups (one warp each)
    constexpr int RG = 8 / CG;    // row groups of 32 * R rows per CTA
    constexpr int H = R / 2;      // 16-byte loads per row of M and thread
    constexpr int KC = mv_kc(B);  // rows of X per shared-memory chunk
    constexpr int CHUNK2 = KC * B / 2;
    __shared__ double2 xs[2][CHUNK2];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int cg = warp % CG, rg = warp / CG;
    const uint32_t r0 = (blockIdx.x * RG + rg) * (32u * R) + lane * R;
    const bool active = r0 < ld;
    const uint32_t kbeg = blockIdx.y * k_per_split;
    const uint32_t kend = min(ld, kbeg + k_per_split); // ld and k_per_split are multiples of KC
    double acc[R][8];
#pragma unroll
    for (int i = 0; i < R; ++i) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            acc[i][j] = 0.0;
        }
    }
    const double2 *mp = reinterpret_cast<const double2 *>(M + static_cast<size_t>(kbeg) * ld + (active ? r0 : 0));
    const size_t ld2 = ld / 2;
    double2 m0[U][H], m1[U][H];
    auto loadU = [&](double2 (&m)[U][H], uint32_t k) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const double2 *p = mp + static_cast<size_t>(k - kbeg + u) * ld2;
#pragma unroll
            for (int h = 0; h < H; ++h) {
                m[u][h] = __ldg(p + h);
            }
        }
    };
    auto fmaU = [&](const double2 (&m)[U][H], const double2 *xc, int kk) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const double2 *xr = xc + ((kk + u) * B + cg * 8) / 2;
            const double2 x01 = xr[0], x23 = xr[1], x45 = xr[2], x67 = xr[3];
            const double x[8] = { x01.x, x01.y, x23.x, x23.y, x45.x, x45.y, x67.x, x67.y };
#pragma unroll
            for (int h = 0; h < H; ++h) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    acc[2 * h][j] = fma(m[u][h].x, x[j], acc[2 * h][j]);
                    acc[2 * h + 1][j] = fma(m[u][h].y, x[j], acc[2 * h + 1][j]);
                }
            }
        }
    };
    // rows [k0, k0 + KC) of X -> xs[buf] with cp.async (16 bytes per copy), one commit group per chunk
    auto stage_x = [&](uint32_t k0, int buf) {
        const double2 *xg = reinterpret_cast<const double2 *>(X + static_cast<size_t>(k0) * B);
        for (int i = threadIdx.x; i < CHUNK2; i += MV_THREADS) {
            const uint32_t dst = static_cast<uint32_t>(__cvta_generic_to_shared(&xs[buf][i]));
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(xg + i) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    if (kbeg < kend) {
        stage_x(kbeg, 0);
        if (active) {
            loadU(m0, kbeg);
        }
    }
    int buf = 0;
    for (uint32_t k0 = kbeg; k0 < kend; k0 += KC, buf ^= 1) {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads(); // chunk k0 has landed for every thread, and everybody is done with the other buffer
        if (k0 + KC < kend) {
            stage_x(k0 + KC, buf ^ 1); // overlaps the arithmetic on this chunk
        }
        if (active) {
            const double2 *xc = xs[buf];
#pragma unroll
            for (int kk = 0; kk < KC; kk += 2 * U) {
                loadU(m1, k0 + kk + U);
                fmaU(m0, xc, kk);
                if (k0 + kk + 2 * U < kend) {
                    loadU(m0, k0 + kk + 2 * U);
                }
                fmaU(m1, xc, kk + U);
            }
        }
    }
    if (active) {
        double *out = partial + (static_cast<size_t>(blockIdx.y) * ld + r0) * B + cg * 8;
#pragma unroll
        for (int i = 0; i < R; ++i) {
            double2 *o = reinterpret_cast<double2 *>(out + static_cast<size_t>(i) * B);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                o[j] = make_double2(acc[i][2 * j], acc[i][2 * j + 1]);
            }
        }
    }
}

// ---- the same product with the matrix streamed by the TMA engine (widths <= 32) ---------------------------------
// The register-prefetch kernel above is latency bound at two CTAs per SM (ncu: 23 % warps active, the first DFMA
// after every group of loads waits on the long scoreboard, 3.5 TB/s). Here ONE thread per CTA issues bulk copies
// (cp.async.bulk, 4 KB per row of M) into a ring of TS_STAGES shared-memory stages of TS_K rows, completion through
// mbarriers, so that ~160 KB per SM are in flight without holding a single register; the 8 compute warps read their
// 64 rows x B columns from shared memory (conflict-free 16-byte reads for M, broadcasts for X). One CTA per SM,
// grid = (column tiles of 512) x (splits over K) <= number of SMs.
constexpr int TS_COLS = 512;  // rows of the output (= columns of the stored rows of M) per CTA
constexpr int TS_K = 8;       // rows of M per stage
constexpr int TS_STAGES = 6;
constexpr int TS_THREADS = 288; // 8 compute warps + 1 producer warp

__device__ __forceinline__ uint32_t sp_smem_u32(const void *p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void sp_mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void sp_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void sp_mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void sp_mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "SP_WAIT_LOOP:\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
            "@p bra SP_WAIT_DONE;\n\t"
            "bra SP_WAIT_LOOP;\n\t"
            "SP_WAIT_DONE:\n\t"
            "}" ::"r"(bar),
            "r"(parity)
            : "memory");
}
__device__ __forceinline__ void sp_bulk_load(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar)
                 : "memory");
}

template <int B>
__global__ void __launch_bounds__(TS_THREADS, 1)
symm_block_tma_kernel(const double *__restrict__ M, uint32_t ld, const double *__restrict__ X, double *__restrict__ partial,
                      uint32_t k_per_split) {
    constexpr uint32_t M_BYTES = TS_K * TS_COLS * 8, X_BYTES = TS_K * B * 8, STAGE_BYTES = M_BYTES + X_BYTES;
    extern __shared__ __align__(128) unsigned char ts_smem[];
    __shared__ __align__(8) uint64_t bars[2 * TS_STAGES];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t c0 = blockIdx.x * TS_COLS;
    const uint32_t ncols = min(static_cast<uint32_t>(TS_COLS), ld - c0); // multiple of 64
    const uint32_t kbeg = blockIdx.y * k_per_split;
    const uint32_t kend = min(ld, kbeg + k_per_split);
    const uint32_t n_it = kend > kbeg ? (kend - kbeg) / TS_K : 0;       // ld and k_per_split are multiples of TS_K
    const uint32_t full0 = sp_smem_u32(bars), empty0 = sp_smem_u32(bars + TS_STAGES), stage0 = sp_smem_u32(ts_smem);
    if (threadIdx.x == 0) {
        for (int s = 0; s < TS_STAGES; ++s) {
            sp_mbar_init(full0 + 8 * s, 1);  // the producer's arrive.expect_tx
            sp_mbar_init(empty0 + 8 * s, 8); // one arrival per compute warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (warp == 8) {
        if (lane == 0) {
            for (uint32_t it = 0; it < n_it; ++it) {
                const uint32_t s = it % TS_STAGES, ph = (it / TS_STAGES) & 1u;
                sp_mbar_wait(empty0 + 8 * s, ph ^ 1u); // passes at once on the first round
                const uint32_t dst = stage0 + s * STAGE_BYTES, bar = full0 + 8 * s;
                const uint32_t k0 = kbeg + it * TS_K;
                sp_mbar_expect_tx(bar, TS_K * ncols * 8 + X_BYTES);
#pragma unroll
                for (int u = 0; u < TS_K; ++u) {
                    sp_bulk_load(dst + u * TS_COLS * 8, M + static_cast<size_t>(k0 + u) * ld + c0, ncols * 8, bar);
                }
                sp_bulk_load(dst + M_BYTES, X + static_cast<size_t>(k0) * B, X_BYTES, bar);
            }
        }
        return;
    }
    // ---- compute warps: rows c0 + warp * 64 + lane * 2 (+1), all B columns ----
    const uint32_t rl = warp * 64u + lane * 2u;
    const bool active = rl < ncols;
    double acc[2][B];
#pragma unroll
    for (int j = 0; j < B; ++j) {
        acc[0][j] = 0.0;
        acc[1][j] = 0.0;
    }
    for (uint32_t it = 0; it < n_it; ++it) {
        const uint32_t s = it % TS_STAGES, ph = (it / TS_STAGES) & 1u;
        sp_mbar_wait(full0 + 8 * s, ph);
        if (active) {
            const double *ms = reinterpret_cast<const double *>(ts_smem + s * STAGE_BYTES);
            const double2 *xs = reinterpret_cast<const double2 *>(ts_smem + s * STAGE_BYTES + M_BYTES);
#pragma unroll
            for (int u = 0; u < TS_K; ++u) {
                const double2 m = *reinterpret_cast<const double2 *>(ms + u * TS_COLS + rl);
#pragma unroll
                for (int j = 0; j < B / 2; ++j) {
                    const double2 x = xs[u * (B / 2) + j];
                    acc[0][2 * j] = fma(m.x, x.x, acc[0][2 * j]);
                    acc[0][2 * j + 1] = fma(m.x, x.y, acc[0][2 * j + 1]);
                    acc[1][2 * j] = fma(m.y, x.x, acc[1][2 * j]);
                    acc[1][2 * j + 1] = fma(m.y, x.y, acc[1][2 * j + 1]);
                }
            }
        }
        __syncwarp();
        if (lane == 0) {
            sp_mbar_arrive(empty0 + 8 * s);
        }
    }
    if (active) {
        double *out = partial + (static_cast<size_t>(blockIdx.y) * ld + c0 + rl) * B;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            double2 *o = reinterpret_cast<double2 *>(out + static_cast<size_t>(i) * B);
#pragma unroll
            for (int j = 0; j < B / 2; ++j) {
                o[j] = make_double2(acc[i][2 * j], acc[i][2 * j + 1]);
            }
        }
    }
}

template <int B>
constexpr size_t ts_smem_bytes() {
    return static_cast<size_t>(TS_STAGES) * (TS_K * TS_COLS * 8 + TS_K * B * 8);
}

// out = alpha * sum_s partial[s] + beta * Xin + gamma * W   (element-wise over ld x B, two doubles per thread)
__global__ void combine_kernel(const double2 *__restrict__ partial, uint32_t n_split, size_t n2, double alpha,
                               const double2 *__restrict__ xin, double beta, const double2 *__restrict__ w, double gamma,
                               double2 *__restrict__ out) {
    const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n2) {
        return;
    }
    double2 s = partial[i];
    for (uint32_t k = 1; k < n_split; ++k) {
        const double2 p = partial[k * n2 + i];
        s.x += p.x;
        s.y += p.y;
    }
    double2 r = make_double2(alpha * s.x, alpha * s.y);
    if (beta != 0.0) {
        const double2 v = xin[i];
        r.x = fma(beta, v.x, r.x);
        r.y = fma(beta, v.y, r.y);
    }
    if (gamma != 0.0) {
        const double2 v = w[i];
        r.x = fma(gamma, v.x, r.x);
        r.y = fma(gamma, v.y, r.y);
    }
    out[i] = r;
}

// G_partial[cta][p x q] = X[rows of the cta]^T Y[rows of the cta]; X is [rows][p], Y is [rows][q], p, q <= 64
constexpr int GR_ROWS = 32;
__global__ void __launch_bounds__(256) gram_kernel(const double *__restrict__ X, int p, const double *__restrict__ Y, int q,
                                                   uint32_t rows, uint32_t rows_per_cta, double *__restrict__ gp) {
    __shared__ double xs[GR_ROWS * 64];
    __shared__ double ys[GR_ROWS * 64];
    const int ti = threadIdx.x >> 4, tj = threadIdx.x & 15;
    double acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a) {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            acc[a][c] = 0.0;
        }
    }
    const uint32_t rbeg = blockIdx.x * rows_per_cta, rend = min(rows, rbeg + rows_per_cta);
    for (uint32_t r0 = rbeg; r0 < rend; r0 += GR_ROWS) {
        const uint32_t nr = min(static_cast<uint32_t>(GR_ROWS), rend - r0);
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < nr * p; i += 256) {
            xs[i] = X[static_cast<size_t>(r0) * p + i];
        }
        for (uint32_t i = threadIdx.x; i < nr * q; i += 256) {
            ys[i] = Y[static_cast<size_t>(r0) * q + i];
        }
        __syncthreads();
        for (uint32_t r = 0; r < nr; ++r) {
            double xv[4], yv[4];
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                xv[a] = (ti + 16 * a < p) ? xs[r * p + ti + 16 * a] : 0.0;
                yv[a] = (tj + 16 * a < q) ? ys[r * q + tj + 16 * a] : 0.0;
            }
#pragma unroll
            for (int a = 0; a < 4; ++a) {
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    acc[a][c] = fma(xv[a], yv[c], acc[a][c]);
                }
            }
        }
    }
    double *g = gp + static_cast<size_t>(blockIdx.x) * p * q;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int i = ti + 16 * a, j = tj + 16 * c;
            if (i < p && j < q) {
                g[i * q + j] = acc[a][c];
            }
        }
    }
}

__global__ void gram_reduce_kernel(const double *__restrict__ gp, uint32_t n_cta, uint32_t pq, double *__restrict__ g) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= pq) {
        return;
    }
    double s = 0.0;
    for (uint32_t c = 0; c < n_cta; ++c) {
        s += gp[static_cast<size_t>(c) * pq + i];
    }
    g[i] = s;
}

// Z[rows][q] = X1[rows][p1] R1[p1][q] + X2[rows][p2] R2[p2][q]   (X2 may be NULL); R1, R2 in shared memory
__global__ void __launch_bounds__(256) xr_kernel(const double *__restrict__ X1, int p1, const double *__restrict__ R1,
                                                 const double *__restrict__ X2, int p2, const double *__restrict__ R2, int q,
                                                 uint32_t rows, double *__restrict__ Z) {
    extern __shared__ double rs[];
    double *r1 = rs, *r2 = rs + p1 * q;
    for (int i = threadIdx.x; i < p1 * q; i += 256) {
        r1[i] = R1[i];
    }
    if (X2) {
        for (int i = threadIdx.x; i < p2 * q; i += 256) {
            r2[i] = R2[i];
        }
    }
    __syncthreads();
    const int cpt = q / 8; // columns per thread (q is a multiple of 8, <= 64)
    const uint32_t row = blockIdx.x * 32u + (threadIdx.x >> 3);
    const int c0 = (threadIdx.x & 7) * cpt;
    if (row >= rows) {
        return;
    }
    double acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        acc[j] = 0.0;
    }
    const double *x1 = X1 + static_cast<size_t>(row) * p1;
    for (int k = 0; k < p1; ++k) {
        const double x = x1[k];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (j < cpt) {
                acc[j] = fma(x, r1[k * q + c0 + j], acc[j]);
            }
        }
    }
    if (X2) {
        const double *x2 = X2 + static_cast<size_t>(row) * p2;
        for (int k = 0; k < p2; ++k) {
            const double x = x2[k];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                if (j < cpt) {
                    acc[j] = fma(x, r2[k * q + c0 + j], acc[j]);
                }
            }
        }
    }
    double *z = Z + static_cast<size_t>(row) * q + c0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        if (j < cpt) {
            z[j] = acc[j];
        }
    }
}

// degree d[r] = sum_c A[r][c] (laplacian(), spectral_clustering.cpp:34-40); one warp per row
__global__ void rowsum_kernel(const double *__restrict__ A, uint32_t n, double *__restrict__ d) {
    const uint32_t row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= n) {
        return;
    }
    const double *a = A + static_cast<size_t>(row) * n;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    uint32_t c = lane;
    for (; c + 96 < n; c += 128) {
        s0 += a[c];
        s1 += a[c + 32];
        s2 += a[c + 64];
        s3 += a[c + 96];
    }
    for (; c < n; c += 32) {
        s0 += a[c];
    }
    double s = (s0 + s1) + (s2 + s3);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
    }
    if (lane == 0) {
        d[row] = s;
    }
}

// M[r][c] = s_r s_c A[r][c] - v0_r v0_c for r, c < n (without the v0 term when v0 is null), zero in the padding
// (ld x ld); with lap != 0 instead the reference's Laplacian itself: out[r][c] = (r == c) - s_r s_c A[r][c], n x n
// (spectral_clustering.cpp:44-50)
__global__ void scale_kernel(const double *__restrict__ A, uint32_t n, uint32_t ld, const double *__restrict__ s,
                             const double *__restrict__ v0, int lap, double *__restrict__ out) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y;
    if (lap) {
        if (c < n) {
            const double x = (s[r] * s[c]) * A[static_cast<size_t>(r) * n + c];
            out[static_cast<size_t>(r) * n + c] = (r == c ? 1.0 : 0.0) - x;
        }
        return;
    }
    if (c >= ld) {
        return;
    }
    double v = 0.0;
    if (r < n && c < n) {
        v = (s[r] * s[c]) * A[static_cast<size_t>(r) * n + c];
        if (v0) {
            v -= v0[r] * v0[c];
        }
    }
    out[static_cast<size_t>(r) * ld + c] = v;
}

// M[r][c] -= sum_i lam[i] Q[r][off + i] Q[c][off + i], i < nl <= 64 (deflation of locked Ritz pairs); 32 x 128 tiles
__global__ void __launch_bounds__(256) rank_update_kernel(double *__restrict__ M, uint32_t ld, const double *__restrict__ Q, int kq,
                                                          int off, int nl, const double *__restrict__ lam) {
    extern __shared__ double sm[];
    double *qr = sm;             // [32][nl], scaled by lam
    double *qc = sm + 32 * nl;   // [128][nl + 1]
    const uint32_t r0 = blockIdx.y * 32u, c0 = blockIdx.x * 128u;
    for (int i = threadIdx.x; i < 32 * nl; i += 256) {
        const uint32_t r = r0 + i / nl;
        qr[i] = r < ld ? lam[i % nl] * Q[static_cast<size_t>(r) * kq + off + i % nl] : 0.0;
    }
    for (int i = threadIdx.x; i < 128 * nl; i += 256) {
        const uint32_t c = c0 + i / nl;
        qc[(i / nl) * (nl + 1) + i % nl] = c < ld ? Q[static_cast<size_t>(c) * kq + off + i % nl] : 0.0;
    }
    __syncthreads();
    const int tc = threadIdx.x & 127, tr = threadIdx.x >> 7; // 2 row phases x 128 columns
    const uint32_t c = c0 + tc;
    if (c >= ld) {
        return;
    }
    for (int rr = tr; rr < 32; rr += 2) {
        const uint32_t r = r0 + rr;
        if (r >= ld) {
            break;
        }
        double s = 0.0;
        for (int i = 0; i < nl; ++i) {
            s = fma(qr[rr * nl + i], qc[tc * (nl + 1) + i], s);
        }
        M[static_cast<size_t>(r) * ld + c] -= s;
    }
}

// One Lanczos step after w = M v, on column 0 of blocks of `width` columns, by ONE CTA (n is a few thousand):
// alpha = v.w; w -= alpha v + beta_prev v_prev; beta = |w|; w /= beta. ab[2j] = alpha, ab[2j + 1] = beta.
__device__ double block_sum_1024(double v, double *red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    }
    __syncthreads(); // red may still be read from the previous reduction
    if ((threadIdx.x & 31) == 0) {
        red[threadIdx.x >> 5] = v;
    }
    __syncthreads();
    double s = 0.0;
    for (int i = 0; i < 32; ++i) {
        s += red[i];
    }
    return s;
}

__global__ void __launch_bounds__(1024) lanczos_tail_kernel(const double *__restrict__ v, const double *__restrict__ vp,
                                                            double *__restrict__ w, int width, uint32_t rows, int j,
                                                            double *__restrict__ ab) {
    __shared__ double red[32];
    double a = 0.0;
    for (uint32_t r = threadIdx.x; r < rows; r += 1024) {
        a = fma(v[static_cast<size_t>(r) * width], w[static_cast<size_t>(r) * width], a);
    }
    a = block_sum_1024(a, red);
    const double bp = j > 0 ? ab[2 * (j - 1) + 1] : 0.0;
    double nn = 0.0;
    for (uint32_t r = threadIdx.x; r < rows; r += 1024) {
        const size_t i = static_cast<size_t>(r) * width;
        const double x = w[i] - a * v[i] - bp * vp[i];
        w[i] = x;
        nn = fma(x, x, nn);
    }
    nn = block_sum_1024(nn, red);
    const double b = sqrt(nn);
    const double inv = b > 1e-14 ? 1.0 / b : 0.0;
    for (uint32_t r = threadIdx.x; r < rows; r += 1024) {
        w[static_cast<size_t>(r) * width] *= inv;
    }
    if (threadIdx.x == 0) {
        ab[2 * j] = a;
        ab[2 * j + 1] = b;
    }
}

// ------------------------------------------------------------------------------------------------------------
struct Solver {
    sgpu_ctx *ctx;
    cudaStream_t st;
    uint32_t n = 0, ld = 0; // ld = padded size (multiple of 32): M is ld x ld, blocks are ld x b
    int b = 16, kq = 8;
    DevBuf<double> M, partial, gp, g, rmat;
    uint32_t n_split = 1, k_per_split = 0, gram_ctas = 1, gram_rows = 0;
    uint64_t mv_columns = 0, mv_launches = 0;
    float ms_mv = 0.f;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool time_mv = true;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pending;

    bool use_tma(int width) const { return width <= 32 && !no_tma; }
    bool no_tma = std::getenv("SECEDO_B200_SPECTRAL_NO_TMA") != nullptr;
    uint32_t grid_x = 1;

    int setup(int width) {
        if (use_tma(width)) { // one CTA per SM, one wave
            grid_x = (ld + TS_COLS - 1) / TS_COLS;
            const uint32_t want = std::max(1u, static_cast<uint32_t>(ctx->sm_count) / grid_x);
            k_per_split = ((ld + want - 1) / want + TS_K - 1) / TS_K * TS_K;
        } else {
            const int rg = 8 / (width / 8);
            grid_x = (ld + rg * 32 * mv_r(width) - 1) / (rg * 32 * mv_r(width));
            // two CTAs per SM, ONE wave: splits rounded down so that no second, nearly empty wave is started
            const uint32_t want = std::max(1u, 2u * ctx->sm_count / grid_x);
            const uint32_t kc = mv_kc(width);
            k_per_split = ((ld + want - 1) / want + kc - 1) / kc * kc;
        }
        n_split = (ld + k_per_split - 1) / k_per_split;
        return SGPU_OK;
    }

    // out = alpha M in + beta in + gamma w       (blocks of width `width`)
    int mv(int width, double *out, const double *in, double alpha, double beta, double gamma, const double *w) {
        setup(width);
        const size_t need = static_cast<size_t>(n_split) * ld * width;
        if (partial.n < need) {
            SGPU_CUDA(ctx, partial.alloc(need, ctx));
        }
        dim3 grid(grid_x, n_split);
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        if (time_mv) {
            SGPU_TRY(get_event(&e0));
            SGPU_TRY(get_event(&e1));
            SGPU_CUDA(ctx, cudaEventRecord(e0, st));
        }
        if (use_tma(width)) {
            switch (width) {
            case 8: SGPU_LAUNCH(ctx, (symm_block_tma_kernel<8><<<grid, TS_THREADS, ts_smem_bytes<8>(), st>>>(M.p, ld, in, partial.p, k_per_split))); break;
            case 16: SGPU_LAUNCH(ctx, (symm_block_tma_kernel<16><<<grid, TS_THREADS, ts_smem_bytes<16>(), st>>>(M.p, ld, in, partial.p, k_per_split))); break;
            case 32: SGPU_LAUNCH(ctx, (symm_block_tma_kernel<32><<<grid, TS_THREADS, ts_smem_bytes<32>(), st>>>(M.p, ld, in, partial.p, k_per_split))); break;
            default: return sgpu_fail(ctx, SGPU_E_ARG, "block width %d", width);
            }
        } else {
            switch (width) {
            case 8: SGPU_LAUNCH(ctx, (symm_block_kernel<8, mv_r(8), mv_u(8)><<<grid, MV_THREADS, 0, st>>>(M.p, ld, in, partial.p, k_per_split))); break;
            case 16: SGPU_LAUNCH(ctx, (symm_block_kernel<16, mv_r(16), mv_u(16)><<<grid, MV_THREADS, 0, st>>>(M.p, ld, in, partial.p, k_per_split))); break;
            case 32: SGPU_LAUNCH(ctx, (symm_block_kernel<32, mv_r(32), mv_u(32)><<<grid, MV_THREADS, 0, st>>>(M.p, ld, in, partial.p, k_per_split))); break;
            case 64: SGPU_LAUNCH(ctx, (symm_block_kernel<64, mv_r(64), mv_u(64)><<<grid, MV_THREADS, 0, st>>>(M.p, ld, in, partial.p, k_per_split))); break;
            default: return sgpu_fail(ctx, SGPU_E_ARG, "block width %d", width);
            }
        }
        if (time_mv) {
            SGPU_CUDA(ctx, cudaEventRecord(e1, st));
            pending.emplace_back(e0, e1);
        }
        const size_t n2 = static_cast<size_t>(ld) * width / 2;
        SGPU_LAUNCH(ctx, (combine_kernel<<<static_cast<unsigned>((n2 + 255) / 256), 256, 0, st>>>(
                              reinterpret_cast<const double2 *>(partial.p), n_split, n2, alpha, reinterpret_cast<const double2 *>(in),
                              beta, reinterpret_cast<const double2 *>(w), gamma, reinterpret_cast<double2 *>(out))));
        SGPU_CUDA(ctx, cudaGetLastError());
        mv_columns += width;
        ++mv_launches;
        return SGPU_OK;
    }

    std::vector<cudaEvent_t> spare_events; // recycled: hundreds of products per solve
    int get_event(cudaEvent_t *e) {
        if (!spare_events.empty()) {
            *e = spare_events.back();
            spare_events.pop_back();
            return SGPU_OK;
        }
        SGPU_CUDA(ctx, cudaEventCreate(e));
        return SGPU_OK;
    }
    int collect_times() { // after a stream synchronisation
        for (auto &pr : pending) {
            float ms = 0.f;
            SGPU_CUDA(ctx, cudaEventElapsedTime(&ms, pr.first, pr.second));
            ms_mv += ms;
            spare_events.push_back(pr.first);
            spare_events.push_back(pr.second);
        }
        pending.clear();
        return SGPU_OK;
    }

    // ---- the rest of the backend interface of sgpu_spectral::subspace_iteration ----
    std::vector<double *> owned;
    DevBuf<double> d_lam;
    ~Solver() {
        for (double *p : owned) {
            sgpu_dev_free(ctx, p);
        }
        for (auto &pr : pending) {
            cudaEventDestroy(pr.first);
            cudaEventDestroy(pr.second);
        }
        for (cudaEvent_t e : spare_events) {
            cudaEventDestroy(e);
        }
    }
    double *alloc(size_t count) {
        void *p = nullptr;
        if (sgpu_dev_alloc(ctx, &p, count * sizeof(double)) != cudaSuccess) {
            sgpu_fail(ctx, SGPU_E_CUDA, "spectral: out of device memory (%zu doubles)", count);
            return nullptr;
        }
        owned.push_back(static_cast<double *>(p));
        return static_cast<double *>(p);
    }
    int upload(double *dst, const double *src, size_t count) {
        SGPU_CUDA(ctx, cudaMemcpyAsync(dst, src, count * sizeof(double), cudaMemcpyHostToDevice, st));
        SGPU_CUDA(ctx, cudaStreamSynchronize(st));
        return SGPU_OK;
    }
    int upload_cols(double *dst, int dst_width, const double *src, int ncols, uint32_t rows) {
        SGPU_CUDA(ctx, cudaMemcpy2DAsync(dst, dst_width * sizeof(double), src, ncols * sizeof(double), ncols * sizeof(double), rows,
                                         cudaMemcpyHostToDevice, st));
        SGPU_CUDA(ctx, cudaStreamSynchronize(st));
        return SGPU_OK;
    }
    int copy_cols(double *dst, int dst_width, const double *src, int src_width, int ncols, uint32_t rows) {
        SGPU_CUDA(ctx, cudaMemcpy2DAsync(dst, dst_width * sizeof(double), src, src_width * sizeof(double), ncols * sizeof(double), rows,
                                         cudaMemcpyDeviceToDevice, st));
        return SGPU_OK;
    }
    DevBuf<double> d_ab;
    int lanczos_tail(const double *v, const double *vp, double *w, int width, int j) {
        if (d_ab.n < 128) {
            SGPU_CUDA(ctx, d_ab.alloc(128, ctx));
        }
        if (j >= 64) {
            return sgpu_fail(ctx, SGPU_E_ARG, "spectral: too many Lanczos steps");
        }
        SGPU_LAUNCH(ctx, (lanczos_tail_kernel<<<1, 1024, 0, st>>>(v, vp, w, width, ld, j, d_ab.p)));
        SGPU_CUDA(ctx, cudaGetLastError());
        return SGPU_OK;
    }
    int lanczos_fetch(int steps, std::vector<double> &al, std::vector<double> &be) {
        std::vector<double> ab(2 * static_cast<size_t>(steps));
        SGPU_CUDA(ctx, cudaMemcpyAsync(ab.data(), d_ab.p, ab.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
        SGPU_CUDA(ctx, cudaStreamSynchronize(st));
        al.resize(steps);
        be.resize(steps);
        for (int j = 0; j < steps; ++j) {
            al[j] = ab[2 * j];
            be[j] = ab[2 * j + 1];
        }
        return collect_times();
    }
    int rank_update(const double *Q, int q_width, int off, int nl, const double *lam) {
        if (d_lam.n < 64) {
            SGPU_CUDA(ctx, d_lam.alloc(64, ctx));
        }
        SGPU_CUDA(ctx, cudaMemcpyAsync(d_lam.p, lam, nl * sizeof(double), cudaMemcpyHostToDevice, st));
        const size_t smem = (32 * nl + 128 * (nl + 1)) * sizeof(double);
        SGPU_LAUNCH(ctx, (rank_update_kernel<<<dim3((ld + 127) / 128, (ld + 31) / 32), 256, smem, st>>>(M.p, ld, Q, q_width, off, nl, d_lam.p)));
        SGPU_CUDA(ctx, cudaGetLastError());
        SGPU_CUDA(ctx, cudaStreamSynchronize(st));
        return collect_times();
    }

    // host <- X^T Y (p x q, row-major); synchronises
    int gram(const double *X, int p, const double *Y, int q, std::vector<double> &h) {
        const uint32_t ctas = std::min<uint32_t>(ctx->sm_count, (ld + GR_ROWS - 1) / GR_ROWS);
        const uint32_t rpc = ((ld + ctas - 1) / ctas + GR_ROWS - 1) / GR_ROWS * GR_ROWS;
        const uint32_t nc = (ld + rpc - 1) / rpc;
        if (gp.n < static_cast<size_t>(nc) * 64 * 64) {
            SGPU_CUDA(ctx, gp.alloc(static_cast<size_t>(nc) * 64 * 64, ctx));
        }
        if (g.n < 64 * 64) {
            SGPU_CUDA(ctx, g.alloc(64 * 64, ctx));
        }
        SGPU_LAUNCH(ctx, (gram_kernel<<<nc, 256, 0, st>>>(X, p, Y, q, ld, rpc, gp.p)));
        SGPU_LAUNCH(ctx, (gram_reduce_kernel<<<(p * q + 255) / 256, 256, 0, st>>>(gp.p, nc, p * q, g.p)));
        SGPU_CUDA(ctx, cudaGetLastError());
        h.resize(static_cast<size_t>(p) * q);
        SGPU_CUDA(ctx, cudaMemcpyAsync(h.data(), g.p, h.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
        SGPU_CUDA(ctx, cudaStreamSynchronize(st));
        return collect_times();
    }

    // Z = X1 R1 + X2 R2 with host matrices R1 (p1 x q), R2 (p2 x q)
    int xr(double *Z, const double *X1, int p1, const std::vector<double> &R1, const double *X2, int p2,
           const std::vector<double> &R2, int q) {
        const size_t n1 = static_cast<size_t>(p1) * q, n2 = X2 ? static_cast<size_t>(p2) * q : 0;
        if (rmat.n < 2 * 64 * 64) {
            SGPU_CUDA(ctx, rmat.alloc(2 * 64 * 64, ctx));
        }
        // stream-ordered copies from pageable memory return after staging the source
        SGPU_CUDA(ctx, cudaMemcpyAsync(rmat.p, R1.data(), n1 * sizeof(double), cudaMemcpyHostToDevice, st));
        if (X2) {
            SGPU_CUDA(ctx, cudaMemcpyAsync(rmat.p + n1, R2.data(), n2 * sizeof(double), cudaMemcpyHostToDevice, st));
        }
        const size_t smem = (n1 + n2) * sizeof(double);
        SGPU_LAUNCH(ctx, (xr_kernel<<<(ld + 31) / 32, 256, smem, st>>>(X1, p1, rmat.p, X2, p2, rmat.p + n1, q, ld, Z)));
        SGPU_CUDA(ctx, cudaGetLastError());
        // rmat is overwritten by the next call: keep the stream order simple
        SGPU_CUDA(ctx, cudaStreamSynchronize(st));
        return collect_times();
    }
};


// kernels with more than 48 KB of dynamic shared memory; function attributes are per device, so per context
int sgpu_spectral_attributes(sgpu_ctx *ctx) {
    if (!ctx->spectral_attr_done) {
        SGPU_CUDA(ctx, cudaFuncSetAttribute(symm_block_tma_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(ts_smem_bytes<8>())));
        SGPU_CUDA(ctx, cudaFuncSetAttribute(symm_block_tma_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(ts_smem_bytes<16>())));
        SGPU_CUDA(ctx, cudaFuncSetAttribute(symm_block_tma_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(ts_smem_bytes<32>())));
        SGPU_CUDA(ctx, cudaFuncSetAttribute(xr_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 64 * 64 * 8));
        SGPU_CUDA(ctx, cudaFuncSetAttribute(rank_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (32 * 64 + 128 * 65) * 8));
        ctx->spectral_attr_done = true;
    }
    return SGPU_OK;
}

int block_width_for(uint32_t k) {
    const uint32_t want = std::max(2 * k, k + 8);
    return want <= 8 ? 8 : want <= 16 ? 16 : want <= 32 ? 32 : 64;
}

} // namespace

// B = D^-1/2 A D^-1/2 of the reference's laplacian() (spectral_clustering.cpp:33-52), L = I - B, into M (allocated
// here, ld x ld, zero padding); with d_v0 the unit vector v0 = sqrt(d / sum d) (B v0 = v0) is stored there and M = B -
// v0 v0^T. A cell of degree 0 gets scale 0 (its row of L is the unit row, eigenvalue 1); a negative or NaN degree is
// SGPU_E_ARG (the reference would take the square root of a negative number). An all-zero A (L = I) sets *all_zero and
// allocates nothing.
int sgpu_scaled_similarity(sgpu_ctx *ctx, const double *d_A, uint32_t n, uint32_t ld, DevBuf<double> &M, DevBuf<double> *d_v0,
                           bool *all_zero) {
    cudaStream_t st = ctx->stream;
    DevBuf<double> d_deg, d_s;
    SGPU_CUDA(ctx, d_deg.alloc(n, ctx));
    SGPU_LAUNCH(ctx, (rowsum_kernel<<<(n + 7) / 8, 256, 0, st>>>(d_A, n, d_deg.p)));
    std::vector<double> deg(n), sc(n);
    SGPU_CUDA(ctx, cudaMemcpyAsync(deg.data(), d_deg.p, n * sizeof(double), cudaMemcpyDeviceToHost, st));
    SGPU_CUDA(ctx, cudaStreamSynchronize(st));
    double total = 0.0;
    for (uint32_t r = 0; r < n; ++r) {
        if (!(deg[r] >= 0.0)) {
            return sgpu_fail(ctx, SGPU_E_ARG, "spectral: cell %u has degree %g (similarities must be non-negative)", r, deg[r]);
        }
        sc[r] = deg[r] == 0.0 ? 0.0 : 1.0 / std::sqrt(deg[r]);
        total += deg[r];
    }
    *all_zero = !(total > 0.0);
    if (*all_zero) {
        return SGPU_OK;
    }
    // stream-ordered copies from pageable memory return after staging the source: the locals may go
    SGPU_CUDA(ctx, d_s.alloc(n, ctx));
    SGPU_CUDA(ctx, cudaMemcpyAsync(d_s.p, sc.data(), n * sizeof(double), cudaMemcpyHostToDevice, st));
    if (d_v0) {
        std::vector<double> v0(n);
        for (uint32_t r = 0; r < n; ++r) {
            v0[r] = std::sqrt(deg[r] / total);
        }
        SGPU_CUDA(ctx, d_v0->alloc(n, ctx));
        SGPU_CUDA(ctx, cudaMemcpyAsync(d_v0->p, v0.data(), n * sizeof(double), cudaMemcpyHostToDevice, st));
    }
    SGPU_CUDA(ctx, M.alloc(static_cast<size_t>(ld) * ld, ctx));
    SGPU_LAUNCH(ctx, (scale_kernel<<<dim3((ld + 255) / 256, ld), 256, 0, st>>>(d_A, n, ld, d_s.p, d_v0 ? d_v0->p : nullptr, 0, M.p)));
    SGPU_CUDA(ctx, cudaGetLastError());
    return SGPU_OK;
}

// d_A: n x n similarity matrix on the device (row-major, symmetric, zero diagonal)
int sgpu_spectral_device(sgpu_ctx *ctx, const double *d_A, uint32_t n, uint32_t k, double tol, double *h_evals,
                         double *h_evecs, sgpu_spectral_stats *stats) {
    using namespace sgpu_spectral;
    cudaStream_t st = ctx->stream;
    if (n < 2 || k < 1 || k > 32 || k > n) {
        return sgpu_fail(ctx, SGPU_E_ARG, "spectral: need 2 <= n and 1 <= k <= min(32, n) (n = %u, k = %u)", n, k);
    }
    tol = std::max(tol > 0 ? tol : 1e-10, 1e-13);
    SGPU_TRY(sgpu_spectral_attributes(ctx));
    struct Events { // destroyed on every return path
        cudaEvent_t e[3] = { nullptr, nullptr, nullptr };
        ~Events() {
            for (cudaEvent_t x : e) {
                if (x) {
                    cudaEventDestroy(x);
                }
            }
        }
    } evs;
    for (auto &x : evs.e) {
        SGPU_CUDA(ctx, cudaEventCreate(&x));
    }
    const cudaEvent_t t0 = evs.e[0], t1 = evs.e[1], t2 = evs.e[2];
    SGPU_CUDA(ctx, cudaEventRecord(t0, st));
    const uint64_t launches0 = ctx->launches;

    Solver S;
    S.ctx = ctx;
    S.st = st;
    S.n = n;
    S.ld = (n + MV_PAD - 1) / MV_PAD * MV_PAD;
    const uint32_t ld = S.ld;
    const int b = std::min<int>(block_width_for(k), static_cast<int>(ld)); // ld >= 64
    const int kq = static_cast<int>((k + 7) / 8 * 8);
    if (k > 1 && n < 2u * b) {
        return sgpu_fail(ctx, SGPU_E_ARG, "spectral: %u cells are too few for a block of %d vectors (k = %u)", n, b, k);
    }
    S.b = b;
    S.kq = kq;

    // ---- Laplacian: degrees, scaling, trivial eigenvector (spectral_clustering.cpp:33-52) ----
    DevBuf<double> d_v0;
    bool all_zero = false;
    SGPU_TRY(sgpu_scaled_similarity(ctx, d_A, n, ld, S.M, &d_v0, &all_zero));
    if (all_zero) {
        // all-zero similarity (tests/test_spectral_clustering.cpp:186-196 exercises it): the reference's Laplacian is
        // the identity, whose LAPACK decomposition is eigenvalue 1 with the unit vectors
        for (uint32_t i = 0; i < k; ++i) {
            if (h_evals) {
                h_evals[i] = 1.0;
            }
            if (h_evecs) {
                std::memset(h_evecs + static_cast<size_t>(i) * n, 0, n * sizeof(double));
                h_evecs[static_cast<size_t>(i) * n + i] = 1.0;
            }
        }
        if (stats) {
            std::memset(stats, 0, sizeof(*stats));
        }
        return SGPU_OK;
    }
    SGPU_CUDA(ctx, cudaEventRecord(t1, st));

    // ---- locked eigenpairs: column 0 = v0 (eigenvalue 1 of B); the iteration itself is spectral_host.hpp ----
    double *Q = S.alloc(static_cast<size_t>(ld) * kq);
    if (!Q) {
        return SGPU_E_CUDA;
    }
    SGPU_CUDA(ctx, cudaMemsetAsync(Q, 0, static_cast<size_t>(ld) * kq * sizeof(double), st));
    SGPU_CUDA(ctx, cudaMemcpy2DAsync(Q, kq * sizeof(double), d_v0.p, sizeof(double), sizeof(double), n, cudaMemcpyDeviceToDevice, st));
    SolveResult res;
    SGPU_TRY(subspace_iteration(S, n, ld, k, b, kq, tol, Q, ctx->trace, &res));
    if (!res.converged) {
        return sgpu_fail(ctx, SGPU_E_CONVERGENCE, "spectral: %zu of %u eigenpairs after %u iterations (residual %.3e, tol %.1e)",
                         res.lam.size(), k, res.outer, res.last_residual, tol);
    }
    const std::vector<double> &lam = res.lam;
    const uint32_t outer = res.outer;
    const double lo = res.lo, max_res = res.max_residual;
    SGPU_CUDA(ctx, cudaEventRecord(t2, st));
    // ---- results: eigenvalues of L ascending, eigenvectors column by column (arma::mat layout) ----
    std::vector<double> hq(static_cast<size_t>(ld) * kq);
    SGPU_CUDA(ctx, cudaMemcpyAsync(hq.data(), Q, hq.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
    SGPU_CUDA(ctx, cudaStreamSynchronize(st));
    SGPU_TRY(S.collect_times());
    std::vector<int> order(k);
    for (uint32_t i = 0; i < k; ++i) {
        order[i] = static_cast<int>(i);
    }
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return lam[x] > lam[y]; });
    for (uint32_t i = 0; i < k; ++i) {
        const int src = order[i];
        if (h_evals) {
            h_evals[i] = 1.0 - lam[src];
        }
        if (h_evecs) {
            // sign: the component of largest magnitude is positive (LAPACK's sign is arbitrary)
            double big = 0.0;
            for (uint32_t r = 0; r < n; ++r) {
                const double v = hq[static_cast<size_t>(r) * kq + src];
                if (std::fabs(v) > std::fabs(big)) {
                    big = v;
                }
            }
            const double sgn = big < 0.0 ? -1.0 : 1.0;
            for (uint32_t r = 0; r < n; ++r) {
                h_evecs[static_cast<size_t>(i) * n + r] = sgn * hq[static_cast<size_t>(r) * kq + src];
            }
        }
    }
    if (stats) {
        std::memset(stats, 0, sizeof(*stats));
        stats->outer_iterations = outer;
        stats->block = static_cast<uint32_t>(b);
        stats->matvec_columns = S.mv_columns;
        stats->matvec_launches = S.mv_launches;
        stats->launches = ctx->launches - launches0;
        stats->max_residual = max_res;
        stats->lower_bound = lo;
        SGPU_CUDA(ctx, cudaEventElapsedTime(&stats->ms_laplacian, t0, t1));
        SGPU_CUDA(ctx, cudaEventElapsedTime(&stats->ms_solver, t1, t2));
        stats->ms_matvec = S.ms_mv;
    }
    return SGPU_OK;
}

// laplacian() of the reference on the device: out is n x n on the HOST
int sgpu_laplacian_device(sgpu_ctx *ctx, const double *d_A, uint32_t n, double *h_out) {
    cudaStream_t st = ctx->stream;
    DevBuf<double> d_deg, d_s, d_out;
    SGPU_CUDA(ctx, d_deg.alloc(n, ctx));
    SGPU_CUDA(ctx, d_s.alloc(n, ctx));
    SGPU_CUDA(ctx, d_out.alloc(static_cast<size_t>(n) * n, ctx));
    SGPU_LAUNCH(ctx, (rowsum_kernel<<<(n + 7) / 8, 256, 0, st>>>(d_A, n, d_deg.p)));
    std::vector<double> deg(n);
    SGPU_CUDA(ctx, cudaMemcpyAsync(deg.data(), d_deg.p, n * sizeof(double), cudaMemcpyDeviceToHost, st));
    SGPU_CUDA(ctx, cudaStreamSynchronize(st));
    for (uint32_t r = 0; r < n; ++r) {
        deg[r] = deg[r] == 0.0 ? 0.0 : 1.0 / std::sqrt(deg[r]); // NaN for a negative degree, as in the reference
    }
    SGPU_CUDA(ctx, cudaMemcpyAsync(d_s.p, deg.data(), n * sizeof(double), cudaMemcpyHostToDevice, st));
    SGPU_LAUNCH(ctx, (scale_kernel<<<dim3((n + 255) / 256, n), 256, 0, st>>>(d_A, n, n, d_s.p, nullptr, 1, d_out.p)));
    SGPU_CUDA(ctx, cudaGetLastError());
    SGPU_CUDA(ctx, cudaMemcpyAsync(h_out, d_out.p, static_cast<size_t>(n) * n * sizeof(double), cudaMemcpyDeviceToHost, st));
    SGPU_CUDA(ctx, cudaStreamSynchronize(st));
    return SGPU_OK;
}

// test hook: out = alpha M X + beta X + gamma W with a host matrix M (n x n symmetric) and host blocks (n x width)
int sgpu_spectral_matvec_host(sgpu_ctx *ctx, const double *h_M, uint32_t n, int width, const double *h_X, const double *h_W,
                              double alpha, double beta, double gamma, double *h_out) {
    cudaStream_t st = ctx->stream;
    Solver S;
    S.ctx = ctx;
    S.st = st;
    S.n = n;
    S.ld = (n + MV_PAD - 1) / MV_PAD * MV_PAD;
    const uint32_t ld = S.ld;
    std::vector<double> pm(static_cast<size_t>(ld) * ld, 0.0), px(static_cast<size_t>(ld) * width, 0.0), pw(px.size(), 0.0);
    for (uint32_t r = 0; r < n; ++r) {
        std::memcpy(&pm[static_cast<size_t>(r) * ld], h_M + static_cast<size_t>(r) * n, n * sizeof(double));
        std::memcpy(&px[static_cast<size_t>(r) * width], h_X + static_cast<size_t>(r) * width, width * sizeof(double));
        if (h_W) {
            std::memcpy(&pw[static_cast<size_t>(r) * width], h_W + static_cast<size_t>(r) * width, width * sizeof(double));
        }
    }
    DevBuf<double> X, W, O;
    SGPU_CUDA(ctx, S.M.alloc(pm.size(), ctx));
    SGPU_CUDA(ctx, X.alloc(px.size(), ctx));
    SGPU_CUDA(ctx, W.alloc(px.size(), ctx));
    SGPU_CUDA(ctx, O.alloc(px.size(), ctx));
    SGPU_CUDA(ctx, cudaMemcpyAsync(S.M.p, pm.data(), pm.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    SGPU_CUDA(ctx, cudaMemcpyAsync(X.p, px.data(), px.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    SGPU_CUDA(ctx, cudaMemcpyAsync(W.p, pw.data(), pw.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    SGPU_TRY(sgpu_spectral_attributes(ctx));
    SGPU_TRY(S.mv(width, O.p, X.p, alpha, beta, gamma, W.p));
    SGPU_CUDA(ctx, cudaMemcpyAsync(px.data(), O.p, px.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
    SGPU_CUDA(ctx, cudaStreamSynchronize(st));
    SGPU_TRY(S.collect_times());
    for (uint32_t r = 0; r < n; ++r) {
        std::memcpy(h_out + static_cast<size_t>(r) * width, &px[static_cast<size_t>(r) * width], width * sizeof(double));
    }
    return SGPU_OK;
}
