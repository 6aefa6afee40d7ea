// Every eigenvalue of the reference's laplacian(similarity) (spectral_clustering.cpp:33-52, :127-143: arma::eig_sym of
// the whole Laplacian, whose eigenvalues go to the per-node sim_mat_eigenvalues CSV), on the device in fp64.
//
//   B = D^-1/2 A D^-1/2 (sgpu_scaled_similarity, shared with the eigenpair solver), eigenvalues of L = 1 - those of B.
//   B rather than L: a cell of degree 0 has a zero row in B, and an all-zero B has the exact eigenvalue 0, so those
//   eigenvalues of L come out as exactly 1 (L = I would leave them to the bisection tolerance).
//
//   1. Blocked Householder reduction Q^T B Q = T (LAPACK DSYTRD with DLATRD panels of NB columns). Per column j of a
//      panel: the column brought up to date with the panel's earlier reflectors (col_update_kernel), the reflector
//      (reflector_kernel, one CTA: the scalars stay on the device), w = A22 v (symv_kernel + w_kernel; the only O(n^2)
//      work of the column: one triangle of the trailing matrix is read once), the corrections - V (W^T v) - W (V^T v)
//      (dots_kernel, w_kernel) and w += alpha v (wfix_kernel). After the panel the rank-2 NB update A22 -= V W^T +
//      W V^T of the upper triangle (update_kernel). The working copy keeps only its upper triangle (c >= r) current.
//   2. Eigenvalues of T by bisection on Sturm counts (sturm.hpp, DSTEBZ's rules), one eigenvalue index per thread.
//
// Every reduction runs in a fixed order and nothing uses floating-point atomics: a call is bit-reproducible. The column
// loop neither synchronises with the host nor copies anything back.
#include "common.cuh"
#include "sturm.hpp"

#include <algorithm>
#include <cmath>
#include <cstring>

namespace {

constexpr int NB = 32;      // columns per panel: faster than 64 at 2 000 - 20 000 cells (profiles/eigenvalues_bench*.json)
constexpr int EG_PAD = 64;  // the working copy is ld x ld, ld = n rounded up to this (the symv tile)
constexpr int TT = 64;      // tile of the symmetric product and of the trailing update
constexpr int SV_CH = 8;    // tiles of one tile row per CTA of the symmetric product
constexpr int DOT_ROWS = 128;
constexpr int ROW_THREADS = 256;

// col[r] = A[j][r] - sum_{k < jj} (V[k][r] W[k][j] + W[k][r] V[k][j]) for r in [j, n): column j of the matrix brought up
// to date with the panel's first jj reflectors (row j of the upper triangle = column j below the diagonal)
__global__ void __launch_bounds__(ROW_THREADS) col_update_kernel(const double *__restrict__ A, uint32_t ld, uint32_t n, uint32_t j,
                                                                 int jj, const double *__restrict__ V, const double *__restrict__ W,
                                                                 double *__restrict__ col) {
    __shared__ double vj[NB], wj[NB];
    if (threadIdx.x < jj) {
        vj[threadIdx.x] = V[static_cast<size_t>(threadIdx.x) * ld + j];
        wj[threadIdx.x] = W[static_cast<size_t>(threadIdx.x) * ld + j];
    }
    __syncthreads();
    const uint32_t r = j + blockIdx.x * ROW_THREADS + threadIdx.x;
    if (r >= n) {
        return;
    }
    double a = A[static_cast<size_t>(j) * ld + r];
    for (int k = 0; k < jj; ++k) {
        a = fma(-V[static_cast<size_t>(k) * ld + r], wj[k], a);
        a = fma(-W[static_cast<size_t>(k) * ld + r], vj[k], a);
    }
    col[r] = a;
}

// sum over a CTA of 1024 threads in a fixed order
__device__ double cta_sum_1024(double v, double *red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    }
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

// DLARFG on col[j+1 .. n): H = I - tau v v^T with v[j+1] = 1 maps the column to beta e_{j+1}. d[j] = col[j], e[j] = beta,
// V[jj] = v (zero at rows <= j and in the padding), scal[0] = tau. The last column (j = n - 1) only has d[j].
__global__ void __launch_bounds__(1024) reflector_kernel(const double *__restrict__ col, uint32_t ld, uint32_t n, uint32_t j, int jj,
                                                         double *__restrict__ V, double *__restrict__ d, double *__restrict__ e,
                                                         double *__restrict__ scal) {
    __shared__ double red[32];
    if (threadIdx.x == 0) {
        d[j] = col[j];
    }
    if (j + 1 >= n) {
        return;
    }
    double ss = 0.0;
    for (uint32_t r = j + 2 + threadIdx.x; r < n; r += 1024) {
        ss = fma(col[r], col[r], ss);
    }
    const double xnorm = sqrt(cta_sum_1024(ss, red));
    const double alpha = col[j + 1];
    double tau = 0.0, beta = alpha, scale = 0.0;
    if (xnorm > 0.0) {
        beta = -copysign(hypot(alpha, xnorm), alpha);
        tau = (beta - alpha) / beta;
        scale = 1.0 / (alpha - beta);
    }
    double *v = V + static_cast<size_t>(jj) * ld;
    for (uint32_t r = threadIdx.x; r < ld; r += 1024) {
        v[r] = r <= j || r >= n ? 0.0 : r == j + 1 ? 1.0 : col[r] * scale;
    }
    if (threadIdx.x == 0) {
        e[j] = beta;
        scal[0] = tau;
    }
}

// The symmetric product y = A22 v from the upper triangle of the rows / columns [s, n), read once: tile (I, J >= I) adds
// A_IJ v_J to the rows of I (ypart[chunk][rows of I], summed over the CTA's chunk of SV_CH tiles) and A_IJ^T v_I to the
// rows of J (zpart[I][rows of J]); diagonal tiles use their upper triangle. v is zero outside [s, n), so the stale
// entries left of s in the first tile row do not count. grid = (chunks, tile rows from s / TT).
__global__ void __launch_bounds__(256) symv_kernel(const double *__restrict__ A, uint32_t ld, uint32_t n, uint32_t s,
                                                   const double *__restrict__ v, double *__restrict__ ypart,
                                                   double *__restrict__ zpart) {
    __shared__ double tile[TT][TT + 1];
    __shared__ double vi[TT], vj[TT], red[4][TT];
    const uint32_t nt = (n + TT - 1) / TT;
    const uint32_t I = s / TT + blockIdx.y;
    const uint32_t J0 = I + blockIdx.x * SV_CH, J1 = min(nt, J0 + SV_CH);
    if (J0 >= J1) {
        return;
    }
    const int t = threadIdx.x, lo = t & 63, q = t >> 6;
    if (t < TT) {
        vi[t] = v[I * TT + t];
    }
    const double *arow = A + static_cast<size_t>(I) * TT * ld;
    double pre[16];
    auto load = [&](uint32_t J) {
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            pre[i] = arow[static_cast<size_t>(i * 4 + q) * ld + J * TT + lo];
        }
    };
    load(J0);
    double yacc = 0.0;
    for (uint32_t J = J0; J < J1; ++J) {
        __syncthreads(); // everybody is done with the previous tile
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            tile[i * 4 + q][lo] = pre[i];
        }
        if (t < TT) {
            vj[t] = v[J * TT + t];
        }
        __syncthreads();
        if (J + 1 < J1) {
            load(J + 1); // in flight during the arithmetic on this tile
        }
        const bool diag = J == I;
        // rows of I: row lo, columns q*16 .. q*16 + 15
        double z = 0.0;
#pragma unroll
        for (int c = q * 16; c < q * 16 + 16; ++c) {
            if (!diag || c >= lo) {
                yacc = fma(tile[lo][c], vj[c], yacc);
            }
        }
        // rows of J: column lo, rows q*16 .. q*16 + 15 (strictly above the diagonal in a diagonal tile)
#pragma unroll
        for (int r = q * 16; r < q * 16 + 16; ++r) {
            if (!diag || r < lo) {
                z = fma(tile[r][lo], vi[r], z);
            }
        }
        red[q][lo] = z;
        __syncthreads();
        if (t < TT) {
            zpart[static_cast<size_t>(I) * ld + J * TT + t] = ((red[0][t] + red[1][t]) + red[2][t]) + red[3][t];
        }
    }
    __syncthreads();
    red[q][lo] = yacc;
    __syncthreads();
    if (t < TT) {
        ypart[static_cast<size_t>(blockIdx.x) * ld + I * TT + t] = ((red[0][t] + red[1][t]) + red[2][t]) + red[3][t];
    }
}

// part[cta][k] = sum over the CTA's DOT_ROWS rows of W[k][r] v[r] (k < jj) and V[k - jj][r] v[r] (jj <= k < 2 jj);
// one warp per k, rows [s, n)
__global__ void __launch_bounds__(256) dots_kernel(const double *__restrict__ V, const double *__restrict__ W, uint32_t ld, uint32_t n,
                                                   uint32_t s, int jj, const double *__restrict__ v, double *__restrict__ part) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t r0 = s + blockIdx.x * DOT_ROWS, r1 = min(n, r0 + DOT_ROWS);
    for (int k = warp; k < 2 * jj; k += 8) {
        const double *x = k < jj ? W + static_cast<size_t>(k) * ld : V + static_cast<size_t>(k - jj) * ld;
        double a = 0.0;
        for (uint32_t r = r0 + lane; r < r1; r += 32) {
            a = fma(x[r], v[r], a);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            a += __shfl_xor_sync(0xFFFFFFFFu, a, o);
        }
        if (lane == 0) {
            part[static_cast<size_t>(blockIdx.x) * 2 * NB + k] = a;
        }
    }
}

// w[r] = tau (y[r] - sum_k V[k][r] (W^T v)_k - sum_k W[k][r] (V^T v)_k) into W[jj] for r in [s, n), y = the sums of the
// symmetric product's parts; wvpart[cta] = sum of w[r] v[r] over the CTA's rows
__global__ void __launch_bounds__(ROW_THREADS) w_kernel(const double *__restrict__ ypart, const double *__restrict__ zpart, uint32_t ld,
                                                        uint32_t n, uint32_t s, int jj, const double *__restrict__ dpart,
                                                        uint32_t n_dot, const double *__restrict__ V, double *__restrict__ W,
                                                        const double *__restrict__ scal, double *__restrict__ wvpart) {
    __shared__ double dots[2 * NB];
    __shared__ double red[ROW_THREADS / 32];
    if (threadIdx.x < 2 * jj) {
        double a = 0.0;
        for (uint32_t c = 0; c < n_dot; ++c) {
            a += dpart[static_cast<size_t>(c) * 2 * NB + threadIdx.x];
        }
        dots[threadIdx.x] = a; // [0, jj): W^T v, [jj, 2 jj): V^T v
    }
    __syncthreads();
    const uint32_t r = s + blockIdx.x * ROW_THREADS + threadIdx.x;
    const double *v = V + static_cast<size_t>(jj) * ld;
    double wv = 0.0;
    if (r < n) {
        const uint32_t nt = (n + TT - 1) / TT, I = r / TT, I0 = s / TT;
        double y = 0.0;
        for (uint32_t c = 0; c * SV_CH < nt - I; ++c) {
            y += ypart[static_cast<size_t>(c) * ld + r];
        }
        for (uint32_t i = I0; i <= I; ++i) {
            y += zpart[static_cast<size_t>(i) * ld + r];
        }
        for (int k = 0; k < jj; ++k) {
            y = fma(-V[static_cast<size_t>(k) * ld + r], dots[k], y);
        }
        for (int k = 0; k < jj; ++k) {
            y = fma(-W[static_cast<size_t>(k) * ld + r], dots[jj + k], y);
        }
        const double w = scal[0] * y;
        W[static_cast<size_t>(jj) * ld + r] = w;
        wv = w * v[r];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        wv += __shfl_xor_sync(0xFFFFFFFFu, wv, o);
    }
    if ((threadIdx.x & 31) == 0) {
        red[threadIdx.x >> 5] = wv;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0;
        for (int i = 0; i < ROW_THREADS / 32; ++i) {
            a += red[i];
        }
        wvpart[blockIdx.x] = a;
    }
}

// W[jj] += alpha v, alpha = -tau / 2 (w^T v), for r in [s, n)
__global__ void __launch_bounds__(ROW_THREADS) wfix_kernel(uint32_t ld, uint32_t n, uint32_t s, int jj, const double *__restrict__ V,
                                                           double *__restrict__ W, const double *__restrict__ scal,
                                                           const double *__restrict__ wvpart, uint32_t n_w) {
    __shared__ double alpha;
    if (threadIdx.x == 0) {
        double a = 0.0;
        for (uint32_t c = 0; c < n_w; ++c) {
            a += wvpart[c];
        }
        alpha = -0.5 * scal[0] * a;
    }
    __syncthreads();
    const uint32_t r = s + blockIdx.x * ROW_THREADS + threadIdx.x;
    if (r < n) {
        double *w = W + static_cast<size_t>(jj) * ld;
        w[r] = fma(alpha, V[static_cast<size_t>(jj) * ld + r], w[r]);
    }
}

// A[r][c] -= sum_k (V[k][r] W[k][c] + W[k][r] V[k][c]) on the tiles (I, J >= I) of rows / columns [p1, n), k < nbp: the
// rank-2 nbp update of the upper triangle after a panel. 4 x 4 outputs per thread, k in steps of 16 through shared memory.
__global__ void __launch_bounds__(256) update_kernel(double *__restrict__ A, uint32_t ld, uint32_t n, uint32_t p1,
                                                     const double *__restrict__ V, const double *__restrict__ W, int nbp) {
    const uint32_t I = p1 / TT + blockIdx.y, J = p1 / TT + blockIdx.x;
    if (J < I) {
        return;
    }
    __shared__ double xr[16][TT], yc[16][TT];
    const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
    double acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a) {
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            acc[a][b] = 0.0;
        }
    }
    for (int k0 = 0; k0 < 2 * nbp; k0 += 16) {
        __syncthreads();
        for (int i = t; i < 16 * TT; i += 256) {
            const int kk = k0 + i / TT, x = i % TT;
            double a = 0.0, b = 0.0;
            if (kk < 2 * nbp) {
                // X = [V | W] on the rows of I, Y = [W | V] on the rows of J
                const double *xs = kk < nbp ? V + static_cast<size_t>(kk) * ld : W + static_cast<size_t>(kk - nbp) * ld;
                const double *ys = kk < nbp ? W + static_cast<size_t>(kk) * ld : V + static_cast<size_t>(kk - nbp) * ld;
                a = xs[I * TT + x];
                b = ys[J * TT + x];
            }
            xr[i / TT][x] = a;
            yc[i / TT][x] = b;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; ++kk) {
            double xv[4], yv[4];
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                xv[a] = xr[kk][ty + 16 * a];
                yv[a] = yc[kk][tx + 16 * a];
            }
#pragma unroll
            for (int a = 0; a < 4; ++a) {
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    acc[a][b] = fma(xv[a], yv[b], acc[a][b]);
                }
            }
        }
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const uint32_t r = I * TT + ty + 16 * a;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const uint32_t c = J * TT + tx + 16 * b;
            if (r >= p1 && r < n && c < n) {
                A[static_cast<size_t>(r) * ld + c] -= acc[a][b];
            }
        }
    }
}

// e2 = e^2, then pivmin and the Gershgorin interval of T (one thread: the host-checked code of sturm.hpp)
__global__ void sturm_setup_kernel(const double *__restrict__ d, const double *__restrict__ e, uint32_t n, double *__restrict__ e2,
                                   double *__restrict__ iv) {
    for (uint32_t i = threadIdx.x; i + 1 < n; i += blockDim.x) {
        e2[i] = e[i] * e[i];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const double pmin = sturm::pivmin(e2, n);
        const sturm::Interval g = sturm::gershgorin(d, e, n, pmin);
        iv[0] = g.lo;
        iv[1] = g.hi;
        iv[2] = g.atol;
        iv[3] = pmin;
    }
}

// eigenvalue k of T (ascending) per thread; out[n - 1 - k] = 1 - lambda_k, the eigenvalues of L ascending
__global__ void __launch_bounds__(128) bisect_kernel(const double *__restrict__ d, const double *__restrict__ e2, uint32_t n,
                                                     const double *__restrict__ iv, double *__restrict__ out) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) {
        return;
    }
    const sturm::Interval g{ iv[0], iv[1], iv[2] };
    out[n - 1 - k] = 1.0 - sturm::bisect(d, e2, n, k, g, iv[3]);
}

} // namespace

int sgpu_eigenvalues_device(sgpu_ctx *ctx, const double *d_A, uint32_t n, double *h_evals, sgpu_eigenvalue_stats *stats) {
    cudaStream_t st = ctx->stream;
    if (n == 0 || !h_evals) {
        return sgpu_fail(ctx, SGPU_E_ARG, "eigenvalues: empty matrix or no output");
    }
    struct Events { // destroyed on every return path
        cudaEvent_t e[4] = { nullptr, nullptr, nullptr, nullptr };
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
    const uint64_t launches0 = ctx->launches;
    SGPU_CUDA(ctx, cudaEventRecord(evs.e[0], st));
    const uint32_t ld = (n + EG_PAD - 1) / EG_PAD * EG_PAD;
    DevBuf<double> A;
    bool all_zero = false;
    SGPU_TRY(sgpu_scaled_similarity(ctx, d_A, n, ld, A, nullptr, &all_zero));
    if (stats) {
        std::memset(stats, 0, sizeof(*stats));
        const double m = n - 1.0;
        stats->bytes_matvec = static_cast<uint64_t>(8.0 * m * (m + 1.0) * (m + 2.0) / 6.0);
    }
    if (all_zero) { // L = I
        std::fill(h_evals, h_evals + n, 1.0);
        if (stats) {
            stats->launches = ctx->launches - launches0;
        }
        return SGPU_OK;
    }
    SGPU_CUDA(ctx, cudaEventRecord(evs.e[1], st));

    const uint32_t nt = ld / TT, n_chunk = (nt + SV_CH - 1) / SV_CH;
    const uint32_t max_dot = (n + DOT_ROWS - 1) / DOT_ROWS, max_w = (n + ROW_THREADS - 1) / ROW_THREADS;
    DevBuf<double> V, W, col, d, e, e2, scal, iv, ypart, zpart, dpart, wvpart, out;
    SGPU_CUDA(ctx, V.alloc(static_cast<size_t>(NB) * ld, ctx));
    SGPU_CUDA(ctx, W.alloc(static_cast<size_t>(NB) * ld, ctx));
    SGPU_CUDA(ctx, col.alloc(ld, ctx));
    SGPU_CUDA(ctx, d.alloc(ld, ctx));
    SGPU_CUDA(ctx, e.alloc(ld, ctx));
    SGPU_CUDA(ctx, e2.alloc(ld, ctx));
    SGPU_CUDA(ctx, scal.alloc(1, ctx));
    SGPU_CUDA(ctx, iv.alloc(4, ctx));
    SGPU_CUDA(ctx, ypart.alloc(static_cast<size_t>(n_chunk) * ld, ctx));
    SGPU_CUDA(ctx, zpart.alloc(static_cast<size_t>(nt) * ld, ctx));
    SGPU_CUDA(ctx, dpart.alloc(static_cast<size_t>(max_dot) * 2 * NB, ctx));
    SGPU_CUDA(ctx, wvpart.alloc(max_w, ctx));
    SGPU_CUDA(ctx, out.alloc(n, ctx));
    // rows of W outside [s, n) are never written by w_kernel; the trailing update reads (and masks) the padding rows
    SGPU_CUDA(ctx, cudaMemsetAsync(W.p, 0, W.n * sizeof(double), st));

    // ---- Householder reduction, panels of NB columns ----
    for (uint32_t p0 = 0; p0 < n; p0 += NB) {
        const int nbp = static_cast<int>(std::min<uint32_t>(NB, n - p0));
        for (int jj = 0; jj < nbp; ++jj) {
            const uint32_t j = p0 + jj;
            SGPU_LAUNCH(ctx, (col_update_kernel<<<(n - j + ROW_THREADS - 1) / ROW_THREADS, ROW_THREADS, 0, st>>>(A.p, ld, n, j, jj, V.p,
                                                                                                             W.p, col.p)));
            SGPU_LAUNCH(ctx, (reflector_kernel<<<1, 1024, 0, st>>>(col.p, ld, n, j, jj, V.p, d.p, e.p, scal.p)));
            if (j + 1 >= n) {
                break;
            }
            const uint32_t s = j + 1, tr = nt - s / TT; // trailing tile rows
            const double *v = V.p + static_cast<size_t>(jj) * ld;
            SGPU_LAUNCH(ctx, (symv_kernel<<<dim3((tr + SV_CH - 1) / SV_CH, tr), 256, 0, st>>>(A.p, ld, n, s, v, ypart.p, zpart.p)));
            const uint32_t n_dot = jj > 0 ? (n - s + DOT_ROWS - 1) / DOT_ROWS : 0;
            if (n_dot) {
                SGPU_LAUNCH(ctx, (dots_kernel<<<n_dot, 256, 0, st>>>(V.p, W.p, ld, n, s, jj, v, dpart.p)));
            }
            const uint32_t n_w = (n - s + ROW_THREADS - 1) / ROW_THREADS;
            SGPU_LAUNCH(ctx, (w_kernel<<<n_w, ROW_THREADS, 0, st>>>(ypart.p, zpart.p, ld, n, s, jj, dpart.p, n_dot, V.p, W.p, scal.p,
                                                                    wvpart.p)));
            SGPU_LAUNCH(ctx, (wfix_kernel<<<n_w, ROW_THREADS, 0, st>>>(ld, n, s, jj, V.p, W.p, scal.p, wvpart.p, n_w)));
        }
        const uint32_t p1 = p0 + nbp;
        if (p1 < n) {
            const uint32_t tr = nt - p1 / TT;
            SGPU_LAUNCH(ctx, (update_kernel<<<dim3(tr, tr), 256, 0, st>>>(A.p, ld, n, p1, V.p, W.p, nbp)));
        }
    }
    SGPU_CUDA(ctx, cudaGetLastError());
    SGPU_CUDA(ctx, cudaEventRecord(evs.e[2], st));

    // ---- bisection ----
    SGPU_LAUNCH(ctx, (sturm_setup_kernel<<<1, 256, 0, st>>>(d.p, e.p, n, e2.p, iv.p)));
    SGPU_LAUNCH(ctx, (bisect_kernel<<<(n + 127) / 128, 128, 0, st>>>(d.p, e2.p, n, iv.p, out.p)));
    SGPU_CUDA(ctx, cudaGetLastError());
    SGPU_CUDA(ctx, cudaEventRecord(evs.e[3], st));
    SGPU_CUDA(ctx, cudaMemcpyAsync(h_evals, out.p, static_cast<size_t>(n) * sizeof(double), cudaMemcpyDeviceToHost, st));
    SGPU_CUDA(ctx, cudaStreamSynchronize(st));
    if (stats) {
        stats->launches = ctx->launches - launches0;
        SGPU_CUDA(ctx, cudaEventElapsedTime(&stats->ms_laplacian, evs.e[0], evs.e[1]));
        SGPU_CUDA(ctx, cudaEventElapsedTime(&stats->ms_tridiagonal, evs.e[1], evs.e[2]));
        SGPU_CUDA(ctx, cudaEventElapsedTime(&stats->ms_bisection, evs.e[2], evs.e[3]));
    }
    return SGPU_OK;
}
