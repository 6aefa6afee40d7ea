// K6 — log-likelihood transform and normalisation.
//
//   logprob_kernel    LS / LD tables of similarity_matrix.cpp:117-170, one thread per (x_s, x_d),
//                     fp64, from power tables built by repeated multiplication exactly as the
//                     reference's Cache does (:76-103) and a uint64 Pascal triangle
//   transform_kernel  raw[i][j] = F(1,0) S + F(0,1) D + sum_classes G(s,d) H_sd (+ spill), mirrored,
//                     with a fused min/max reduction (similarity_matrix.cpp:428 + util/mat.hpp:35-53)
//   normalize_kernel  ADD_MIN / EXPONENTIATE / SCALE_MAX_1 and the zero diagonal (:271-293)
// Compiled with -fmad=false so that the table arithmetic rounds like the reference's x86 build.
#include "common.cuh"

#include <cfloat>
#include <cstring>
#include <cmath>
#include <vector>

namespace {

constexpr int TBL = LOGPROB_TBL; // power tables / Pascal rows kept (x_s + x_d <= 126 for classes < 64)

struct CacheTables {
    double pss[TBL], psd[TBL], pds[TBL], pdd[TBL];
    double p1he[TBL], p1he2[TBL], phe2[TBL], ph[TBL], pe[TBL], p05[TBL], psspds[TBL], psdpdd[TBL];
    uint32_t len;
};

void extend(double *a, uint32_t n) { // similarity_matrix.cpp:81
    for (uint32_t p = 2; p < n; ++p) {
        a[p] = a[p - 1] * a[1];
    }
}

void make_cache(CacheTables *c, double epsilon, double h, double theta, uint32_t max_read_size) {
    // similarity_matrix.cpp:42-67
    const double theta2 = theta * theta;
    const double p_same_diff = 2 * theta * (1 - theta) + 2 * theta2 / 3;
    const double p_same_same = 1 - p_same_diff;
    const double p_diff_same = 2 * (1 - theta) * theta / 3 + 2 * theta2 / 9;
    const double p_diff_diff = 1 - p_diff_same;
    const uint32_t n = logprob_table_len(max_read_size);
    c->len = n;
    auto init = [n](double *arr, double v) {
        arr[0] = 1;
        arr[1] = v;
        extend(arr, n);
    };
    init(c->pss, p_same_same);
    init(c->psd, p_same_diff);
    init(c->pds, p_diff_same);
    init(c->pdd, p_diff_diff);
    init(c->p1he, 1 - epsilon - h);
    init(c->p1he2, 1 - epsilon * 0.5 - h);
    init(c->phe2, h + epsilon * 0.5);
    init(c->ph, h);
    init(c->pe, epsilon);
    init(c->p05, 0.5);
    init(c->psspds, p_same_same + p_diff_same);
    init(c->psdpdd, p_same_diff + p_diff_diff);
}

__global__ void pascal_kernel(uint64_t *__restrict__ comb) { // single thread block, row by row
    for (int r = 0; r < TBL; ++r) {
        for (int i = threadIdx.x; i < TBL; i += blockDim.x) {
            uint64_t v = 0;
            if (i == 0 || i == r) {
                v = 1;
            } else if (i < r) {
                v = comb[(r - 1) * TBL + i - 1] + comb[(r - 1) * TBL + i]; // wraps like the reference's uint64
            }
            comb[r * TBL + i] = v;
        }
        __syncthreads();
    }
}

// one thread per (x_s, x_d)
__global__ void logprob_kernel(const CacheTables *__restrict__ cp, const uint64_t *__restrict__ comb, uint32_t n,
                               uint32_t L, double *__restrict__ ls_out, double *__restrict__ ld_out) {
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n * n) {
        return;
    }
    const uint32_t x_s = idx / n, x_d = idx % n;
    const CacheTables &c = *cp;
    if (x_s + x_d >= c.len || x_s >= L || x_d >= L) { // the reference's tables end here
        ls_out[idx] = nan("");
        ld_out[idx] = nan("");
        return;
    }
#define COMB(r, i) comb[(r) * TBL + (i)]
    // similarity_matrix.cpp:153-170
    double p = 0;
    for (uint32_t k = 0; k <= x_s; ++k) {
        for (uint32_t l = 0; l <= x_d; ++l) {
            const uint64_t cc = COMB(x_s, k) * COMB(x_d, l);
            p += cc * c.p1he2[k + l] * 0.5 * (c.pss[k] * c.psd[l] + c.pds[k] * c.pdd[l]) * c.phe2[x_s + x_d - k - l]
                    * c.pss[x_s - k] * c.psd[x_d - l];
        }
    }
    p *= COMB(x_s + x_d, x_s);
    ls_out[idx] = log(p);
    // similarity_matrix.cpp:117-141
    double prob = 0;
    for (uint32_t k = 0; k <= x_s; ++k) {
        for (uint32_t l = 0; l <= x_d; ++l) {
            for (uint32_t pp = 0; pp <= x_s - k; ++pp) {
                for (uint32_t q = 0; q <= x_d - l; ++q) {
                    const uint64_t cc = COMB(x_s, k) * COMB(x_d, l) * COMB(x_s - k, pp) * COMB(x_d - l, q);
                    const uint32_t rest = x_s + x_d - k - l - pp - q;
                    prob += cc * c.p1he[k + l] * 0.5 * (c.pss[k] * c.psd[l] + c.pds[k] * c.pdd[l]) * c.pe[rest]
                            * c.p05[rest] * c.psspds[x_s - k - pp] * c.psdpdd[x_d - l - q] * c.ph[pp + q] * c.pss[pp]
                            * c.psd[q];
                }
            }
        }
    }
    prob *= COMB(x_s + x_d, x_s);
    ld_out[idx] = log(prob);
#undef COMB
}

// F = LD - LS; G(s,d) = F(s,d) - s F(1,0) - d F(0,1)
__global__ void gtable_kernel(const double *__restrict__ ls, const double *__restrict__ ld, uint32_t n,
                              double *__restrict__ G, double *__restrict__ F) {
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= SGPU_MAX_CLASS * SGPU_MAX_CLASS) {
        return;
    }
    const uint32_t s = idx / SGPU_MAX_CLASS, d = idx % SGPU_MAX_CLASS;
    double f = nan(""), g = nan("");
    if (s < n && d < n) {
        f = ld[s * n + d] - ls[s * n + d];
        const double f10 = n > 1 ? ld[1 * n + 0] - ls[1 * n + 0] : 0.0;
        const double f01 = n > 1 ? ld[0 * n + 1] - ls[0 * n + 1] : 0.0;
        g = f - s * f10 - d * f01;
    }
    G[idx] = g;
    if (F) {
        F[idx] = f;
    }
}

// ordered-int encoding so that atomicMin/atomicMax on uint64 order doubles
__device__ __forceinline__ unsigned long long enc(double x) {
    unsigned long long u = static_cast<unsigned long long>(__double_as_longlong(x));
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__host__ inline double dec(unsigned long long u) {
    unsigned long long v = (u >> 63) ? (u & 0x7FFFFFFFFFFFFFFFull) : ~u;
    double d;
    memcpy(&d, &v, sizeof(d));
    return d;
}

struct TransformArgs {
    const int32_t *i32;
    const double *spill;
    uint32_t n;
    uint64_t nn;
    int planes_used;
    double f10, f01;
    double g2[3], g3[4];
};

constexpr int TR_THREADS = 256;

// raw[i][j] = F(1,0) S + F(0,1) D + sum G(s,d) N_sd  (the upper triangle of mat_diff - mat_same)
__device__ __forceinline__ double raw_value(const TransformArgs &a, uint64_t idx) {
    double v = a.f10 * a.i32[PLANE_S * a.nn + idx] + a.f01 * a.i32[PLANE_D * a.nn + idx];
    if (a.planes_used > 2) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const int32_t h = a.i32[(PLANE_H2 + k) * a.nn + idx];
            if (h) {
                v += a.g2[k] * h;
            }
        }
    }
    if (a.planes_used > PLANE_H3) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int32_t h = a.i32[(PLANE_H3 + k) * a.nn + idx];
            if (h) {
                v += a.g3[k] * h;
            }
        }
    }
    if (a.spill) {
        v += a.spill[idx];
    }
    return v;
}

// max (and min) of the raw matrix over the upper triangle; the zero diagonal counts, util/mat.hpp:35-53
// scans the whole matrix. One CTA per 32 x 32 tile of the upper triangle of tiles.
__global__ void __launch_bounds__(TR_THREADS) minmax_kernel(TransformArgs a, const uint2 *__restrict__ tiles,
                                                           unsigned long long *__restrict__ minmax) {
    const uint2 t = tiles[blockIdx.x];
    const uint32_t tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    double mn = 0.0, mx = 0.0; // the diagonal
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t i = t.x * 32 + ty + 8 * k, j = t.y * 32 + tx;
        if (i < j && j < a.n) {
            const double v = raw_value(a, static_cast<uint64_t>(i) * a.n + j);
            mn = fmin(mn, v);
            mx = fmax(mx, v);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    __shared__ double s_mn[TR_THREADS / 32], s_mx[TR_THREADS / 32];
    if (tx == 0) {
        s_mn[ty] = mn;
        s_mx[ty] = mx;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < TR_THREADS / 32; ++w) {
            mn = fmin(mn, s_mn[w]);
            mx = fmax(mx, s_mx[w]);
        }
        atomicMin(&minmax[0], enc(mn));
        atomicMax(&minmax[1], enc(mx));
    }
}

__device__ __forceinline__ double dec_dev(unsigned long long u) {
    const unsigned long long v = (u >> 63) ? (u & 0x7FFFFFFFFFFFFFFFull) : ~u;
    return __longlong_as_double(static_cast<long long>(v));
}

// similarity_matrix.cpp:271-293 on one element
__device__ __forceinline__ double normalized(double v, int normalization, double mx) {
    switch (normalization) {
        case SGPU_NORM_ADD_MIN: // M *= -1; M += |min(M)|   (min(-raw) = -max(raw))
            v = v * -1;
            v += fabs(-mx);
            break;
        case SGPU_NORM_EXPONENTIATE:
            v = 1. / (exp(v) + 1);
            break;
        case SGPU_NORM_SCALE_MAX_1:
            v = v * (1. / mx);
            break;
    }
    return v;
}

// The whole output in one pass: every 32 x 32 tile of the upper triangle is evaluated once, normalised,
// written as rows (i, j..) and, through a shared-memory transpose, as rows (j, i..) of the mirror
// image; the diagonal is zero (fill_diagonal(0), :292).
__global__ void __launch_bounds__(TR_THREADS) finalize_kernel(TransformArgs a, const uint2 *__restrict__ tiles,
                                                             const unsigned long long *__restrict__ minmax,
                                                             int normalization, double *__restrict__ out) {
    __shared__ double tile[32][33];
    const uint2 t = tiles[blockIdx.x];
    const uint32_t tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const double mx = dec_dev(minmax[1]);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t r = ty + 8 * k;
        const uint32_t i = t.x * 32 + r, j = t.y * 32 + tx;
        double v = 0.0;
        if (i < j && j < a.n) {
            v = normalized(raw_value(a, static_cast<uint64_t>(i) * a.n + j), normalization, mx);
        }
        tile[r][tx] = v;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t r = ty + 8 * k;
        // rows of the tile itself
        uint32_t i = t.x * 32 + r, j = t.y * 32 + tx;
        if (i < a.n && j < a.n) {
            if (i < j) {
                out[static_cast<uint64_t>(i) * a.n + j] = tile[r][tx];
            } else if (t.x == t.y) { // diagonal tile: zero diagonal, lower half mirrored
                out[static_cast<uint64_t>(i) * a.n + j] = i == j ? 0.0 : tile[tx][r];
            }
        }
        // rows of the mirrored tile
        if (t.x != t.y) {
            i = t.y * 32 + r;
            j = t.x * 32 + tx;
            if (i < a.n && j < a.n) {
                out[static_cast<uint64_t>(i) * a.n + j] = tile[tx][r];
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Multi-GPU epilogue over peer memory: reduce-scatter and log-likelihood transform in ONE kernel.
// Every GPU owns a contiguous share of the 32 x 32 tiles of the upper triangle. For its tiles it reads the
// count planes of ALL GPUs (its own and, through NVLink peer mappings, the others'), adds them and applies the
// transform: the summed integers never exist in memory and nothing travels but the operands themselves
// (each element of every GPU's planes crosses NVLink at most once). The raw values stay in a local buffer;
// after the ranks have exchanged max(raw) (one scalar) the second kernel normalises and writes each tile and
// its mirror image to the output, which may be mapped host memory (every GPU writes its share of the matrix
// over its own PCIe link).
// ------------------------------------------------------------------------------------------------
struct SlabArgs {
    const int32_t *peer[SGPU_MAX_PEERS];
    const double *spill[SGPU_MAX_PEERS]; // fp64 spill planes of the GPUs (overlaps at >= 4 loci), null where there is none
    uint32_t n_peers;
    uint32_t n;
    uint64_t nn;
    int planes_used;
    double f10, f01;
    double g2[3], g3[4];
};

// tile number t of the upper triangle of nb x nb tiles (row-major over bj >= bi) -> (bi, bj)
__device__ __forceinline__ uint2 tri_tile(uint64_t t, uint32_t nb) {
    // rows before bi hold bi * nb - bi (bi - 1) / 2 tiles; solve by the quadratic formula, then fix up
    const double b = 2.0 * nb + 1.0;
    uint32_t bi = static_cast<uint32_t>((b - sqrt(b * b - 8.0 * static_cast<double>(t))) * 0.5);
    auto before = [nb](uint32_t r) { return static_cast<uint64_t>(r) * nb - static_cast<uint64_t>(r) * (r - 1) / 2; };
    while (bi > 0 && before(bi) > t) {
        --bi;
    }
    while (before(bi + 1) <= t) {
        ++bi;
    }
    return make_uint2(bi, bi + static_cast<uint32_t>(t - before(bi)));
}

__global__ void __launch_bounds__(TR_THREADS) slab_raw_kernel(SlabArgs a, uint64_t t0, uint32_t nb, double *__restrict__ raw,
                                                             unsigned long long *__restrict__ minmax) {
    const uint2 t = tri_tile(t0 + blockIdx.x, nb);
    const uint32_t tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    double mn = 0.0, mx = 0.0; // the diagonal
    double *dst = raw + static_cast<uint64_t>(blockIdx.x) * 1024;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t r = ty + 8 * k;
        const uint32_t i = t.x * 32 + r, j = t.y * 32 + tx;
        double v = 0.0;
        if (i < j && j < a.n) {
            const uint64_t idx = static_cast<uint64_t>(i) * a.n + j;
            int32_t acc[N_PLANES];
#pragma unroll
            for (int pl = 0; pl < N_PLANES; ++pl) {
                acc[pl] = 0;
            }
            for (uint32_t q = 0; q < a.n_peers; ++q) { // integer sums: the order of the GPUs does not matter
                const int32_t *pp = a.peer[q] + idx;
                acc[PLANE_S] += pp[PLANE_S * a.nn];
                acc[PLANE_D] += pp[PLANE_D * a.nn];
                if (a.planes_used > 2) {
#pragma unroll
                    for (int pl = PLANE_H2; pl < PLANE_H3; ++pl) {
                        acc[pl] += pp[pl * a.nn];
                    }
                }
                if (a.planes_used > PLANE_H3) {
#pragma unroll
                    for (int pl = PLANE_H3; pl < N_PLANES; ++pl) {
                        acc[pl] += pp[pl * a.nn];
                    }
                }
            }
            // same expression, in the same order, as raw_value() of the single-GPU epilogue: identical bits
            v = a.f10 * acc[PLANE_S] + a.f01 * acc[PLANE_D];
            if (a.planes_used > 2) {
#pragma unroll
                for (int kk = 0; kk < 3; ++kk) {
                    if (acc[PLANE_H2 + kk]) {
                        v += a.g2[kk] * acc[PLANE_H2 + kk];
                    }
                }
            }
            if (a.planes_used > PLANE_H3) {
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    if (acc[PLANE_H3 + kk]) {
                        v += a.g3[kk] * acc[PLANE_H3 + kk];
                    }
                }
            }
            for (uint32_t q = 0; q < a.n_peers; ++q) { // fixed order: every rank would add them in the same one
                if (a.spill[q]) {
                    v += a.spill[q][idx];
                }
            }
            mn = fmin(mn, v);
            mx = fmax(mx, v);
        }
        dst[r * 32 + tx] = v;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    __shared__ double s_mn[TR_THREADS / 32], s_mx[TR_THREADS / 32];
    if (tx == 0) {
        s_mn[ty] = mn;
        s_mx[ty] = mx;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < TR_THREADS / 32; ++w) {
            mn = fmin(mn, s_mn[w]);
            mx = fmax(mx, s_mx[w]);
        }
        atomicMin(&minmax[0], enc(mn));
        atomicMax(&minmax[1], enc(mx));
    }
}

// {-min, max} of this GPU's share as doubles: ONE all-reduce with MAX over the ranks gives both global extrema
__global__ void slab_extrema_kernel(const unsigned long long *__restrict__ minmax, double *__restrict__ ext) {
    ext[0] = -dec_dev(minmax[0]);
    ext[1] = dec_dev(minmax[1]);
}

__global__ void __launch_bounds__(TR_THREADS) slab_finalize_kernel(const double *__restrict__ raw, uint64_t t0, uint32_t nb, uint32_t n,
                                                                  const double *__restrict__ ext, int normalization,
                                                                  double *__restrict__ out) {
    __shared__ double tile[32][33];
    const uint2 t = tri_tile(t0 + blockIdx.x, nb);
    const uint32_t tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const double mx = ext[1];
    const double *src = raw + static_cast<uint64_t>(blockIdx.x) * 1024;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t r = ty + 8 * k;
        const uint32_t i = t.x * 32 + r, j = t.y * 32 + tx;
        double v = 0.0;
        if (i < j && j < n) {
            v = normalized(src[r * 32 + tx], normalization, mx);
        }
        tile[r][tx] = v;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t r = ty + 8 * k;
        uint32_t i = t.x * 32 + r, j = t.y * 32 + tx;
        if (i < n && j < n) {
            if (i < j) {
                out[static_cast<uint64_t>(i) * n + j] = tile[r][tx];
            } else if (t.x == t.y) { // diagonal tile: zero diagonal, lower half mirrored
                out[static_cast<uint64_t>(i) * n + j] = i == j ? 0.0 : tile[tx][r];
            }
        }
        if (t.x != t.y) { // rows of the mirrored tile
            i = t.y * 32 + r;
            j = t.x * 32 + tx;
            if (i < n && j < n) {
                out[static_cast<uint64_t>(i) * n + j] = tile[tx][r];
            }
        }
    }
}

int device_log_probs(sgpu_ctx *ctx, double eps, double h, double theta, uint32_t L, uint32_t n, DevBuf<double> &ls,
                     DevBuf<double> &ld) {
    cudaStream_t st = ctx->stream;
    CacheTables hc;
    make_cache(&hc, eps, h, theta, L);
    DevBuf<CacheTables> dc;
    DevBuf<uint64_t> comb;
    SGPU_CUDA(ctx, dc.alloc(1, ctx));
    SGPU_CUDA(ctx, comb.alloc(TBL * TBL, ctx));
    SGPU_CUDA(ctx, ls.alloc(static_cast<size_t>(n) * n, ctx));
    SGPU_CUDA(ctx, ld.alloc(static_cast<size_t>(n) * n, ctx));
    SGPU_CUDA(ctx, cudaMemcpyAsync(dc.p, &hc, sizeof(hc), cudaMemcpyHostToDevice, st));
    SGPU_CUDA(ctx, cudaStreamSynchronize(st)); SGPU_LAUNCH(ctx, (// hc lives on this stack frame
    pascal_kernel<<<1, 128, 0, st>>>(comb.p)));
    SGPU_LAUNCH(ctx, (logprob_kernel<<<(n * n + 63) / 64, 64, 0, st>>>(dc.p, comb.p, n, L, ls.p, ld.p)));
    SGPU_CUDA(ctx, cudaGetLastError());
    SGPU_CUDA(ctx, cudaStreamSynchronize(st));
    return SGPU_OK;
}

} // namespace

int sgpu_log_probs_impl(sgpu_ctx *ctx, double eps, double h, double theta, uint32_t L, uint32_t n, double *h_ls,
                        double *h_ld) {
    if (n == 0 || n > SGPU_MAX_CLASS) {
        return sgpu_fail(ctx, SGPU_E_ARG, "n must be 1..%d", SGPU_MAX_CLASS);
    }
    DevBuf<double> ls, ld;
    SGPU_TRY(device_log_probs(ctx, eps, h, theta, L, n, ls, ld));
    SGPU_CUDA(ctx, cudaMemcpyAsync(h_ls, ls.p, sizeof(double) * n * n, cudaMemcpyDeviceToHost, ctx->stream));
    SGPU_CUDA(ctx, cudaMemcpyAsync(h_ld, ld.p, sizeof(double) * n * n, cudaMemcpyDeviceToHost, ctx->stream));
    SGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SGPU_OK;
}

int sgpu_build_gtable(sgpu_ctx *ctx, double eps, double h, double theta, uint32_t L, uint32_t n, double *d_G,
                      double *d_F) {
    DevBuf<double> ls, ld;
    SGPU_TRY(device_log_probs(ctx, eps, h, theta, L, n, ls, ld));
    SGPU_LAUNCH(ctx, (gtable_kernel<<<(SGPU_MAX_CLASS * SGPU_MAX_CLASS + 255) / 256, 256, 0, ctx->stream>>>(ls.p, ld.p, n, d_G, d_F)));
    SGPU_CUDA(ctx, cudaGetLastError());
    SGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SGPU_OK;
}

int sgpu_output_wait_impl(sgpu_ctx *ctx) {
    if (ctx->pending_out) {
        SGPU_CUDA(ctx, cudaEventSynchronize(ctx->out_done));
        // the block's last user ran on the download stream and has finished: safe to hand out again
        sgpu_dev_free(ctx, ctx->pending_out);
        ctx->pending_out = nullptr;
    }
    return SGPU_OK;
}

// F and G for the classes of the integer planes (s + d <= 3); kept for the next call with the same
// likelihood parameters (divide_cluster calls with the same ones at every node of its recursion)
static int ensure_ftable(sgpu_ctx *ctx, uint32_t L, double eps, double h, double theta) {
    cudaStream_t st = ctx->stream;
    if (!(ctx->ft_valid && ctx->ft_eps == eps && ctx->ft_h == h && ctx->ft_theta == theta && ctx->ft_L == L)) {
        DevBuf<double> d_G, d_F;
        SGPU_CUDA(ctx, d_G.alloc(SGPU_MAX_CLASS * SGPU_MAX_CLASS, ctx));
        SGPU_CUDA(ctx, d_F.alloc(SGPU_MAX_CLASS * SGPU_MAX_CLASS, ctx));
        SGPU_TRY(sgpu_build_gtable(ctx, eps, h, theta, L, 4, d_G.p, d_F.p));
        std::vector<double> G(SGPU_MAX_CLASS * SGPU_MAX_CLASS), F(SGPU_MAX_CLASS * SGPU_MAX_CLASS);
        SGPU_CUDA(ctx, cudaMemcpyAsync(G.data(), d_G.p, G.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
        SGPU_CUDA(ctx, cudaMemcpyAsync(F.data(), d_F.p, F.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
        SGPU_CUDA(ctx, cudaStreamSynchronize(st));
        ctx->ft_f10 = F[1 * SGPU_MAX_CLASS + 0];
        ctx->ft_f01 = F[0 * SGPU_MAX_CLASS + 1];
        for (int d = 0; d < 3; ++d) {
            ctx->ft_g2[d] = G[(2 - d) * SGPU_MAX_CLASS + d];
        }
        for (int d = 0; d < 4; ++d) {
            ctx->ft_g3[d] = G[(3 - d) * SGPU_MAX_CLASS + d];
        }
        ctx->ft_eps = eps;
        ctx->ft_h = h;
        ctx->ft_theta = theta;
        ctx->ft_L = L;
        ctx->ft_valid = true;
    }
    return SGPU_OK;
}

int sgpu_epilogue(sgpu_ctx *ctx, sgpu_counts *c, uint32_t L, double eps, double h, double theta, int normalization,
                  double *h_out, double **d_keep, bool async_out) {
    cudaStream_t st = ctx->stream;
    if (normalization < 0 || normalization > 2) {
        return sgpu_fail(ctx, SGPU_E_ARG, "Invalid normalization: %d", normalization); // similarity_matrix.cpp:264
    }
    if (c->nn == 0) {
        return SGPU_OK;
    }
    SGPU_TRY(ensure_ftable(ctx, L, eps, h, theta));
    TransformArgs a;
    a.i32 = c->i32;
    a.spill = c->spill;
    a.n = c->n;
    a.nn = c->nn;
    a.planes_used = c->planes_used;
    a.f10 = ctx->ft_f10;
    a.f01 = ctx->ft_f01;
    for (int d = 0; d < 3; ++d) {
        // NaN: class impossible with this max_fragment_length; its plane is all zero
        a.g2[d] = std::isnan(ctx->ft_g2[d]) ? 0.0 : ctx->ft_g2[d];
    }
    for (int d = 0; d < 4; ++d) {
        a.g3[d] = std::isnan(ctx->ft_g3[d]) ? 0.0 : ctx->ft_g3[d];
    }
    // 32 x 32 tiles of the upper triangle (list kept on the device per matrix size)
    const uint32_t nb = (c->n + 31) / 32;
    const uint32_t n_tiles = nb * (nb + 1) / 2;
    if (!(ctx->ep_tiles && ctx->ep_tiles_n == c->n)) {
        std::vector<uint2> tiles;
        tiles.reserve(n_tiles);
        for (uint32_t bi = 0; bi < nb; ++bi) {
            for (uint32_t bj = bi; bj < nb; ++bj) {
                tiles.push_back(make_uint2(bi, bj));
            }
        }
        if (ctx->ep_tiles) {
            SGPU_CUDA(ctx, cudaStreamSynchronize(st));
            SGPU_CUDA(ctx, cudaFree(ctx->ep_tiles));
            ctx->ep_tiles = nullptr;
        }
        SGPU_CUDA(ctx, cudaMalloc(&ctx->ep_tiles, tiles.size() * sizeof(uint2)));
        SGPU_CUDA(ctx, cudaMemcpy(ctx->ep_tiles, tiles.data(), tiles.size() * sizeof(uint2), cudaMemcpyHostToDevice));
        ctx->ep_tiles_n = c->n;
    }
    const uint2 *d_tiles = static_cast<const uint2 *>(ctx->ep_tiles);
    DevBuf<double> out;
    DevBuf<unsigned long long> d_minmax;
    SGPU_CUDA(ctx, out.alloc(c->nn, ctx));
    SGPU_CUDA(ctx, d_minmax.alloc(2, ctx));
    // min starts at +inf, max at -inf in the ordered encoding; both kernels also see the zero diagonal
    SGPU_CUDA(ctx, cudaMemsetAsync(d_minmax.p, 0xFF, sizeof(unsigned long long), st));
    SGPU_CUDA(ctx, cudaMemsetAsync(d_minmax.p + 1, 0x00, sizeof(unsigned long long), st));
    if (normalization != SGPU_NORM_EXPONENTIATE) { // the only normalisation that does not need max(M)
        SGPU_LAUNCH(ctx, (minmax_kernel<<<n_tiles, TR_THREADS, 0, st>>>(a, d_tiles, d_minmax.p)));
    }
    SGPU_LAUNCH(ctx, (finalize_kernel<<<n_tiles, TR_THREADS, 0, st>>>(a, d_tiles, d_minmax.p, normalization, out.p)));
    SGPU_CUDA(ctx, cudaGetLastError());
    if (h_out && async_out) {
        // download on a stream of its own, behind the kernels above; the caller collects it with sgpu_output_wait
        SGPU_TRY(sgpu_output_wait_impl(ctx));
        if (!ctx->d2h_stream) {
            SGPU_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->d2h_stream, cudaStreamNonBlocking));
            SGPU_CUDA(ctx, cudaEventCreateWithFlags(&ctx->out_done, cudaEventDisableTiming));
        }
        cudaEvent_t ev;
        SGPU_CUDA(ctx, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        SGPU_CUDA(ctx, cudaEventRecord(ev, st));
        SGPU_CUDA(ctx, cudaStreamWaitEvent(ctx->d2h_stream, ev, 0));
        SGPU_CUDA(ctx, cudaEventDestroy(ev));
        SGPU_CUDA(ctx, cudaMemcpyAsync(h_out, out.p, c->nn * sizeof(double), cudaMemcpyDeviceToHost, ctx->d2h_stream));
        SGPU_CUDA(ctx, cudaEventRecord(ctx->out_done, ctx->d2h_stream));
        ctx->pending_out = out.take();
        return SGPU_OK;
    }
    if (h_out) { // NULL: leave the result on the device (timing of the device-resident path)
        SGPU_CUDA(ctx, cudaMemcpyAsync(h_out, out.p, c->nn * sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    SGPU_CUDA(ctx, cudaStreamSynchronize(st));
    if (d_keep) {
        *d_keep = out.take();
    }
    return SGPU_OK;
}

// ---- multi-GPU epilogue over peer memory (see slab_raw_kernel) ---------------------------------------------------
int sgpu_slab_raw_impl(sgpu_ctx *ctx, sgpu_counts *c, const int32_t *const *peer_planes, const double *const *peer_spill,
                       uint32_t n_peers, uint32_t slab, uint32_t n_slabs, uint32_t L, double eps, double h, double theta,
                       double **d_extrema) {
    cudaStream_t st = ctx->stream;
    if (n_peers == 0 || n_peers > SGPU_MAX_PEERS || n_slabs == 0 || slab >= n_slabs) {
        return sgpu_fail(ctx, SGPU_E_ARG, "slab epilogue: %u peers (1..%d), slab %u of %u", n_peers, SGPU_MAX_PEERS, slab, n_slabs);
    }
    if (c->spill && !peer_spill) {
        return sgpu_fail(ctx, SGPU_E_ARG, "slab epilogue: this GPU holds a spill plane (overlaps at >= 4 loci); pass the spill planes of all GPUs");
    }
    SGPU_TRY(ensure_ftable(ctx, L, eps, h, theta));
    SlabArgs a;
    for (uint32_t q = 0; q < SGPU_MAX_PEERS; ++q) {
        a.peer[q] = q < n_peers ? peer_planes[q] : nullptr;
        a.spill[q] = (peer_spill && q < n_peers) ? peer_spill[q] : nullptr;
    }
    a.n_peers = n_peers;
    a.n = c->n;
    a.nn = c->nn;
    a.planes_used = c->planes_used;
    a.f10 = ctx->ft_f10;
    a.f01 = ctx->ft_f01;
    for (int d = 0; d < 3; ++d) {
        a.g2[d] = std::isnan(ctx->ft_g2[d]) ? 0.0 : ctx->ft_g2[d];
    }
    for (int d = 0; d < 4; ++d) {
        a.g3[d] = std::isnan(ctx->ft_g3[d]) ? 0.0 : ctx->ft_g3[d];
    }
    const uint32_t nb = (c->n + 31) / 32;
    const uint64_t n_tiles = static_cast<uint64_t>(nb) * (nb + 1) / 2;
    // equal numbers of tiles per slab: equal work and equal NVLink traffic for every GPU
    c->slab_t0 = n_tiles * slab / n_slabs;
    c->slab_t1 = n_tiles * (slab + 1) / n_slabs;
    c->slab_nb = nb;
    const uint64_t mine = c->slab_t1 - c->slab_t0;
    if (c->slab_raw_tiles < mine) {
        sgpu_dev_free(ctx, c->slab_raw);
        c->slab_raw = nullptr;
        SGPU_CUDA(ctx, sgpu_dev_alloc(ctx, reinterpret_cast<void **>(&c->slab_raw), std::max<uint64_t>(mine, 1) * 1024 * sizeof(double)));
        c->slab_raw_tiles = mine;
    }
    if (!c->slab_minmax) {
        SGPU_CUDA(ctx, cudaMalloc(&c->slab_minmax, 2 * sizeof(unsigned long long) + 2 * sizeof(double)));
    }
    double *ext = reinterpret_cast<double *>(c->slab_minmax + 2);
    SGPU_CUDA(ctx, cudaMemsetAsync(c->slab_minmax, 0xFF, sizeof(unsigned long long), st));
    SGPU_CUDA(ctx, cudaMemsetAsync(c->slab_minmax + 1, 0x00, sizeof(unsigned long long), st));
    if (mine) {
        SGPU_LAUNCH(ctx, (slab_raw_kernel<<<static_cast<unsigned>(mine), TR_THREADS, 0, st>>>(a, c->slab_t0, nb, c->slab_raw, c->slab_minmax)));
    } else { // a GPU without tiles still contributes the zero diagonal
        const unsigned long long z = 0x8000000000000000ull;
        SGPU_CUDA(ctx, cudaMemcpyAsync(c->slab_minmax, &z, sizeof(z), cudaMemcpyHostToDevice, st));
        SGPU_CUDA(ctx, cudaMemcpyAsync(c->slab_minmax + 1, &z, sizeof(z), cudaMemcpyHostToDevice, st));
        SGPU_CUDA(ctx, cudaStreamSynchronize(st));
    }
    SGPU_LAUNCH(ctx, (slab_extrema_kernel<<<1, 1, 0, st>>>(c->slab_minmax, ext)));
    SGPU_CUDA(ctx, cudaGetLastError());
    if (d_extrema) {
        *d_extrema = ext;
    }
    return SGPU_OK;
}

int sgpu_slab_finalize_impl(sgpu_ctx *ctx, sgpu_counts *c, int normalization, double *out, double **d_out) {
    cudaStream_t st = ctx->stream;
    if (normalization < 0 || normalization > 2) {
        return sgpu_fail(ctx, SGPU_E_ARG, "Invalid normalization: %d", normalization);
    }
    if (!c->slab_minmax) {
        return sgpu_fail(ctx, SGPU_E_ARG, "sgpu_slab_finalize without sgpu_slab_raw");
    }
    if (!out) { // keep this GPU's share on the device, in an n x n matrix of which only its tiles (and their mirror images) are written
        if (!c->slab_out) {
            SGPU_CUDA(ctx, cudaMalloc(&c->slab_out, std::max<uint64_t>(1, c->nn) * sizeof(double)));
        }
        out = c->slab_out;
    }
    const uint64_t mine = c->slab_t1 - c->slab_t0;
    if (mine) {
        SGPU_LAUNCH(ctx, (slab_finalize_kernel<<<static_cast<unsigned>(mine), TR_THREADS, 0, st>>>(
                                 c->slab_raw, c->slab_t0, c->slab_nb, c->n, reinterpret_cast<const double *>(c->slab_minmax + 2), normalization, out)));
        SGPU_CUDA(ctx, cudaGetLastError());
    }
    if (d_out) {
        *d_out = out;
    }
    return SGPU_OK;
}
