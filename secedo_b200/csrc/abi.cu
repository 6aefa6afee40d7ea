// C ABI entry points (include/secedo_b200.h) and the orchestration of the kernels.
#include "common.cuh"

#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <vector>

int sgpu_fail(sgpu_ctx *ctx, int code, const char *fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx) {
        ctx->error = buf;
    }
    return code;
}

void sgpu_trace_point(sgpu_ctx *ctx, const char *what) {
    cudaStreamSynchronize(ctx->stream);
    const double now = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
    fprintf(stderr, "[sgpu trace] %-28s %8.3f ms\n", what, ctx->trace_t0 == 0.0 ? 0.0 : now - ctx->trace_t0);
    ctx->trace_t0 = now;
}

// ---- device memory cache -------------------------------------------------------------------------
cudaError_t sgpu_dev_alloc(sgpu_ctx *ctx, void **p, size_t bytes) {
    // size classes with 3 mantissa bits (<= 12.5 % slack): the same logical buffer keeps landing in the
    // same class although its exact size changes from call to call, so the cache stops growing after
    // the first pass over a workload
    bytes = std::max<size_t>(bytes, 256);
    int top = 63;
    while (!(bytes >> top)) {
        --top;
    }
    const size_t gran = std::max<size_t>(256, static_cast<size_t>(1) << (top > 3 ? top - 3 : 0));
    bytes = (bytes + gran - 1) / gran * gran;
    auto it = ctx->free_blocks.lower_bound(bytes);
    if (it != ctx->free_blocks.end() && it->first <= 2 * bytes) {
        *p = it->second;
        ctx->live_blocks.emplace(it->second, it->first);
        ctx->cached_bytes -= it->first;
        ctx->free_blocks.erase(it);
        return cudaSuccess;
    }
    if (ctx->trace_alloc) {
        fprintf(stderr, "[sgpu trace] cudaMalloc %.1f MB (cache holds %.1f MB in %zu blocks)\n", bytes / 1048576.0,
                ctx->cached_bytes / 1048576.0, ctx->free_blocks.size());
    }
    cudaError_t e = cudaMalloc(p, bytes);
    if (e == cudaErrorMemoryAllocation) { // out of memory: give the cached blocks back and retry
        cudaGetLastError();
        sgpu_dev_release_cache(ctx);
        e = cudaMalloc(p, bytes);
    }
    if (e == cudaSuccess) {
        ctx->live_blocks.emplace(*p, bytes);
    }
    return e;
}

void sgpu_dev_free(sgpu_ctx *ctx, void *p) {
    if (!p) {
        return;
    }
    if (ctx) {
        auto it = ctx->live_blocks.find(p);
        if (it != ctx->live_blocks.end()) {
            // everything that uses the block is already queued on ctx->stream, and so will be its next user
            ctx->free_blocks.emplace(it->second, p);
            ctx->cached_bytes += it->second;
            ctx->live_blocks.erase(it);
            return;
        }
        cudaStreamSynchronize(ctx->stream);
    }
    cudaFree(p);
}

void sgpu_dev_release_cache(sgpu_ctx *ctx) {
    cudaStreamSynchronize(ctx->stream);
    for (auto &b : ctx->free_blocks) {
        cudaFree(b.second);
    }
    ctx->free_blocks.clear();
    ctx->cached_bytes = 0;
}

namespace {

// upper triangle (i < j) of `planes` N x N planes <-> rows packed back to back
template <bool PACK>
__global__ void __launch_bounds__(256) tri_pack_kernel(int32_t *__restrict__ planes, int32_t *__restrict__ packed, uint32_t n,
                                                       uint32_t n_planes) {
    const uint64_t nn = static_cast<uint64_t>(n) * n, tri = static_cast<uint64_t>(n) * (n - 1) / 2;
    for (uint64_t row = blockIdx.x; row < static_cast<uint64_t>(n_planes) * n; row += gridDim.x) {
        const uint32_t pl = static_cast<uint32_t>(row / n), i = static_cast<uint32_t>(row - static_cast<uint64_t>(pl) * n);
        int32_t *src = planes + pl * nn + static_cast<uint64_t>(i) * n;
        int32_t *dst = packed + pl * tri + (static_cast<uint64_t>(i) * n - static_cast<uint64_t>(i) * (i + 1) / 2);
        for (uint32_t j = i + 1 + threadIdx.x; j < n; j += 256) {
            if (PACK) {
                dst[j - i - 1] = src[j];
            } else {
                src[j] = dst[j - i - 1];
            }
        }
    }
}

// non-zeros of the upper triangles (i < j) of `n_planes` planes as a list (index relative to the first of the planes =
// plane * n^2 + i * n + j, value), row by row: pass 1 counts per row, an exclusive scan gives every row its place,
// pass 2 writes with a block-wide prefix sum per 256 columns. No global atomics (a first version appended through one
// global cursor: 1.8 M same-address atomics made it 1.7 ms at 8 000 cells) and a deterministic order.
template <bool WRITE>
__global__ void __launch_bounds__(256) sparse_rows_kernel(const int32_t *__restrict__ planes, uint32_t n, uint32_t n_planes,
                                                          uint32_t *__restrict__ row_cnt, const uint64_t *__restrict__ row_off,
                                                          uint32_t *__restrict__ idx, int32_t *__restrict__ val) {
    __shared__ uint32_t warp_tot[8];
    const uint64_t nn = static_cast<uint64_t>(n) * n;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint64_t row = blockIdx.x; row < static_cast<uint64_t>(n_planes) * n; row += gridDim.x) {
        const uint32_t pl = static_cast<uint32_t>(row / n), i = static_cast<uint32_t>(row - static_cast<uint64_t>(pl) * n);
        const int32_t *src = planes + pl * nn + static_cast<uint64_t>(i) * n;
        uint64_t base = WRITE ? row_off[row] : 0;
        uint32_t mine = 0;
        for (uint32_t j0 = i + 1; j0 < n; j0 += 256) {
            const uint32_t j = j0 + threadIdx.x;
            const int32_t v = j < n ? src[j] : 0;
            const unsigned m = __ballot_sync(0xFFFFFFFFu, v != 0);
            if (!WRITE) {
                mine += lane == 0 ? __popc(m) : 0;
            } else {
                if (lane == 0) {
                    warp_tot[warp] = __popc(m);
                }
                __syncthreads();
                uint32_t before = 0, total = 0;
#pragma unroll
                for (int w = 0; w < 8; ++w) {
                    const uint32_t t = warp_tot[w];
                    before += w < warp ? t : 0;
                    total += t;
                }
                if (v != 0) {
                    const uint64_t o = base + before + __popc(m & ((1u << lane) - 1u));
                    idx[o] = static_cast<uint32_t>(pl * nn + static_cast<uint64_t>(i) * n + j);
                    val[o] = v;
                }
                base += total;
                __syncthreads();
            }
        }
        if (!WRITE) {
            if (lane == 0) {
                warp_tot[warp] = mine;
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                uint32_t t = 0;
                for (int w = 0; w < 8; ++w) {
                    t += warp_tot[w];
                }
                row_cnt[row] = t;
            }
            __syncthreads();
        }
    }
}

__global__ void sparse_add_kernel(int32_t *__restrict__ planes, const uint32_t *__restrict__ idx, const int32_t *__restrict__ val,
                                  uint64_t nnz) {
    const uint64_t k = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (k < nnz && val[k] != 0) {
        planes[idx[k]] += val[k]; // the indices of one list are distinct
    }
}

// order-independent checksum of (sums of) upper triangles, see sgpu_counts_checksum
struct ChecksumArgs {
    const int32_t *peer[SGPU_MAX_PEERS];
    uint32_t n_peers, n, planes, nb;
    uint64_t nn, t0, t1;
};
__device__ __forceinline__ uint64_t mix_weight(uint64_t x) { // splitmix64 finaliser: weight of a (plane, i, j) position
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
__global__ void __launch_bounds__(256) checksum_kernel(ChecksumArgs a, unsigned long long *__restrict__ sum) {
    unsigned long long acc = 0;
    const uint32_t tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (uint64_t t = a.t0 + blockIdx.x; t < a.t1; t += gridDim.x) {
        // tile number -> (bi, bj), row-major over bj >= bi (same numbering as the slab epilogue)
        const double b = 2.0 * a.nb + 1.0;
        uint32_t bi = static_cast<uint32_t>((b - sqrt(b * b - 8.0 * static_cast<double>(t))) * 0.5);
        auto before = [&](uint32_t r) { return static_cast<uint64_t>(r) * a.nb - static_cast<uint64_t>(r) * (r - 1) / 2; };
        while (bi > 0 && before(bi) > t) {
            --bi;
        }
        while (before(bi + 1) <= t) {
            ++bi;
        }
        const uint32_t bj = bi + static_cast<uint32_t>(t - before(bi));
        for (int k = 0; k < 4; ++k) {
            const uint32_t i = bi * 32 + ty + 8 * k, j = bj * 32 + tx;
            if (i < j && j < a.n) {
                const uint64_t idx = static_cast<uint64_t>(i) * a.n + j;
                for (uint32_t pl = 0; pl < a.planes; ++pl) {
                    long long v = 0;
                    for (uint32_t q = 0; q < a.n_peers; ++q) {
                        v += a.peer[q][pl * a.nn + idx];
                    }
                    acc += static_cast<unsigned long long>(v) * mix_weight(pl * a.nn + idx);
                }
            }
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        acc += __shfl_xor_sync(0xffffffffu, acc, o);
    }
    if (tx == 0 && acc) {
        atomicAdd(sum, acc);
    }
}

struct EventTimer {
    cudaEvent_t a = nullptr, b = nullptr;
    cudaStream_t st;
    explicit EventTimer(cudaStream_t s) : st(s) {
        cudaEventCreate(&a);
        cudaEventCreate(&b);
        cudaEventRecord(a, st);
    }
    float stop() {
        float ms = 0;
        cudaEventRecord(b, st);
        cudaEventSynchronize(b);
        cudaEventElapsedTime(&ms, a, b);
        return ms;
    }
    // the same without making the host wait at the end of every phase (each wait leaves the stream empty for a launch
    // latency): mark() now, ms() once the stream has been synchronised anyway
    void mark() { cudaEventRecord(b, st); }
    float ms() {
        float v = 0;
        cudaEventSynchronize(b);
        cudaEventElapsedTime(&v, a, b);
        return v;
    }
    ~EventTimer() {
        cudaEventDestroy(a);
        cudaEventDestroy(b);
    }
};

// Cost model fitted to profiles/r1_path_crossover.txt (16 384 loci, 500 .. 16 000 cells, 0.002x .. 0.5x), in ms:
//   scatter: 0.03 + pairs / rate, pairs = L c^2 / 2 (c = entries per locus); rate 150 pairs/ns while the two N^2 int32
//            planes stay in L2 (N <= 2800), 35 pairs/ns beyond (HBM atomics)
//   GEMM:    0.15 + L * 4 N_pad^2 / 4.0e12 (the tcgen05 kernel at ~4 POP/s issued) + 4.4e-9 per entry (staging)
// The dense path wins for every BASELINE config except the 500-cell one; scatter wins where fewer than ~50 reads
// cover a locus of several thousand cells.
int choose_path_impl(const sgpu_pileup *p, uint32_t num_cells) {
    if (p->n_loci == 0 || num_cells < 256) {
        return SGPU_PATH_SCATTER;
    }
    const double L = static_cast<double>(p->n_loci), E = static_cast<double>(p->n_entries);
    const double c = E / L; // reads per locus
    const double n_pad = (num_cells + 255) / 256 * 256.0;
    const double t_scatter = 0.03 + 0.5 * c * c * L / (num_cells <= 2800 ? 150e6 : 35e6);
    const double t_gemm = 0.15 + L * 4.0 * n_pad * n_pad / 4.0e12 + E * 4.4e-9;
    return t_scatter < t_gemm ? SGPU_PATH_SCATTER : SGPU_PATH_GEMM;
}

} // namespace

int sgpu_choose_path(const sgpu_pileup *p, uint32_t num_cells) { return choose_path_impl(p, num_cells); }

extern "C" {

int sgpu_init(int device, sgpu_ctx **out) {
    if (!out) {
        return SGPU_E_ARG;
    }
    *out = nullptr;
    sgpu_ctx *ctx = new sgpu_ctx();
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || device < 0 || device >= n_dev) {
        // no CPU fallback: the caller gets an error and a context that only carries the message
        sgpu_fail(ctx, SGPU_E_CUDA, "no usable CUDA device %d (%s, %d devices)", device,
                  e == cudaSuccess ? "out of range" : cudaGetErrorString(e), n_dev);
        *out = ctx;
        return SGPU_E_CUDA;
    }
    ctx->device = device;
    const char *tr = getenv("SECEDO_B200_TRACE");
    ctx->trace = tr && tr[0] == '1';
    ctx->trace_alloc = tr && tr[0] == '2';
    *out = ctx;
    SGPU_CUDA(ctx, cudaSetDevice(device));
    cudaDeviceProp prop;
    SGPU_CUDA(ctx, cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        return sgpu_fail(ctx, SGPU_E_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major,
                         prop.minor);
    }
    ctx->sm_count = prop.multiProcessorCount;
    SGPU_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking));
    ctx->stream = ctx->own_stream;
    SGPU_CUDA(ctx, cudaMallocHost(&ctx->h_scratch, 64 * sizeof(uint64_t)));
    SGPU_CUDA(ctx, cudaMalloc(&ctx->d_scratch, 64 * sizeof(uint64_t)));
    {
        // the tensor kernels' own stream, highest priority: a pending tensor CTA is placed before the CTAs of the staging
        // kernels it shares the SMs with
        int least = 0, greatest = 0;
        SGPU_CUDA(ctx, cudaDeviceGetStreamPriorityRange(&least, &greatest));
        SGPU_CUDA(ctx, cudaStreamCreateWithPriority(&ctx->tensor.stream, cudaStreamNonBlocking, greatest));
        const char *as = getenv("SECEDO_B200_ASYNC_GEMM");
        ctx->tensor.async = !(as && as[0] == '0');
        // kernels only run beside the tensor kernel while the device-wide cache preference is PreferShared (sgpu_ctx::prefer_shared,
        // profiles/coresidency_probe.cu): switched on and off around the window in which that can happen
        const char *ps = getenv("SECEDO_B200_PREFER_SHARED");
        ctx->prefer_shared = ps ? ps[0] != '0' : ctx->tensor.async;
    }
    return SGPU_OK;
}

void sgpu_shutdown(sgpu_ctx *ctx) {
    if (!ctx) {
        return;
    }
    if (ctx->own_stream) { // contexts that failed in sgpu_init carry only the error text
        cudaSetDevice(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        if (ctx->tensor.stream) {
            sgpu_tensor_drain(ctx); // issues a launch that is still held back, waits for all of them
            cudaStreamSynchronize(ctx->tensor.stream);
            for (cudaEvent_t e : ctx->tensor.event_pool) {
                cudaEventDestroy(e);
            }
            ctx->tensor.event_pool.clear();
            cudaStreamDestroy(ctx->tensor.stream);
            ctx->tensor.stream = nullptr;
        }
        if (ctx->cache_pref_now == 1) { // the device-wide preference this context switched on goes with it
            cudaDeviceSetCacheConfig(cudaFuncCachePreferNone);
            ctx->cache_pref_now = 0;
        }
        if (ctx->d2h_stream) {
            cudaStreamSynchronize(ctx->d2h_stream);
            cudaStreamDestroy(ctx->d2h_stream);
            cudaEventDestroy(ctx->out_done);
        }
        sgpu_dev_release_cache(ctx);
        for (auto &b : ctx->live_blocks) { // objects the caller never freed
            cudaFree(b.first);
        }
        ctx->live_blocks.clear();
        if (ctx->tile_cache) {
            cudaFree(ctx->tile_cache);
        }
        if (ctx->ep_tiles) {
            cudaFree(ctx->ep_tiles);
        }
        if (ctx->h_scratch) {
            cudaFreeHost(ctx->h_scratch);
        }
        if (ctx->d_scratch) {
            cudaFree(ctx->d_scratch);
        }
        ctx->stream = nullptr;
        if (ctx->copy_stream) {
            cudaStreamSynchronize(ctx->copy_stream);
            cudaStreamDestroy(ctx->copy_stream);
        }
        cudaStreamSynchronize(ctx->own_stream);
        cudaStreamDestroy(ctx->own_stream);
    }
    delete ctx;
}

const char *sgpu_last_error(const sgpu_ctx *ctx) { return ctx ? ctx->error.c_str() : "null context"; }

int sgpu_set_stream(sgpu_ctx *ctx, void *cuda_stream) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    // cached blocks are only safe to reuse in the order of ONE stream: drain the old one first
    SGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    SGPU_TRY(sgpu_tensor_drain(ctx));
    ctx->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->own_stream;
    return SGPU_OK;
}

uint64_t sgpu_launch_count(const sgpu_ctx *ctx) { return ctx ? ctx->launches : 0; }

int sgpu_synchronize(sgpu_ctx *ctx) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device)); // a held-back tensor kernel may be launched here
    if (ctx->copy_stream) {
        SGPU_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream));
    }
    SGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    SGPU_TRY(sgpu_tensor_poll(ctx, true)); // tensor kernels still in flight (sgpu_ctx::tensor)
    return SGPU_OK;
}

} // extern "C"

int sgpu_cache_preference(sgpu_ctx *ctx, bool shared) {
    if (!ctx->prefer_shared || ctx->cache_pref_now == (shared ? 1 : 0)) {
        return SGPU_OK;
    }
    SGPU_CUDA(ctx, cudaDeviceSetCacheConfig(shared ? cudaFuncCachePreferShared : cudaFuncCachePreferNone));
    ctx->cache_pref_now = shared ? 1 : 0;
    return SGPU_OK;
}

// The prologue of every entry point that reads or writes the count planes of c: a first-order tensor kernel may still be
// adding to them (sgpu_ctx::tensor), so ctx->stream waits for it. The device is set first: the join may issue a held-back
// launch.
static int planes_ready(sgpu_ctx *ctx, const sgpu_counts *c) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    return sgpu_tensor_join(ctx, c->i32);
}

extern "C" {

int sgpu_tensor_times(sgpu_ctx *ctx, float *ms, uint64_t *launches) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    SGPU_TRY(sgpu_tensor_poll(ctx, true));
    float m = 0.f;
    uint64_t n = 0;
    sgpu_tensor_take_times(ctx, &m, &n);
    if (ms) {
        *ms = m;
    }
    if (launches) {
        *launches = n;
    }
    return SGPU_OK;
}

int sgpu_set_option(sgpu_ctx *ctx, const char *name, int value) {
    if (!name) {
        return sgpu_fail(ctx, SGPU_E_ARG, "sgpu_set_option: null name");
    }
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    SGPU_TRY(sgpu_synchronize(ctx));
    const std::string n(name);
    if (n == "async_gemm") {
        ctx->tensor.async = value != 0;
    } else if (n == "prefer_shared") {
        if (value != 0 && value != 1) {
            return sgpu_fail(ctx, SGPU_E_ARG, "prefer_shared must be 0 or 1");
        }
        if (ctx->cache_pref_now == 1) { // back to the default split before the mode changes
            SGPU_CUDA(ctx, cudaDeviceSetCacheConfig(cudaFuncCachePreferNone));
            ctx->cache_pref_now = 0;
        }
        ctx->prefer_shared = value == 1;
    } else {
        return sgpu_fail(ctx, SGPU_E_ARG, "sgpu_set_option: unknown option '%s'", name);
    }
    return SGPU_OK;
}

// ---- pileup ---------------------------------------------------------------------------------------
static int pileup_upload(sgpu_ctx *ctx, uint32_t n_chr, const uint64_t *chr_ptr, const uint64_t *row_ptr,
                         const uint32_t *position, const uint32_t *read_id, const uint16_t *gid_base, bool async,
                         sgpu_pileup **out, bool lazy_read_id = false, const uint32_t *gid_base32 = nullptr) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    if (async) {
        if (!ctx->copy_stream) {
            SGPU_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
        }
        // the blocks may come from the cache with work of their previous life still queued on the
        // compute stream: the copies start behind everything queued there so far
        cudaEvent_t ev;
        SGPU_CUDA(ctx, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        SGPU_CUDA(ctx, cudaEventRecord(ev, ctx->stream));
        SGPU_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ev, 0));
        SGPU_CUDA(ctx, cudaEventDestroy(ev));
        st = ctx->copy_stream;
    }
    sgpu_pileup *p = new sgpu_pileup();
    PileupOwner p_owner(ctx, p);
    p->n_chr = n_chr;
    p->n_loci = chr_ptr[n_chr];
    p->n_entries = p->n_loci ? row_ptr[p->n_loci] : 0;
    p->wide = gid_base32 != nullptr;
    p->h_chr_ptr = new uint64_t[n_chr + 1];
    std::memcpy(p->h_chr_ptr, chr_ptr, (n_chr + 1) * sizeof(uint64_t));
    const uint64_t P = p->n_loci, E = p->n_entries;
    SGPU_CUDA(ctx, sgpu_dev_alloc(ctx, reinterpret_cast<void **>(&p->d_chr_ptr), (n_chr + 1) * sizeof(uint64_t)));
    SGPU_CUDA(ctx, sgpu_dev_alloc(ctx, reinterpret_cast<void **>(&p->d_row_ptr), (P + 1) * sizeof(uint64_t)));
    SGPU_CUDA(ctx, sgpu_dev_alloc(ctx, reinterpret_cast<void **>(&p->d_position), (P ? P : 1) * sizeof(uint32_t)));
    if (lazy_read_id && E) {
        void *alias = nullptr;
        if (cudaHostGetDevicePointer(&alias, const_cast<uint32_t *>(read_id), 0) != cudaSuccess) {
            cudaGetLastError();
            return sgpu_fail(ctx, SGPU_E_ARG, "lazy upload: read_id must be page-locked, mapped host memory (cudaHostAlloc / cudaHostRegister)");
        }
        p->zc_read_id = static_cast<const uint32_t *>(alias);
    } else {
        SGPU_CUDA(ctx, sgpu_dev_alloc(ctx, reinterpret_cast<void **>(&p->d_read_id), (E ? E : 1) * sizeof(uint32_t)));
    }
    if (p->wide) {
        SGPU_CUDA(ctx, sgpu_dev_alloc(ctx, reinterpret_cast<void **>(&p->d_gid_base32), (E ? E : 1) * sizeof(uint32_t)));
    } else {
        SGPU_CUDA(ctx, sgpu_dev_alloc(ctx, reinterpret_cast<void **>(&p->d_gid_base), (E ? E : 1) * sizeof(uint16_t)));
    }
    // the copy of chr_ptr reads p->h_chr_ptr (owned by the pileup), not the caller's array
    SGPU_CUDA(ctx, cudaMemcpyAsync(p->d_chr_ptr, p->h_chr_ptr, (n_chr + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    if (P) {
        SGPU_CUDA(ctx, cudaMemcpyAsync(p->d_row_ptr, row_ptr, (P + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
        SGPU_CUDA(ctx, cudaMemcpyAsync(p->d_position, position, P * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    } else {
        SGPU_CUDA(ctx, cudaMemsetAsync(p->d_row_ptr, 0, sizeof(uint64_t), st));
    }
    if (E) {
        if (p->d_read_id) {
            SGPU_CUDA(ctx, cudaMemcpyAsync(p->d_read_id, read_id, E * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        }
        if (p->wide) {
            SGPU_CUDA(ctx, cudaMemcpyAsync(p->d_gid_base32, gid_base32, E * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        } else {
            SGPU_CUDA(ctx, cudaMemcpyAsync(p->d_gid_base, gid_base, E * sizeof(uint16_t), cudaMemcpyHostToDevice, st));
        }
    }
    if (async) {
        SGPU_CUDA(ctx, cudaEventCreateWithFlags(&p->ready, cudaEventDisableTiming));
        SGPU_CUDA(ctx, cudaEventRecord(p->ready, st));
    } else {
        SGPU_CUDA(ctx, cudaStreamSynchronize(st));
    }
    *out = p_owner.release();
    return SGPU_OK;
}

int sgpu_pileup_upload(sgpu_ctx *ctx, uint32_t n_chr, const uint64_t *chr_ptr, const uint64_t *row_ptr,
                       const uint32_t *position, const uint32_t *read_id, const uint16_t *gid_base,
                       sgpu_pileup **out) {
    return pileup_upload(ctx, n_chr, chr_ptr, row_ptr, position, read_id, gid_base, false, out);
}

int sgpu_pileup_upload_wide(sgpu_ctx *ctx, uint32_t n_chr, const uint64_t *chr_ptr, const uint64_t *row_ptr,
                            const uint32_t *position, const uint32_t *read_id, const uint32_t *gid_base32, sgpu_pileup **out) {
    if (!gid_base32) {
        return sgpu_fail(ctx, SGPU_E_ARG, "upload_wide: gid_base32 missing");
    }
    return pileup_upload(ctx, n_chr, chr_ptr, row_ptr, position, read_id, nullptr, false, out, false, gid_base32);
}

int sgpu_pileup_upload_wide_async(sgpu_ctx *ctx, uint32_t n_chr, const uint64_t *chr_ptr, const uint64_t *row_ptr,
                                  const uint32_t *position, const uint32_t *read_id, const uint32_t *gid_base32, sgpu_pileup **out) {
    if (!gid_base32) {
        return sgpu_fail(ctx, SGPU_E_ARG, "upload_wide: gid_base32 missing");
    }
    return pileup_upload(ctx, n_chr, chr_ptr, row_ptr, position, read_id, nullptr, true, out, false, gid_base32);
}

int sgpu_pileup_is_wide(const sgpu_pileup *p) { return p && p->wide ? 1 : 0; }

int sgpu_pileup_upload_async(sgpu_ctx *ctx, uint32_t n_chr, const uint64_t *chr_ptr, const uint64_t *row_ptr,
                             const uint32_t *position, const uint32_t *read_id, const uint16_t *gid_base,
                             sgpu_pileup **out) {
    return pileup_upload(ctx, n_chr, chr_ptr, row_ptr, position, read_id, gid_base, true, out);
}

int sgpu_pileup_upload_lazy_async(sgpu_ctx *ctx, uint32_t n_chr, const uint64_t *chr_ptr, const uint64_t *row_ptr,
                                  const uint32_t *position, const uint32_t *read_id, const uint16_t *gid_base,
                                  sgpu_pileup **out) {
    return pileup_upload(ctx, n_chr, chr_ptr, row_ptr, position, read_id, gid_base, true, out, true);
}

} // extern "C"

namespace {
// read ids of a view: one warp per locus copies the locus' run of the source into the pileup's own array
__global__ void __launch_bounds__(256) gather_view_kernel(const uint64_t *__restrict__ row_ptr, const uint64_t *__restrict__ view_off,
                                                          uint64_t n_loci, const uint32_t *__restrict__ src, uint32_t *__restrict__ dst) {
    const int lane = threadIdx.x & 31;
    const uint64_t warps_total = static_cast<uint64_t>(gridDim.x) * 8;
    for (uint64_t l = static_cast<uint64_t>(blockIdx.x) * 8 + (threadIdx.x >> 5); l < n_loci; l += warps_total) {
        const uint64_t e0 = row_ptr[l], n = row_ptr[l + 1] - e0, s0 = view_off[l];
        for (uint64_t i = lane; i < n; i += 128) {
            uint32_t v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                v[u] = i + 32 * u < n ? src[s0 + i + 32 * u] : 0;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (i + 32 * u < n) {
                    dst[e0 + i + 32 * u] = v[u];
                }
            }
        }
    }
}

// the last view of a pileup its owner has already freed: free it now
void release_view(sgpu_pileup *p) {
    sgpu_pileup *src = p->view_src;
    p->view_src = nullptr;
    p->view_read_id = nullptr;
    if (src && src->view_refs.fetch_sub(1) == 1 && src->zombie) {
        sgpu_pileup_free(src->zombie_ctx, src);
    }
}
} // namespace

int sgpu_pileup_materialize(sgpu_ctx *ctx, const sgpu_pileup *cp, bool keep_view) {
    sgpu_pileup *p = const_cast<sgpu_pileup *>(cp);
    if (!p || p->d_read_id) {
        return SGPU_OK;
    }
    const uint64_t E = p->n_entries;
    if (p->view_read_id) {
        if (keep_view) {
            return SGPU_OK;
        }
        SGPU_CUDA(ctx, sgpu_dev_alloc(ctx, reinterpret_cast<void **>(&p->d_read_id), (E ? E : 1) * sizeof(uint32_t)));
        if (p->n_loci) {
            const unsigned grid = static_cast<unsigned>(std::min<uint64_t>(ceil_div_u64(p->n_loci, 8), static_cast<uint64_t>(ctx->sm_count) * 16));
            SGPU_LAUNCH(ctx, (gather_view_kernel<<<grid, 256, 0, ctx->stream>>>(p->d_row_ptr, p->view_off, p->n_loci, p->view_read_id, p->d_read_id)));
            SGPU_CUDA(ctx, cudaGetLastError());
        }
        sgpu_dev_free(ctx, p->view_off); // stream ordered behind the gather
        p->view_off = nullptr;
        release_view(p);
        return SGPU_OK;
    }
    if (!p->zc_read_id) {
        return SGPU_OK;
    }
    SGPU_CUDA(ctx, sgpu_dev_alloc(ctx, reinterpret_cast<void **>(&p->d_read_id), (E ? E : 1) * sizeof(uint32_t)));
    SGPU_CUDA(ctx, cudaMemcpyAsync(p->d_read_id, p->zc_read_id, E * sizeof(uint32_t), cudaMemcpyDefault, ctx->stream));
    return SGPU_OK;
}

extern "C" {

int sgpu_pileup_wrap_device(sgpu_ctx *ctx, uint32_t n_chr, const uint64_t *host_chr_ptr, const uint64_t *dev_row_ptr,
                            const uint32_t *dev_position, const uint32_t *dev_read_id, const uint16_t *dev_gid_base,
                            sgpu_pileup **out) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    sgpu_pileup *p = new sgpu_pileup();
    PileupOwner p_owner(ctx, p);
    p->n_chr = n_chr;
    p->n_loci = host_chr_ptr[n_chr];
    p->h_chr_ptr = new uint64_t[n_chr + 1];
    std::memcpy(p->h_chr_ptr, host_chr_ptr, (n_chr + 1) * sizeof(uint64_t));
    SGPU_CUDA(ctx, sgpu_dev_alloc(ctx, reinterpret_cast<void **>(&p->d_chr_ptr), (n_chr + 1) * sizeof(uint64_t)));
    SGPU_CUDA(ctx, cudaMemcpyAsync(p->d_chr_ptr, host_chr_ptr, (n_chr + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
    p->d_row_ptr = const_cast<uint64_t *>(dev_row_ptr);
    p->d_position = const_cast<uint32_t *>(dev_position);
    p->d_read_id = const_cast<uint32_t *>(dev_read_id);
    p->d_gid_base = const_cast<uint16_t *>(dev_gid_base);
    p->owns = false;
    uint64_t last = 0;
    if (p->n_loci) {
        SGPU_CUDA(ctx, cudaMemcpyAsync(&ctx->h_scratch[0], dev_row_ptr + p->n_loci, sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
        SGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        last = ctx->h_scratch[0];
    }
    SGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    p->n_entries = last;
    *out = p_owner.release();
    return SGPU_OK;
}

int sgpu_pileup_dims(const sgpu_pileup *p, uint32_t *n_chr, uint64_t *n_loci, uint64_t *n_entries) {
    if (!p) {
        return SGPU_E_ARG;
    }
    if (n_chr) {
        *n_chr = p->n_chr;
    }
    if (n_loci) {
        *n_loci = p->n_loci;
    }
    if (n_entries) {
        *n_entries = p->n_entries;
    }
    return SGPU_OK;
}

static int pileup_download(sgpu_ctx *ctx, const sgpu_pileup *p, uint64_t *chr_ptr, uint64_t *row_ptr, uint32_t *position,
                           uint32_t *read_id, uint16_t *gid_base, uint32_t *gid_base32);

int sgpu_pileup_download(sgpu_ctx *ctx, const sgpu_pileup *p, uint64_t *chr_ptr, uint64_t *row_ptr, uint32_t *position,
                         uint32_t *read_id, uint16_t *gid_base) {
    if (p->wide && gid_base) {
        return sgpu_fail(ctx, SGPU_E_ARG, "wide pileup: use sgpu_pileup_download_wide");
    }
    return pileup_download(ctx, p, chr_ptr, row_ptr, position, read_id, gid_base, nullptr);
}

int sgpu_pileup_download_wide(sgpu_ctx *ctx, const sgpu_pileup *p, uint64_t *chr_ptr, uint64_t *row_ptr, uint32_t *position,
                              uint32_t *read_id, uint32_t *gid_base32) {
    if (!p->wide && gid_base32) {
        return sgpu_fail(ctx, SGPU_E_ARG, "not a wide pileup: use sgpu_pileup_download");
    }
    return pileup_download(ctx, p, chr_ptr, row_ptr, position, read_id, nullptr, gid_base32);
}

static int pileup_download(sgpu_ctx *ctx, const sgpu_pileup *p, uint64_t *chr_ptr, uint64_t *row_ptr, uint32_t *position,
                           uint32_t *read_id, uint16_t *gid_base, uint32_t *gid_base32) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    SGPU_WAIT_PILEUP(ctx, p);
    if (read_id) {
        SGPU_TRY(sgpu_pileup_materialize(ctx, p));
    }
    cudaStream_t st = ctx->stream;
    if (chr_ptr) {
        std::memcpy(chr_ptr, p->h_chr_ptr, (p->n_chr + 1) * sizeof(uint64_t));
    }
    if (row_ptr) {
        SGPU_CUDA(ctx, cudaMemcpyAsync(row_ptr, p->d_row_ptr, (p->n_loci + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    }
    if (position && p->n_loci) {
        SGPU_CUDA(ctx, cudaMemcpyAsync(position, p->d_position, p->n_loci * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    }
    if (read_id && p->n_entries) {
        SGPU_CUDA(ctx, cudaMemcpyAsync(read_id, p->d_read_id, p->n_entries * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    }
    if (gid_base && p->n_entries) {
        SGPU_CUDA(ctx, cudaMemcpyAsync(gid_base, p->d_gid_base, p->n_entries * sizeof(uint16_t), cudaMemcpyDeviceToHost, st));
    }
    if (gid_base32 && p->n_entries) {
        SGPU_CUDA(ctx, cudaMemcpyAsync(gid_base32, p->d_gid_base32, p->n_entries * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    }
    SGPU_CUDA(ctx, cudaStreamSynchronize(st));
    return SGPU_OK;
}

void sgpu_pileup_free(sgpu_ctx *ctx, sgpu_pileup *p) {
    if (!p) {
        return;
    }
    if (p->view_refs.load() > 0) { // filtered pileups still read this one's ids (sgpu_pileup::view_read_id): the last of them frees it
        p->zombie = true;
        p->zombie_ctx = ctx;
        return;
    }
    if (ctx) {
        cudaSetDevice(ctx->device);
    }
    if (p->view_off) {
        sgpu_dev_free(ctx, p->view_off);
        p->view_off = nullptr;
    }
    if (p->view_src) {
        release_view(p);
    }
    if (p->ready) {
        if (ctx) { // the blocks go back to the cache of the compute stream: order it behind the copies
            cudaStreamWaitEvent(ctx->stream, p->ready, 0);
        }
        cudaEventDestroy(p->ready);
    }
    sgpu_dev_free(ctx, p->d_chr_ptr); // reuse is stream ordered: safe after everything already queued
    if (p->owns) {
        sgpu_dev_free(ctx, p->d_row_ptr);
        sgpu_dev_free(ctx, p->d_position);
        sgpu_dev_free(ctx, p->d_read_id);
        sgpu_dev_free(ctx, p->d_gid_base);
        sgpu_dev_free(ctx, p->d_gid_base32);
    }
    delete[] p->h_chr_ptr;
    delete p;
}

// ---- filter ---------------------------------------------------------------------------------------
int sgpu_is_significant(sgpu_ctx *ctx, const uint16_t *counts4, uint64_t n, double theta, int cell_proportion,
                        uint8_t *out) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    return sgpu_is_significant_impl(ctx, counts4, n, theta, cell_proportion, out);
}

int sgpu_filter(sgpu_ctx *ctx, const sgpu_pileup *in, const uint32_t *id_to_pos, uint32_t n_groups, double theta,
                int cell_proportion, sgpu_pileup **filtered, double *avg_coverage) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    SGPU_WAIT_PILEUP(ctx, in);
    return sgpu_filter_impl(ctx, in, id_to_pos, n_groups, theta, cell_proportion, filtered, avg_coverage);
}

// ---- counts ---------------------------------------------------------------------------------------
int sgpu_counts_create(sgpu_ctx *ctx, uint32_t num_cells, sgpu_counts **out) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    sgpu_counts *c = new sgpu_counts();
    c->n = num_cells;
    c->nn = static_cast<uint64_t>(num_cells) * num_cells;
    c->owner = ctx;
    cudaError_t e = cudaMalloc(&c->i32, std::max<uint64_t>(1, N_PLANES * c->nn) * sizeof(int32_t));
    if (e == cudaSuccess) {
        e = cudaMalloc(&c->hist, SGPU_MAX_CLASS * SGPU_MAX_CLASS * sizeof(uint64_t));
    }
    if (e != cudaSuccess) { // nothing half-built is left behind
        cudaGetLastError();
        sgpu_counts_free(ctx, c);
        return sgpu_fail(ctx, SGPU_E_CUDA, "sgpu_counts_create(%u cells): %s", num_cells, cudaGetErrorString(e));
    }
    *out = c;
    return sgpu_counts_zero(ctx, c);
}

int sgpu_counts_zero(sgpu_ctx *ctx, sgpu_counts *c) {
    SGPU_TRY(planes_ready(ctx, c));
    // only the planes that were used since the last zeroing can be non-zero
    SGPU_CUDA(ctx, cudaMemsetAsync(c->i32, 0, static_cast<uint64_t>(c->planes_dirty) * c->nn * sizeof(int32_t), ctx->stream));
    SGPU_CUDA(ctx, cudaMemsetAsync(c->hist, 0, SGPU_MAX_CLASS * SGPU_MAX_CLASS * sizeof(uint64_t), ctx->stream));
    if (c->spill) {
        SGPU_CUDA(ctx, cudaMemsetAsync(c->spill, 0, c->nn * sizeof(double), ctx->stream));
    }
    c->planes_used = 2;
    c->planes_dirty = 2;
    c->have_params = false;
    c->fresh = true;
    c->poisoned = false;
    return SGPU_OK;
}

void sgpu_counts_free(sgpu_ctx *ctx, sgpu_counts *c) {
    if (!c) {
        return;
    }
    if (ctx) {
        cudaSetDevice(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        sgpu_tensor_drain(ctx);
    }
    cudaFree(c->i32);
    cudaFree(c->hist);
    cudaFree(c->spill);
    cudaFree(c->slab_minmax);
    cudaFree(c->slab_out);
    if (ctx) {
        sgpu_dev_free(ctx, c->slab_raw);
    }
    if (ctx) {
        sgpu_dev_free(ctx, c->packed);
        sgpu_dev_free(ctx, c->sp_idx);
        sgpu_dev_free(ctx, c->sp_val);
    }
    delete c;
}

} // extern "C"

static int accumulate_impl(sgpu_ctx *ctx, sgpu_counts *c, const sgpu_pileup *filtered, uint32_t max_fragment_length,
                           const uint32_t *group_id_to_pos, uint32_t n_groups, double mutation_rate,
                           double homozygous_rate, double seq_error_rate, uint32_t num_threads, int path,
                           sgpu_stats *stats, const RangeSpec *range) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    SGPU_WAIT_PILEUP(ctx, filtered);
    SGPU_TRY(sgpu_pileup_materialize(ctx, filtered, true)); // a view of the unfiltered pileup's read ids stays one
    if (path < SGPU_PATH_AUTO || path > SGPU_PATH_GEMM) {
        return sgpu_fail(ctx, SGPU_E_ARG, "unknown path %d", path);
    }
    if (c->have_params
        && (c->eps != mutation_rate || c->h != homozygous_rate || c->theta != seq_error_rate || c->L != max_fragment_length)) {
        return sgpu_fail(ctx, SGPU_E_ARG, "counts object was accumulated with different likelihood parameters");
    }
    c->have_params = true;
    c->eps = mutation_rate;
    c->h = homozygous_rate;
    c->theta = seq_error_rate;
    c->L = max_fragment_length;
    sgpu_stats s;
    std::memset(&s, 0, sizeof(s));
    s.n_loci = filtered->n_loci;
    s.n_entries = filtered->n_entries;
    const bool auto_path = path == SGPU_PATH_AUTO;
    if (auto_path) {
        path = choose_path_impl(filtered, c->n);
    }
    s.path_used = path;
    if (c->poisoned) {
        return sgpu_fail(ctx, SGPU_E_ARG, "the counts object holds a partial sum after a failed call: sgpu_counts_zero first");
    }

    // tensor kernels of earlier batches that have finished meanwhile: their time goes into this call's statistics
    SGPU_TRY(sgpu_tensor_poll(ctx, false));
    LinkResult lr;
    EventTimer t_link(ctx->stream);
    SGPU_TRY(sgpu_link_reads(ctx, filtered, c->n, max_fragment_length, group_id_to_pos, n_groups, num_threads, &lr, range));
    t_link.mark();
    s.n_reads = lr.n_reads;
    s.n_dropped_entries = lr.n_dropped;
    s.n_multi_reads = lr.n_multi;
    s.n_tail_reads = lr.n_tail;
    s.n_span_splits = static_cast<int32_t>(std::min<uint64_t>(lr.n_span_splits, 0x7FFFFFFF));
    ctx->tensor.ms_stage = 0.f;
    // Once first-order counts have been issued, a failure leaves a partial sum behind, possibly in every plane (the
    // order-2 / order-3 atomics of the other pairs land too): later accumulations are then refused until
    // sgpu_counts_zero, and that clears all planes. Failures before that point leave the object as it was.
    auto issued = [c](int rc) {
        if (rc != SGPU_OK) {
            c->poisoned = true;
            c->planes_dirty = N_PLANES;
        }
        return rc;
    };
    EventTimer t_first(ctx->stream);
    if (path == SGPU_PATH_SCATTER) {
        SGPU_TRY(sgpu_link_dense_codes(ctx, filtered, &lr));
        SGPU_TRY(sgpu_tensor_join(ctx, c->i32)); // the atomics go to the planes a tensor kernel in flight adds to
        SGPU_TRY(issued(sgpu_scatter_pairs(ctx, filtered, lr, c, +1, false, &s.n_pairs_first)));
        c->fresh = false;
    } else {
        // incl. the tail x tail correction. More than 127 reads of one cell at one locus do not fit int8: the first
        // panel is checked before the count planes are touched and, with SGPU_PATH_AUTO, the call takes the scatter
        // path instead
        int rc = sgpu_gemm_counts(ctx, filtered, lr, c, &s.n_pairs_first);
        if (rc == SGPU_E_COUNT_RANGE && auto_path && !c->poisoned) {
            s.path_used = SGPU_PATH_SCATTER;
            SGPU_TRY(sgpu_link_dense_codes(ctx, filtered, &lr));
            SGPU_TRY(sgpu_tensor_join(ctx, c->i32));
            rc = issued(sgpu_scatter_pairs(ctx, filtered, lr, c, +1, false, &s.n_pairs_first));
            c->fresh = false;
        }
        SGPU_TRY(rc);
    }
    t_first.mark();
    s.ms_stage = ctx->tensor.ms_stage;
    // second / third order planes, spill plane, histogram: none of them is touched by the first-order tensor kernel
    // that may still be running
    EventTimer t_multi(ctx->stream);
    SGPU_TRY(issued(sgpu_multilocus(ctx, filtered, lr, c, max_fragment_length, &s.n_pairs_multi)));
    t_multi.mark();
    s.ms_multi = t_multi.ms(); // the one host wait for the three phases
    s.ms_link = t_link.ms();
    s.ms_first_order = t_first.ms();
    // Tensor kernels retired during this call (with SECEDO_B200_ASYNC_GEMM=0: this call's own; otherwise mostly the one of
    // the batch before; sgpu_tensor_times returns what is left)
    SGPU_TRY(issued(sgpu_tensor_poll(ctx, false)));
    sgpu_tensor_take_times(ctx, &s.ms_gemm, &s.gemm_launches);
    c->planes_dirty = std::max(c->planes_dirty, c->planes_used);
    if (stats) {
        *stats = s;
    }
    return SGPU_OK;
}

extern "C" {

int sgpu_counts_accumulate(sgpu_ctx *ctx, sgpu_counts *c, const sgpu_pileup *filtered, uint32_t max_fragment_length,
                           const uint32_t *group_id_to_pos, uint32_t n_groups, double mutation_rate,
                           double homozygous_rate, double seq_error_rate, uint32_t num_threads, int path,
                           sgpu_stats *stats) {
    return accumulate_impl(ctx, c, filtered, max_fragment_length, group_id_to_pos, n_groups, mutation_rate, homozygous_rate,
                           seq_error_rate, num_threads, path, stats, nullptr);
}

int sgpu_counts_accumulate_range(sgpu_ctx *ctx, sgpu_counts *c, const sgpu_pileup *piece, uint32_t max_fragment_length,
                                 const uint32_t *group_id_to_pos, uint32_t n_groups, double mutation_rate,
                                 double homozygous_rate, double seq_error_rate, uint32_t num_threads, const uint32_t *own_pos_begin,
                                 const uint32_t *own_pos_end, const uint32_t *tail_position, int path, sgpu_stats *stats) {
    if (!own_pos_begin || !own_pos_end || !tail_position) {
        return sgpu_fail(ctx, SGPU_E_ARG, "accumulate_range: own_pos_begin, own_pos_end and tail_position are required (one value per chromosome)");
    }
    RangeSpec rs;
    rs.own_pos_begin = own_pos_begin;
    rs.own_pos_end = own_pos_end;
    rs.tail_position = tail_position;
    // num_threads only matters where tail_position is SGPU_TAIL_AUTO: elsewhere the cutoff it selects arrives as a position
    return accumulate_impl(ctx, c, piece, max_fragment_length, group_id_to_pos, n_groups, mutation_rate, homozygous_rate,
                           seq_error_rate, num_threads ? num_threads : 1, path, stats, &rs);
}

int sgpu_chromosome_cutoff(sgpu_ctx *ctx, const sgpu_pileup *ends, uint32_t max_fragment_length, uint32_t num_threads,
                           const uint8_t *whole, uint32_t *tail_position, uint8_t *resolved) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!ends || !whole || !tail_position || !resolved) {
        return sgpu_fail(ctx, SGPU_E_ARG, "chromosome_cutoff: null argument");
    }
    if (num_threads == 0) {
        return sgpu_fail(ctx, SGPU_E_ARG, "num_threads must be >= 1");
    }
    SGPU_WAIT_PILEUP(ctx, ends);
    SGPU_TRY(sgpu_pileup_materialize(ctx, ends, true));
    return sgpu_cutoff_from_suffix(ctx, ends, max_fragment_length, num_threads, whole, tail_position, resolved);
}

int sgpu_counts_buffers(sgpu_counts *c, int32_t **i32, uint64_t *n_i32, double **f64, uint64_t *n_f64, uint64_t **hist,
                        uint64_t *n_hist) {
    if (!c) {
        return SGPU_E_ARG;
    }
    if (c->owner) {
        // whoever reads the planes through these pointers is ordered behind the context's stream (a collective, a peer's
        // kernel after a barrier)
        SGPU_TRY(planes_ready(c->owner, c));
    }
    if (i32) {
        *i32 = c->i32;
    }
    if (n_i32) {
        *n_i32 = static_cast<uint64_t>(c->planes_used) * c->nn;
    }
    if (f64) {
        *f64 = c->spill;
    }
    if (n_f64) {
        *n_f64 = c->spill ? c->nn : 0;
    }
    if (hist) {
        *hist = c->hist;
    }
    if (n_hist) {
        *n_hist = SGPU_MAX_CLASS * SGPU_MAX_CLASS;
    }
    return SGPU_OK;
}

int sgpu_counts_set_layout(sgpu_ctx *ctx, sgpu_counts *c, int planes_used, int want_spill) {
    SGPU_TRY(planes_ready(ctx, c));
    if (planes_used != 2 && planes_used != PLANE_H3 && planes_used != N_PLANES) {
        return sgpu_fail(ctx, SGPU_E_ARG, "planes_used must be 2, %d or %d", PLANE_H3, N_PLANES);
    }
    c->planes_used = std::max(c->planes_used, planes_used);
    c->planes_dirty = std::max(c->planes_dirty, c->planes_used);
    if (want_spill && !c->spill) {
        SGPU_CUDA(ctx, cudaMalloc(&c->spill, std::max<uint64_t>(1, c->nn) * sizeof(double)));
        SGPU_CUDA(ctx, cudaMemsetAsync(c->spill, 0, c->nn * sizeof(double), ctx->stream));
    }
    return SGPU_OK;
}

int sgpu_counts_pack_range(sgpu_ctx *ctx, sgpu_counts *c, int first_plane, int n_planes, int32_t **packed, uint64_t *n) {
    SGPU_TRY(planes_ready(ctx, c));
    if (first_plane < 0 || n_planes < 0 || first_plane + n_planes > c->planes_used) {
        return sgpu_fail(ctx, SGPU_E_ARG, "plane range [%d, %d) outside the %d planes in use", first_plane, first_plane + n_planes, c->planes_used);
    }
    const uint64_t need = static_cast<uint64_t>(n_planes) * c->n * (c->n ? c->n - 1 : 0) / 2;
    if (c->packed_n < need) {
        sgpu_dev_free(ctx, c->packed);
        c->packed = nullptr;
        SGPU_CUDA(ctx, sgpu_dev_alloc(ctx, reinterpret_cast<void **>(&c->packed), std::max<uint64_t>(need, 1) * sizeof(int32_t)));
        c->packed_n = need;
    }
    if (need) {
        const unsigned grid = static_cast<unsigned>(std::min<uint64_t>(static_cast<uint64_t>(n_planes) * c->n,
                                                                      static_cast<uint64_t>(ctx->sm_count) * 16));
        SGPU_LAUNCH(ctx, (tri_pack_kernel<true><<<grid, 256, 0, ctx->stream>>>(c->i32 + static_cast<uint64_t>(first_plane) * c->nn, c->packed,
                                                                              c->n, n_planes)));
        SGPU_CUDA(ctx, cudaGetLastError());
    }
    if (packed) {
        *packed = c->packed;
    }
    if (n) {
        *n = need;
    }
    return SGPU_OK;
}

int sgpu_counts_unpack_range(sgpu_ctx *ctx, sgpu_counts *c, int first_plane, int n_planes) {
    SGPU_TRY(planes_ready(ctx, c));
    if (first_plane < 0 || n_planes < 0 || first_plane + n_planes > c->planes_used) {
        return sgpu_fail(ctx, SGPU_E_ARG, "plane range [%d, %d) outside the %d planes in use", first_plane, first_plane + n_planes, c->planes_used);
    }
    const uint64_t need = static_cast<uint64_t>(n_planes) * c->n * (c->n ? c->n - 1 : 0) / 2;
    if (c->packed == nullptr || c->packed_n < need) {
        return sgpu_fail(ctx, SGPU_E_ARG, "sgpu_counts_unpack without a matching sgpu_counts_pack");
    }
    if (need) {
        const unsigned grid = static_cast<unsigned>(std::min<uint64_t>(static_cast<uint64_t>(n_planes) * c->n,
                                                                      static_cast<uint64_t>(ctx->sm_count) * 16));
        SGPU_LAUNCH(ctx, (tri_pack_kernel<false><<<grid, 256, 0, ctx->stream>>>(c->i32 + static_cast<uint64_t>(first_plane) * c->nn, c->packed,
                                                                               c->n, n_planes)));
        SGPU_CUDA(ctx, cudaGetLastError());
    }
    c->fresh = false;
    return SGPU_OK;
}

int sgpu_counts_pack(sgpu_ctx *ctx, sgpu_counts *c, int32_t **packed, uint64_t *n) {
    return sgpu_counts_pack_range(ctx, c, 0, c->planes_used, packed, n);
}

int sgpu_counts_unpack(sgpu_ctx *ctx, sgpu_counts *c) {
    return sgpu_counts_unpack_range(ctx, c, 0, c->planes_used);
}

int sgpu_counts_sparse_pack(sgpu_ctx *ctx, sgpu_counts *c, int first_plane, uint32_t **idx, int32_t **val, uint64_t *nnz) {
    SGPU_TRY(planes_ready(ctx, c));
    cudaStream_t st = ctx->stream;
    const int n_planes = c->planes_used - first_plane;
    if (first_plane < 0 || n_planes < 0) {
        return sgpu_fail(ctx, SGPU_E_ARG, "first plane %d outside the %d planes in use", first_plane, c->planes_used);
    }
    if (static_cast<uint64_t>(n_planes) * c->nn > 0xFFFFFFFFull) {
        return sgpu_fail(ctx, SGPU_E_ARG, "sparse lists index with 32 bits: %d planes of %u^2 do not fit", n_planes, c->n);
    }
    uint64_t count = 0;
    if (n_planes && c->n > 1) {
        const int32_t *planes = c->i32 + static_cast<uint64_t>(first_plane) * c->nn;
        const uint64_t rows = static_cast<uint64_t>(n_planes) * c->n;
        const unsigned grid = static_cast<unsigned>(std::min<uint64_t>(rows, static_cast<uint64_t>(ctx->sm_count) * 16));
        DevBuf<uint32_t> row_cnt;
        DevBuf<uint64_t> row_off;
        SGPU_CUDA(ctx, row_cnt.alloc(rows, ctx));
        SGPU_CUDA(ctx, row_off.alloc(rows + 1, ctx));
        SGPU_LAUNCH(ctx, (sparse_rows_kernel<false><<<grid, 256, 0, st>>>(planes, c->n, n_planes, row_cnt.p, nullptr, nullptr, nullptr)));
        SGPU_TRY(sgpu_scan_u32_u64(ctx, row_cnt.p, row_off.p, rows));
        SGPU_CUDA(ctx, cudaMemcpyAsync(&ctx->h_scratch[0], row_off.p + rows, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        SGPU_CUDA(ctx, cudaStreamSynchronize(st));
        count = ctx->h_scratch[0];
        if (c->sp_cap < count) {
            sgpu_dev_free(ctx, c->sp_idx);
            sgpu_dev_free(ctx, c->sp_val);
            c->sp_idx = nullptr;
            c->sp_val = nullptr;
            c->sp_cap = 0;
            const uint64_t cap = count + count / 4 + 1024;
            SGPU_CUDA(ctx, sgpu_dev_alloc(ctx, reinterpret_cast<void **>(&c->sp_idx), cap * sizeof(uint32_t)));
            SGPU_CUDA(ctx, sgpu_dev_alloc(ctx, reinterpret_cast<void **>(&c->sp_val), cap * sizeof(int32_t)));
            c->sp_cap = cap;
        }
        if (count) {
            SGPU_LAUNCH(ctx, (sparse_rows_kernel<true><<<grid, 256, 0, st>>>(planes, c->n, n_planes, nullptr, row_off.p, c->sp_idx, c->sp_val)));
        }
        SGPU_CUDA(ctx, cudaGetLastError());
    }
    if (idx) {
        *idx = c->sp_idx;
    }
    if (val) {
        *val = c->sp_val;
    }
    if (nnz) {
        *nnz = count;
    }
    return SGPU_OK;
}

int sgpu_counts_sparse_add(sgpu_ctx *ctx, sgpu_counts *c, int first_plane, const uint32_t *idx, const int32_t *val, uint64_t nnz) {
    SGPU_TRY(planes_ready(ctx, c));
    if (first_plane < 0 || first_plane > c->planes_used) {
        return sgpu_fail(ctx, SGPU_E_ARG, "first plane %d outside the %d planes in use", first_plane, c->planes_used);
    }
    if (nnz) {
        SGPU_LAUNCH(ctx, (sparse_add_kernel<<<static_cast<unsigned>((nnz + 255) / 256), 256, 0, ctx->stream>>>(
                              c->i32 + static_cast<uint64_t>(first_plane) * c->nn, idx, val, nnz)));
        SGPU_CUDA(ctx, cudaGetLastError());
        c->fresh = false;
    }
    return SGPU_OK;
}

int sgpu_counts_download(sgpu_ctx *ctx, sgpu_counts *c, int32_t *S1, int32_t *D1, int32_t *H, uint64_t *hist) {
    SGPU_TRY(planes_ready(ctx, c));
    cudaStream_t st = ctx->stream;
    const uint64_t nn = c->nn, n = c->n;
    std::vector<int32_t> tmp(nn);
    auto fetch_sym = [&](int plane, int32_t *dst) -> int {
        SGPU_CUDA(ctx, cudaMemcpyAsync(tmp.data(), c->i32 + plane * nn, nn * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        SGPU_CUDA(ctx, cudaStreamSynchronize(st));
        for (uint64_t i = 0; i < n; ++i) {
            dst[i * n + i] = 0;
            for (uint64_t j = i + 1; j < n; ++j) {
                dst[i * n + j] = dst[j * n + i] = tmp[i * n + j];
            }
        }
        return SGPU_OK;
    };
    if (S1) {
        SGPU_TRY(fetch_sym(PLANE_S, S1));
    }
    if (D1) {
        SGPU_TRY(fetch_sym(PLANE_D, D1));
    }
    if (H) {
        for (int k = 0; k < 3; ++k) {
            SGPU_TRY(fetch_sym(PLANE_H2 + k, H + k * nn));
        }
    }
    if (hist) {
        SGPU_CUDA(ctx, cudaMemcpyAsync(hist, c->hist, SGPU_MAX_CLASS * SGPU_MAX_CLASS * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        SGPU_CUDA(ctx, cudaStreamSynchronize(st));
    }
    return SGPU_OK;
}

int sgpu_similarity_finalize(sgpu_ctx *ctx, sgpu_counts *c, uint32_t max_fragment_length, double mutation_rate,
                             double homozygous_rate, double seq_error_rate, int normalization, double *out,
                             sgpu_stats *stats) {
    SGPU_TRY(planes_ready(ctx, c));
    if (c->have_params && c->spill
        && (c->eps != mutation_rate || c->h != homozygous_rate || c->theta != seq_error_rate || c->L != max_fragment_length)) {
        return sgpu_fail(ctx, SGPU_E_ARG, "finalize called with likelihood parameters different from accumulate");
    }
    EventTimer t(ctx->stream);
    SGPU_TRY(sgpu_epilogue(ctx, c, max_fragment_length, mutation_rate, homozygous_rate, seq_error_rate, normalization, out));
    const float ms = t.stop();
    if (stats) {
        stats->ms_epilogue = ms;
    }
    return SGPU_OK;
}

int sgpu_similarity_finalize_async(sgpu_ctx *ctx, sgpu_counts *c, uint32_t max_fragment_length, double mutation_rate,
                                   double homozygous_rate, double seq_error_rate, int normalization, double *out) {
    SGPU_TRY(planes_ready(ctx, c));
    if (!out) {
        return sgpu_fail(ctx, SGPU_E_ARG, "finalize_async needs a (page-locked) host buffer");
    }
    if (c->have_params && c->spill
        && (c->eps != mutation_rate || c->h != homozygous_rate || c->theta != seq_error_rate || c->L != max_fragment_length)) {
        return sgpu_fail(ctx, SGPU_E_ARG, "finalize called with likelihood parameters different from accumulate");
    }
    return sgpu_epilogue(ctx, c, max_fragment_length, mutation_rate, homozygous_rate, seq_error_rate, normalization, out, nullptr, true);
}

int sgpu_output_wait(sgpu_ctx *ctx) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    return sgpu_output_wait_impl(ctx);
}

int sgpu_similarity(sgpu_ctx *ctx, const sgpu_pileup *filtered, uint32_t num_cells, uint32_t max_fragment_length,
                    const uint32_t *group_id_to_pos, uint32_t n_groups, double mutation_rate, double homozygous_rate,
                    double seq_error_rate, uint32_t num_threads, int normalization, int path, double *out,
                    sgpu_stats *stats) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    if (normalization < 0 || normalization > 2) {
        return sgpu_fail(ctx, SGPU_E_ARG, "Invalid normalization: %d", normalization);
    }
    sgpu_counts *c = nullptr;
    SGPU_TRY(sgpu_counts_create(ctx, num_cells, &c));
    sgpu_stats s;
    std::memset(&s, 0, sizeof(s));
    int rc = sgpu_counts_accumulate(ctx, c, filtered, max_fragment_length, group_id_to_pos, n_groups, mutation_rate,
                                    homozygous_rate, seq_error_rate, num_threads, path, &s);
    if (rc == SGPU_OK) { // one-shot call: nothing to overlap the tensor kernel with; its time belongs to these statistics
        rc = sgpu_tensor_poll(ctx, true);
        sgpu_tensor_take_times(ctx, &s.ms_gemm, &s.gemm_launches);
    }
    if (rc == SGPU_OK) {
        rc = sgpu_similarity_finalize(ctx, c, max_fragment_length, mutation_rate, homozygous_rate, seq_error_rate,
                                      normalization, out, &s);
    }
    sgpu_counts_free(ctx, c);
    if (stats) {
        *stats = s;
    }
    return rc;
}

// ---- multi-GPU epilogue over peer memory ----------------------------------------------------------
int sgpu_slab_raw(sgpu_ctx *ctx, sgpu_counts *c, const int32_t *const *peer_planes, const double *const *peer_spill,
                  uint32_t n_peers, uint32_t slab, uint32_t n_slabs, uint32_t max_fragment_length, double mutation_rate,
                  double homozygous_rate, double seq_error_rate, double **extrema) {
    SGPU_TRY(planes_ready(ctx, c));
    // the spill plane holds G(x_s, x_d) evaluated with the accumulation's parameters; F and G must not be mixed
    if (c->have_params && c->spill
        && (c->eps != mutation_rate || c->h != homozygous_rate || c->theta != seq_error_rate || c->L != max_fragment_length)) {
        return sgpu_fail(ctx, SGPU_E_ARG, "slab epilogue called with likelihood parameters different from accumulate");
    }
    return sgpu_slab_raw_impl(ctx, c, peer_planes, peer_spill, n_peers, slab, n_slabs, max_fragment_length, mutation_rate,
                              homozygous_rate, seq_error_rate, extrema);
}

int sgpu_slab_finalize(sgpu_ctx *ctx, sgpu_counts *c, int normalization, double *out, double **device_out) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    return sgpu_slab_finalize_impl(ctx, c, normalization, out, device_out);
}

int sgpu_slab_range(const sgpu_counts *c, uint64_t *tile0, uint64_t *tile1) {
    if (!c) {
        return SGPU_E_ARG;
    }
    if (tile0) {
        *tile0 = c->slab_t0;
    }
    if (tile1) {
        *tile1 = c->slab_t1;
    }
    return SGPU_OK;
}

int sgpu_counts_ipc_handle(sgpu_ctx *ctx, sgpu_counts *c, int which, void *handle) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    static_assert(sizeof(cudaIpcMemHandle_t) == SGPU_IPC_HANDLE_BYTES, "IPC handle size");
    if (which == 1 && !c->spill) {
        return sgpu_fail(ctx, SGPU_E_ARG, "no spill plane (sgpu_counts_set_layout with want_spill creates it)");
    }
    cudaIpcMemHandle_t h;
    SGPU_CUDA(ctx, cudaIpcGetMemHandle(&h, which == 1 ? static_cast<void *>(c->spill) : static_cast<void *>(c->i32)));
    std::memcpy(handle, &h, sizeof(h));
    return SGPU_OK;
}

int sgpu_ipc_open(sgpu_ctx *ctx, const void *handle, void **device_ptr) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, sizeof(h));
    SGPU_CUDA(ctx, cudaIpcOpenMemHandle(device_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return SGPU_OK;
}

int sgpu_ipc_close(sgpu_ctx *ctx, void *device_ptr) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    SGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    SGPU_CUDA(ctx, cudaIpcCloseMemHandle(device_ptr));
    return SGPU_OK;
}

int sgpu_host_register(sgpu_ctx *ctx, void *host, uint64_t bytes, void **device_alias) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    SGPU_CUDA(ctx, cudaHostRegister(host, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped));
    SGPU_CUDA(ctx, cudaHostGetDevicePointer(device_alias, host, 0));
    return SGPU_OK;
}

int sgpu_host_unregister(sgpu_ctx *ctx, void *host) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    SGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    SGPU_CUDA(ctx, cudaHostUnregister(host));
    return SGPU_OK;
}

int sgpu_counts_checksum(sgpu_ctx *ctx, sgpu_counts *c, const int32_t *const *peer_planes, uint32_t n_peers, uint32_t slab,
                         uint32_t n_slabs, uint64_t *checksum) {
    SGPU_TRY(planes_ready(ctx, c));
    if (n_peers > SGPU_MAX_PEERS || n_slabs == 0 || slab >= n_slabs) {
        return sgpu_fail(ctx, SGPU_E_ARG, "checksum: %u peers, slab %u of %u", n_peers, slab, n_slabs);
    }
    ChecksumArgs a;
    for (uint32_t q = 0; q < SGPU_MAX_PEERS; ++q) {
        a.peer[q] = (peer_planes && q < n_peers) ? peer_planes[q] : nullptr;
    }
    if (!peer_planes || n_peers == 0) {
        a.peer[0] = c->i32;
        n_peers = 1;
    }
    a.n_peers = n_peers;
    a.n = c->n;
    a.nn = c->nn;
    a.planes = c->planes_used;
    const uint32_t nb = (c->n + 31) / 32;
    const uint64_t n_tiles = static_cast<uint64_t>(nb) * (nb + 1) / 2;
    a.t0 = n_tiles * slab / n_slabs;
    a.t1 = n_tiles * (slab + 1) / n_slabs;
    a.nb = nb;
    DevBuf<unsigned long long> d_sum;
    SGPU_CUDA(ctx, d_sum.alloc(1, ctx));
    SGPU_CUDA(ctx, cudaMemsetAsync(d_sum.p, 0, sizeof(unsigned long long), ctx->stream));
    if (a.t1 > a.t0) {
        const unsigned grid = static_cast<unsigned>(std::min<uint64_t>(a.t1 - a.t0, static_cast<uint64_t>(ctx->sm_count) * 16));
        SGPU_LAUNCH(ctx, (checksum_kernel<<<grid, 256, 0, ctx->stream>>>(a, d_sum.p)));
        SGPU_CUDA(ctx, cudaGetLastError());
    }
    SGPU_CUDA(ctx, cudaMemcpyAsync(&ctx->h_scratch[0], d_sum.p, sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    SGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *checksum = ctx->h_scratch[0];
    return SGPU_OK;
}

int sgpu_log_probs(sgpu_ctx *ctx, double mutation_rate, double homozygous_rate, double seq_error_rate,
                   uint32_t max_fragment_length, uint32_t n, double *ls, double *ld) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    return sgpu_log_probs_impl(ctx, mutation_rate, homozygous_rate, seq_error_rate, max_fragment_length, n, ls, ld);
}

int sgpu_expectation_maximization(sgpu_ctx *ctx, const sgpu_pileup *filtered, const uint32_t *id_to_pos, uint32_t n_groups,
                                  double theta, double *prob_cluster_b, uint32_t n_cells, uint32_t max_iterations,
                                  uint32_t *iterations, float *ms) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!filtered) {
        return sgpu_fail(ctx, SGPU_E_ARG, "expectation_maximization: no pileup");
    }
    if (filtered->wide) {
        return sgpu_fail(ctx, SGPU_E_ARG, "expectation_maximization: wide pileups (> 16 383 groups) are not supported");
    }
    return sgpu_em_impl(ctx, filtered, id_to_pos, n_groups, theta, prob_cluster_b, n_cells, max_iterations, iterations, ms);
}

// ---- Laplacian + leading eigenpairs (spectral.cu) ----
static int upload_matrix(sgpu_ctx *ctx, const double *h, uint32_t n, DevBuf<double> &d) {
    if (!h || n == 0) {
        return sgpu_fail(ctx, SGPU_E_ARG, "similarity matrix missing");
    }
    SGPU_CUDA(ctx, d.alloc(static_cast<size_t>(n) * n, ctx));
    SGPU_CUDA(ctx, cudaMemcpyAsync(d.p, h, static_cast<size_t>(n) * n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    return SGPU_OK;
}

int sgpu_laplacian(sgpu_ctx *ctx, const double *similarity, uint32_t n, double *out) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    DevBuf<double> d;
    SGPU_TRY(upload_matrix(ctx, similarity, n, d));
    return sgpu_laplacian_device(ctx, d.p, n, out);
}

int sgpu_spectral_embedding(sgpu_ctx *ctx, const double *similarity, uint32_t n, uint32_t k, double tol,
                            double *eigenvalues, double *eigenvectors, sgpu_spectral_stats *stats) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    DevBuf<double> d;
    SGPU_TRY(upload_matrix(ctx, similarity, n, d));
    return sgpu_spectral_device(ctx, d.p, n, k, tol, eigenvalues, eigenvectors, stats);
}

int sgpu_similarity_finalize_spectral(sgpu_ctx *ctx, sgpu_counts *c, uint32_t max_fragment_length, double mutation_rate,
                                      double homozygous_rate, double seq_error_rate, int normalization, double *out,
                                      uint32_t k, double tol, double *eigenvalues, double *eigenvectors, sgpu_stats *stats,
                                      sgpu_spectral_stats *spectral_stats) {
    SGPU_TRY(planes_ready(ctx, c));
    if (c->have_params && c->spill
        && (c->eps != mutation_rate || c->h != homozygous_rate || c->theta != seq_error_rate || c->L != max_fragment_length)) {
        return sgpu_fail(ctx, SGPU_E_ARG, "finalize called with likelihood parameters different from accumulate");
    }
    double *d_mat = nullptr;
    EventTimer t(ctx->stream);
    SGPU_TRY(sgpu_epilogue(ctx, c, max_fragment_length, mutation_rate, homozygous_rate, seq_error_rate, normalization, out, &d_mat));
    const float ms = t.stop();
    if (stats) {
        stats->ms_epilogue = ms;
    }
    if (!d_mat) {
        return sgpu_fail(ctx, SGPU_E_ARG, "spectral: empty similarity matrix");
    }
    const int rc = sgpu_spectral_device(ctx, d_mat, c->n, k, tol, eigenvalues, eigenvectors, spectral_stats);
    sgpu_dev_free(ctx, d_mat);
    return rc;
}

int sgpu_laplacian_eigenvalues(sgpu_ctx *ctx, const double *similarity, uint32_t n, double *eigenvalues,
                               sgpu_eigenvalue_stats *stats) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    DevBuf<double> d;
    SGPU_TRY(upload_matrix(ctx, similarity, n, d));
    return sgpu_eigenvalues_device(ctx, d.p, n, eigenvalues, stats);
}

int sgpu_similarity_finalize_eigenvalues(sgpu_ctx *ctx, sgpu_counts *c, uint32_t max_fragment_length, double mutation_rate,
                                         double homozygous_rate, double seq_error_rate, int normalization, double *out,
                                         double *eigenvalues, sgpu_stats *stats, sgpu_eigenvalue_stats *eig_stats) {
    SGPU_TRY(planes_ready(ctx, c));
    if (c->have_params && c->spill
        && (c->eps != mutation_rate || c->h != homozygous_rate || c->theta != seq_error_rate || c->L != max_fragment_length)) {
        return sgpu_fail(ctx, SGPU_E_ARG, "finalize called with likelihood parameters different from accumulate");
    }
    double *d_mat = nullptr;
    EventTimer t(ctx->stream);
    SGPU_TRY(sgpu_epilogue(ctx, c, max_fragment_length, mutation_rate, homozygous_rate, seq_error_rate, normalization, out, &d_mat));
    const float ms = t.stop();
    if (stats) {
        stats->ms_epilogue = ms;
    }
    if (!d_mat) {
        return sgpu_fail(ctx, SGPU_E_ARG, "eigenvalues: empty similarity matrix");
    }
    const int rc = sgpu_eigenvalues_device(ctx, d_mat, c->n, eigenvalues, eig_stats);
    sgpu_dev_free(ctx, d_mat);
    return rc;
}

int sgpu_spectral_matvec(sgpu_ctx *ctx, const double *M, uint32_t n, int width, const double *X, const double *W, double alpha,
                         double beta, double gamma, double *out) {
    SGPU_CUDA(ctx, cudaSetDevice(ctx->device));
    return sgpu_spectral_matvec_host(ctx, M, n, width, X, W, alpha, beta, gamma, out);
}

} // extern "C"
