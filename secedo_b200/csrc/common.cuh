// Shared declarations of the CUDA side of secedo_b200 (sm_100a only).
#pragma once

#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <deque>
#include <map>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/secedo_b200.h"

// ------------------------------------------------------------------------------------------------
// context / error handling
// ------------------------------------------------------------------------------------------------
struct sgpu_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr; // sgpu_pileup_upload_async
    // sgpu_similarity_finalize_async: the matrix goes to the host on its own stream while the next batch is computed
    cudaStream_t d2h_stream = nullptr;
    cudaEvent_t out_done = nullptr;
    void *pending_out = nullptr; // device matrix of the download in flight (returned to the cache by sgpu_output_wait)
    std::string error;
    // small pinned scratch for device->host scalars
    uint64_t *h_scratch = nullptr; // 64 x u64, pinned
    uint64_t *d_scratch = nullptr; // 64 x u64, device
    uint64_t launches = 0;         // kernels launched by this context (sgpu_launch_count)
    // device time of the dominant kernels not yet reported through sgpu_stats / sgpu_tensor_times, from CUDA events
    // recorded on ctx->stream around the launches
    float ms_syrk = 0.f, ms_stage = 0.f;
    uint64_t n_syrk = 0;
    // gemm.cu: the tensor kernel of a first-order accumulation runs on a stream of its own (highest priority), behind an
    // event of the staging kernel, and the call returns without waiting for it: the filter / read linking / staging
    // kernels of the NEXT batch (issue and latency bound, on ctx->stream) then run beside it on the same SMs (the tensor
    // kernel keeps one CTA of 6 warps per SM and leaves ~95 % of the issue slots idle). A job owns what its kernel reads
    // (the operand panel) until its end event has been seen; everything that touches the count planes first makes
    // ctx->stream wait for the last job (sgpu_tensor_join). SECEDO_B200_ASYNC_GEMM=0: the kernel runs on ctx->stream.
    cudaStream_t tensor_stream = nullptr;
    bool async_gemm = true;
    struct TensorJob {
        const void *planes = nullptr; // first of the count planes the kernel adds to (whom a join concerns)
        void *U = nullptr;   // operand panel (context cache)
        int *err = nullptr;  // [0] range check of the staging, [1] wave counter of the tensor kernel (context cache)
        cudaEvent_t t0 = nullptr, t1 = nullptr; // around the kernel, on the stream it was launched on
    };
    std::deque<TensorJob> tensor_jobs;
    void *pending_gemm = nullptr;        // gemm.cu: prepared launch of the last deferred tensor kernel, issued behind the next
                                         // batch's link_window kernel (sgpu_tensor_flush)
    std::vector<cudaEvent_t> event_pool; // recycled timing events
    // Kernels only share an SM with the tensor kernel while the DEVICE-WIDE cache preference is cudaFuncCachePreferShared: a
    // kernel with 16 KB of static shared memory otherwise waited for the whole tensor kernel, and neither the carve-out
    // attribute nor cudaFuncSetCacheConfig of that kernel changed it (profiles/coresidency_probe.cu, r2_coresidency.txt,
    // r2_overlap_probes.txt). The preference costs the kernels that run alone ~4 % (less L1), so it is only in force from
    // the launch of a deferred tensor kernel to the launch of the next batch's link_window kernel (which never fits beside
    // it). false: never switched (the host application keeps its own preference).
    bool prefer_shared = false;
    int cache_pref_now = -1;             // what this context last set (-1: nothing yet)
    // gemm.cu: rasterised list of upper-triangle output tiles for tile_cache_cells cells (device memory)
    void *tile_cache = nullptr;
    uint32_t tile_cache_n = 0, tile_cache_cells = 0;
    // epilogue.cu: F / G coefficients of the last likelihood parameters, tile list of the last matrix size
    bool ft_valid = false;
    double ft_eps = 0, ft_h = 0, ft_theta = 0, ft_f10 = 0, ft_f01 = 0, ft_g2[3] = { 0, 0, 0 }, ft_g3[4] = { 0, 0, 0, 0 };
    uint32_t ft_L = 0;
    void *ep_tiles = nullptr;
    uint32_t ep_tiles_n = 0;
    bool spectral_attr_done = false; // spectral.cu: shared-memory attributes of its kernels set on this device
    // Device memory cache (abi.cu): temporaries and pileups are re-created with identical sizes at every
    // call, and cudaMallocAsync/cudaFreeAsync of GB-sized blocks cost milliseconds each, so freed blocks
    // are kept and handed out again. Reuse is safe because all work of a context is ordered on ONE stream.
    std::multimap<size_t, void *> free_blocks;
    std::unordered_map<void *, size_t> live_blocks;
    size_t cached_bytes = 0;
    // SECEDO_B200_TRACE=1: synchronise and print the wall-clock time between trace points (debug aid)
    bool trace = false;
    bool trace_alloc = false; // SECEDO_B200_TRACE=2: log every real cudaMalloc
    double trace_t0 = 0.0;
};

void sgpu_trace_point(sgpu_ctx *ctx, const char *what);
#define SGPU_TRACE(ctx, what)            \
    do {                                 \
        if ((ctx)->trace) {              \
            sgpu_trace_point((ctx), (what)); \
        }                                \
    } while (0)

#define SGPU_LAUNCH(ctx, call) \
    do {                       \
        ++(ctx)->launches;     \
        call;                  \
    } while (0)

int sgpu_fail(sgpu_ctx *ctx, int code, const char *fmt, ...);
// device-wide shared-memory / L1 preference, switched only when it changes (see sgpu_ctx::prefer_shared)
int sgpu_cache_preference(sgpu_ctx *ctx, bool shared);
// gemm.cu — tensor kernels in flight on ctx->tensor_stream (see sgpu_ctx::tensor_jobs)
int sgpu_tensor_poll(sgpu_ctx *ctx, bool wait_all); // retire finished jobs (timing, operand panel back to the cache)
// ctx->stream waits (on the device) for the last job that writes the count planes starting at `planes` (null: any job); a
// launch still held back is issued first if it writes them. A caller that alternates between two counts objects thereby
// keeps the other object's tensor kernel in flight (or held back) across its epilogue.
int sgpu_tensor_join(sgpu_ctx *ctx, const void *planes = nullptr);
int sgpu_tensor_flush(sgpu_ctx *ctx, bool after_main); // issue the prepared launch, if any (after_main: behind everything queued on ctx->stream)
// make the context's stream wait for an asynchronously uploaded pileup
#define SGPU_WAIT_PILEUP(ctx, p)                                                                   \
    do {                                                                                           \
        if ((p) && (p)->ready) {                                                                   \
            SGPU_CUDA((ctx), cudaStreamWaitEvent((ctx)->stream, (p)->ready, 0));                   \
        }                                                                                          \
    } while (0)

#define SGPU_CUDA(ctx, expr)                                                                       \
    do {                                                                                           \
        cudaError_t err__ = (expr);                                                                \
        if (err__ != cudaSuccess) {                                                                \
            return sgpu_fail((ctx), SGPU_E_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #expr,      \
                             cudaGetErrorString(err__));                                           \
        }                                                                                          \
    } while (0)

#define SGPU_TRY(expr)                                                                             \
    do {                                                                                           \
        int rc__ = (expr);                                                                         \
        if (rc__ != SGPU_OK) {                                                                     \
            return rc__;                                                                           \
        }                                                                                          \
    } while (0)

// Kernels that read (group << 2 | base) entries are templates over the entry type; SGPU_GB runs CALL with GB = uint16_t or
// uint32_t and gid_base_ pointing to the array the pileup holds.
#define SGPU_GB(p, CALL)                                      \
    do {                                                      \
        if ((p)->wide) {                                      \
            using GB = uint32_t;                              \
            const GB *gid_base_ = (p)->d_gid_base32;          \
            CALL;                                             \
        } else {                                              \
            using GB = uint16_t;                              \
            const GB *gid_base_ = (p)->d_gid_base;            \
            CALL;                                             \
        }                                                     \
    } while (0)

struct sgpu_pileup;
// copy lazily uploaded read ids to the device and gather viewed ones (see sgpu_pileup::view_read_id) into an array of the
// pileup's own (no-op otherwise); stream ordered on ctx->stream. keep_view: leave a view as it is (the read linking reads
// through it)
int sgpu_pileup_materialize(sgpu_ctx *ctx, const sgpu_pileup *p, bool keep_view = false);

// device memory from the context's cache (see sgpu_ctx::free_blocks)
cudaError_t sgpu_dev_alloc(sgpu_ctx *ctx, void **p, size_t bytes);
void sgpu_dev_free(sgpu_ctx *ctx, void *p);
void sgpu_dev_release_cache(sgpu_ctx *ctx);

template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    sgpu_ctx *c = nullptr;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { release(); }
    cudaError_t alloc(size_t count, sgpu_ctx *ctx) {
        release();
        c = ctx;
        n = count;
        if (count == 0) {
            return cudaSuccess;
        }
        return sgpu_dev_alloc(ctx, reinterpret_cast<void **>(&p), count * sizeof(T));
    }
    void release() {
        if (p) {
            sgpu_dev_free(c, p);
            p = nullptr;
        }
        n = 0;
    }
    T *take() { // hand ownership to the caller
        T *q = p;
        p = nullptr;
        n = 0;
        return q;
    }
};

// ------------------------------------------------------------------------------------------------
// device-resident objects
// ------------------------------------------------------------------------------------------------
struct sgpu_pileup {
    uint32_t n_chr = 0;
    uint64_t n_loci = 0;
    uint64_t n_entries = 0;
    uint64_t *h_chr_ptr = nullptr; // host copy, n_chr + 1
    uint64_t *d_chr_ptr = nullptr; // device copy
    uint64_t *d_row_ptr = nullptr;
    uint32_t *d_position = nullptr;
    uint32_t *d_read_id = nullptr;
    uint16_t *d_gid_base = nullptr;   // group id << 2 | base, 14-bit group ids (the reference's PosData)
    uint32_t *d_gid_base32 = nullptr; // the same with 30-bit group ids (wide pileups: more than 16 383 cells / groups)
    bool wide = false;                // d_gid_base32 is the one in use; NO_POS is 0xFFFFFFFF instead of 16383
    bool owns = true;
    // sgpu_pileup_upload_lazy_async: the read ids stay in the caller's pinned host memory (zc_read_id is its device
    // alias) and d_read_id is null until somebody other than the filter needs them (sgpu_pileup_materialize)
    const uint32_t *zc_read_id = nullptr;
    // Filtered pileup whose read ids are a VIEW of the pileup the filter read (filter.cu; only when every group belongs to
    // the sub-cluster, so that the entries of a kept locus are one contiguous run of the source): view_read_id is the
    // source's array and view_off[l] the first source entry of locus l. The read linking - the only dense reader of the
    // ids - reads through the view; d_read_id stays null until somebody else asks (sgpu_pileup_materialize gathers). The
    // source outlives its views: sgpu_pileup_free of a pileup with live views is deferred until the last one is gone.
    const uint32_t *view_read_id = nullptr;
    uint64_t *view_off = nullptr;     // context cache, n_loci values
    sgpu_pileup *view_src = nullptr;
    std::atomic<int> view_refs{ 0 };  // views that read THIS pileup's ids
    bool zombie = false;              // freed by the caller while views were alive
    sgpu_ctx *zombie_ctx = nullptr;   // the context that free was asked of
    cudaEvent_t ready = nullptr;   // set by sgpu_pileup_upload_async: the copies are done
    mutable uint32_t max_row = 0;  // entries of the largest locus (0 = not known yet; cached by reads.cu)
};

// Owners of half-built objects: an error return (SGPU_CUDA / SGPU_TRY) between `new` and the hand-over to the caller frees
// the object and gives its device blocks back to the context's cache (ADVICE r1).
extern "C" void sgpu_pileup_free(sgpu_ctx *ctx, sgpu_pileup *p);
struct PileupOwner {
    sgpu_ctx *ctx;
    sgpu_pileup *p;
    PileupOwner(sgpu_ctx *c, sgpu_pileup *q) : ctx(c), p(q) {}
    PileupOwner(const PileupOwner &) = delete;
    PileupOwner &operator=(const PileupOwner &) = delete;
    ~PileupOwner() {
        if (p) {
            sgpu_pileup_free(ctx, p);
        }
    }
    sgpu_pileup *release() {
        sgpu_pileup *q = p;
        p = nullptr;
        return q;
    }
};

// plane indices inside sgpu_counts::i32
enum { PLANE_S = 0, PLANE_D = 1, PLANE_H2 = 2 /* (2,0),(1,1),(0,2) */, PLANE_H3 = 5 /* (3,0)..(0,3) */, N_PLANES = 9 };

struct sgpu_counts {
    uint32_t n = 0;             // num_cells
    uint64_t nn = 0;            // n*n
    sgpu_ctx *owner = nullptr;  // the context it was created with (sgpu_counts_buffers has no context argument)
    int32_t *i32 = nullptr;     // N_PLANES planes of n*n, only the upper triangle (i<j) is meaningful
    int planes_used = 2;        // 2, 5 or 9: planes that can be non-zero
    int planes_dirty = N_PLANES; // planes to clear at the next sgpu_counts_zero
    bool fresh = false;         // S and D are all zero (nothing accumulated since sgpu_counts_zero)
    bool poisoned = false;      // a failed call left a partial sum in the planes: only sgpu_counts_zero / free are accepted
    int32_t *packed = nullptr;  // upper triangles of the planes in use, for the cross-rank reduction (lazy)
    uint64_t packed_n = 0;
    uint32_t *sp_idx = nullptr; // non-zeros of the sparse (second / third order) planes as (index, value) lists (lazy)
    int32_t *sp_val = nullptr;
    uint64_t sp_cap = 0;
    double *spill = nullptr;    // n*n doubles: sum of G(x_s,x_d) over pairs with x_s+x_d >= 4 (lazy)
    uint64_t *hist = nullptr;   // SGPU_MAX_CLASS^2 class histogram (pairs with x_s+x_d >= 2)
    // log-likelihood parameters the spill plane was accumulated with (must match at finalize)
    bool have_params = false;
    double eps = 0, h = 0, theta = 0;
    uint32_t L = 0;
    // multi-GPU epilogue over peer memory (sgpu_slab_raw / sgpu_slab_finalize): this GPU's share of the 32 x 32 tiles of
    // the upper triangle, their raw (summed, transformed, not yet normalised) values, local extrema
    uint64_t slab_t0 = 0, slab_t1 = 0, slab_raw_tiles = 0;
    uint32_t slab_nb = 0;
    double *slab_raw = nullptr;               // context cache
    unsigned long long *slab_minmax = nullptr; // cudaMalloc: encoded {min, max}, then {-min, max} as doubles
    double *slab_out = nullptr;               // cudaMalloc, n x n, only when the result stays on the device
};

// ------------------------------------------------------------------------------------------------
// entry "codes" produced by read linking (reads.cu) and consumed by scatter / staging / multilocus
//   bit 31      dropped (mate rule) -> whole word is CODE_DROPPED
//   bits 4..30  cell index (mapped through group_id_to_pos, taken from the read's FIRST entry)
//   bits 2..3   base
//   bit 1       tail: read index >= K, never the first read of a pair
//   bit 0       multi: the read keeps >= 2 loci
// ------------------------------------------------------------------------------------------------
constexpr uint32_t CODE_DROPPED = 0xFFFFFFFFu;
__host__ __device__ inline uint32_t code_cell(uint32_t c) { return c >> 4; }
__host__ __device__ inline uint32_t code_base(uint32_t c) { return (c >> 2) & 3u; }
__host__ __device__ inline bool code_tail(uint32_t c) { return (c >> 1) & 1u; }
__host__ __device__ inline bool code_multi(uint32_t c) { return c & 1u; }

struct LinkResult {
    // Entries that share their read with another entry are "special"; all other entries are the
    // only entry of their read (cell = own group, created at the own locus, never dropped).
    DevBuf<uint32_t> sp_bits;   // bitmap over entries: bit e set = special
    DevBuf<uint64_t> sp_rank;   // per bitmap word: number of special entries before it (dense numbering "sid")
    DevBuf<uint32_t> sp_entry;  // per sid: entry index (ascending)
    DevBuf<uint32_t> sp_locus;  // per sid: locus index
    DevBuf<uint32_t> sp_start;  // per locus (n_loci + 1): first sid of the locus (all zero without special entries)
    DevBuf<uint32_t> sp_head;   // per sid: sid of the first entry of the read
    DevBuf<uint32_t> sp_code;   // per sid: code, see above
    DevBuf<uint8_t> sp_drop;    // per sid: removed by the mate rule
    DevBuf<uint32_t> sp_rcode;  // per head: cell << 4 | tail << 1 | multi of the READ (set even if the head entry is dropped)
    // per read with >= 2 entries, indexed by the sid of its first entry ("head")
    DevBuf<uint64_t> g_off;     // [n_special + 1] offsets into g_list / g_base (only heads own a range)
    DevBuf<uint32_t> g_list;    // stored loci, ascending (first g_nst[head] elements of the range)
    DevBuf<uint8_t> g_base;     // stored bases
    DevBuf<uint32_t> g_nst;     // per head: number of loci the read keeps after the mate rule
    uint64_t n_special = 0;
    // candidates of the multi-locus correction: surviving entries of reads that keep >= 2 loci and keep
    // one AFTER the entry's own locus (a pair is accounted at its first common locus, so it needs a
    // later one). Compact, in entry order; the count stays on the device (me_idx[n_special]).
    DevBuf<uint64_t> me_idx;    // scan of the candidate flags
    DevBuf<uint32_t> me_code;   // cell << 4 | base << 2 | tail << 1 | 1
    DevBuf<uint32_t> me_locus;
    DevBuf<uint32_t> me_pos;    // index into g_list / g_base of the element stored for this locus
    DevBuf<uint32_t> me_beg;    // stored list of the read: [me_beg, me_end)
    DevBuf<uint32_t> me_end;
    // per locus / chromosome
    DevBuf<uint8_t> lchr;        // chromosome of every locus
    DevBuf<uint64_t> tail_locus; // per chromosome: reads created at loci >= this one have index >= K
    std::vector<uint64_t> h_tail_locus; // host copy
    DevBuf<uint32_t> tail_loci;  // loci that can hold tail reads (from the cutoff locus to the chromosome end)
    uint64_t n_tail_loci = 0;
    DevBuf<uint32_t> gmap;       // group_id_to_pos on the device
    uint32_t n_groups = 0, num_cells = 0;
    bool gmap_identity = false;  // group g is cell g (the root of the recursion): the partition kernel needs no table
    // Ranged accumulation (sgpu_counts_accumulate_range): the pileup is a piece of its chromosomes plus halos; only the
    // OWNED loci contribute first-order counts, and a multi-locus pair is accounted by the piece that owns its first
    // common locus. Not ranged: everything is owned (owned.p == nullptr, own_loci.p == nullptr).
    bool ranged = false;
    DevBuf<uint8_t> owned;       // per locus
    DevBuf<uint32_t> own_loci;   // owned loci, ascending
    uint64_t n_own = 0;
    DevBuf<uint32_t> code;       // dense per-entry codes, only built for the pair-scatter path
    uint64_t n_reads = 0, n_multi = 0, n_dropped = 0, n_tail = 0;
    uint64_t n_span_splits = 0;  // reads opened because a read id was chained over >= max_fragment_length (see split_span_kernel)
};

// ------------------------------------------------------------------------------------------------
// kernels' host launchers (one translation unit each)
// ------------------------------------------------------------------------------------------------
// scan.cu — exclusive prefix sum, out has n + 1 elements (out[n] = total)
int sgpu_scan_u8_u64(sgpu_ctx *ctx, const uint8_t *in, uint64_t *out, uint64_t n);
int sgpu_scan_u32_u64(sgpu_ctx *ctx, const uint32_t *in, uint64_t *out, uint64_t n);

// filter.cu
int sgpu_filter_impl(sgpu_ctx *ctx, const sgpu_pileup *in, const uint32_t *h_id_to_pos, uint32_t n_groups,
                     double theta, int cell_proportion, sgpu_pileup **filtered, double *avg_coverage);
int sgpu_is_significant_impl(sgpu_ctx *ctx, const uint16_t *h_counts4, uint64_t n, double theta,
                             int cell_proportion, uint8_t *h_out);

// reads.cu
// Ownership of a ranged call, one entry per chromosome of the pileup: the loci with position in [own_pos_begin,
// own_pos_end) are owned; reads created at positions >= tail_position have index >= K (from sgpu_chromosome_cutoff).
struct RangeSpec {
    const uint32_t *own_pos_begin, *own_pos_end, *tail_position;
};
struct CutoffQuery { // suffix mode: only the cutoff is computed (host arrays, one entry per chromosome)
    const uint8_t *whole;      // in: the chromosome is complete (not just its end)
    uint32_t *tail_position;   // out
    uint8_t *resolved;         // out
};
int sgpu_link_reads(sgpu_ctx *ctx, const sgpu_pileup *p, uint32_t num_cells, uint32_t L,
                    const uint32_t *h_group_id_to_pos, uint32_t n_groups, uint32_t num_threads,
                    LinkResult *out, const RangeSpec *range = nullptr, const CutoffQuery *cutq = nullptr);
// cutoff K of chromosomes of which only the END is given (suffix): per chromosome the position from which reads are
// tail reads, and whether the suffix was long enough to decide it
int sgpu_cutoff_from_suffix(sgpu_ctx *ctx, const sgpu_pileup *p, uint32_t L, uint32_t num_threads, const uint8_t *h_whole,
                            uint32_t *h_tail_position, uint8_t *h_resolved);
int sgpu_link_dense_codes(sgpu_ctx *ctx, const sgpu_pileup *p, LinkResult *lr);
// (re)build the compact candidate list of the multi-locus correction from the reads that keep >= min_nst loci
int sgpu_link_candidates(sgpu_ctx *ctx, LinkResult *lr, uint32_t min_nst);

// abi.cu — the measured cost model behind SGPU_PATH_AUTO (only n_loci and n_entries of the pileup are looked at)
int sgpu_choose_path(const sgpu_pileup *p, uint32_t num_cells);

// scatter.cu — first-order counts by pair enumeration; only_tail_pairs: enumerate just the pairs of
// two tail reads (used with sign = -1 to correct the GEMM path)
int sgpu_scatter_pairs(sgpu_ctx *ctx, const sgpu_pileup *p, const LinkResult &lr, sgpu_counts *c,
                       int sign, bool only_tail_pairs, uint64_t *n_pairs);

// multilocus.cu
int sgpu_multilocus(sgpu_ctx *ctx, const sgpu_pileup *p, LinkResult &lr, sgpu_counts *c,
                    uint32_t L, uint64_t *n_pairs_multi);

// epilogue.cu
// The log-probability power tables hold min(max(L, 2), LOGPROB_TBL) entries (similarity_matrix.cpp:42-67, capped like
// the oracle's): a class with x_s + x_d >= that length has no LS / LD and is refused
constexpr uint32_t LOGPROB_TBL = 132;
inline uint32_t logprob_table_len(uint32_t L) { return L < 2 ? 2u : (L > LOGPROB_TBL ? LOGPROB_TBL : L); }
struct FTable {
    double F[SGPU_MAX_CLASS * SGPU_MAX_CLASS]; // LD - LS, NaN where never needed
};
int sgpu_log_probs_impl(sgpu_ctx *ctx, double eps, double h, double theta, uint32_t L, uint32_t n,
                        double *h_ls, double *h_ld);
// d_keep != NULL: the device matrix is handed to the caller (free with sgpu_dev_free)
int sgpu_epilogue(sgpu_ctx *ctx, sgpu_counts *c, uint32_t L, double eps, double h, double theta,
                  int normalization, double *h_out, double **d_keep = nullptr, bool async_out = false);
int sgpu_output_wait_impl(sgpu_ctx *ctx);
int sgpu_slab_raw_impl(sgpu_ctx *ctx, sgpu_counts *c, const int32_t *const *peer_planes, const double *const *peer_spill,
                       uint32_t n_peers, uint32_t slab, uint32_t n_slabs, uint32_t L, double eps, double h, double theta,
                       double **d_extrema);
int sgpu_slab_finalize_impl(sgpu_ctx *ctx, sgpu_counts *c, int normalization, double *out, double **d_out);

// em.cu
int sgpu_em_impl(sgpu_ctx *ctx, const sgpu_pileup *p, const uint32_t *h_id_to_pos, uint32_t n_groups, double theta,
                 double *h_prob_b, uint32_t n_cells, uint32_t max_iterations, uint32_t *iterations, float *ms_total);

// spectral.cu
int sgpu_spectral_device(sgpu_ctx *ctx, const double *d_A, uint32_t n, uint32_t k, double tol, double *h_evals,
                         double *h_evecs, sgpu_spectral_stats *stats);
int sgpu_laplacian_device(sgpu_ctx *ctx, const double *d_A, uint32_t n, double *h_out);
int sgpu_spectral_matvec_host(sgpu_ctx *ctx, const double *h_M, uint32_t n, int width, const double *h_X, const double *h_W,
                              double alpha, double beta, double gamma, double *h_out);
// device table of G(s,d) = F(s,d) - s F(1,0) - d F(0,1) for the spill plane (SGPU_MAX_CLASS^2 doubles)
int sgpu_build_gtable(sgpu_ctx *ctx, double eps, double h, double theta, uint32_t L, uint32_t n,
                      double *d_G /* device, SGPU_MAX_CLASS^2 */, double *d_F /* device, optional */);

// gemm.cu — int8 tcgen05 path
struct GemmInput {
    const uint64_t *row_ptr;   // CSR over n_loci loci
    const uint16_t *gid_base;  // group << 2 | letter per entry (14-bit groups), or
    const uint32_t *gid_base32; // the same with wide groups (exactly one of the two is set)
    uint64_t n_loci, n_main;   // loci [0, n_main) are counted (main_loci != null: the loci main_loci[0 .. n_main)); other
                               // loci only through tail_loci
    const uint32_t *main_loci; // ascending list of the loci to count, or null
    uint64_t n_entries;
    const uint32_t *sp_bits;   // entries to leave out (staged from the special list instead)
    const uint32_t *gmap;      // group -> cell
    bool gmap_identity = false; // gmap[g] == g for every group
    uint32_t n_groups;
    const uint32_t *sp_code, *sp_locus, *sp_start; // special entries (may be empty: n_special = 0, sp_start all zero)
    uint64_t n_special;
    const uint32_t *tail_loci; // loci whose entries are subtracted as Z Z^T (ascending)
    uint64_t n_tail_loci;
    bool may_defer = false;    // the tensor kernel of the last panel may still be running when the call returns (see
                               // sgpu_ctx::tensor_jobs); false: the result is complete in the order of ctx->stream
};
int sgpu_gemm_run(sgpu_ctx *ctx, const GemmInput &in, uint32_t num_cells, int32_t *S_plane, int32_t *D_plane, bool *fresh,
                  bool *poisoned = nullptr);
// SGPU_E_COUNT_RANGE of the first panel is returned with the count planes untouched (SGPU_PATH_AUTO falls back to the
// scatter path); for later panels the counts object is marked as holding a partial sum
int sgpu_gemm_counts(sgpu_ctx *ctx, const sgpu_pileup *p, const LinkResult &lr, sgpu_counts *c, uint64_t *n_pairs);

static inline uint64_t ceil_div_u64(uint64_t a, uint64_t b) { return (a + b - 1) / b; }
