/*
 * secedo_b200 — C ABI of the B200-native similarity-matrix hot path of SECEDO.
 *
 * The reference has no FFI; its boundary for this path is two C++ functions
 *   Filter::filter(...)            util/is_significant.hpp:68-72   (body util/is_significant.cpp:149-193)
 *   computeSimilarityMatrix(...)   similarity_matrix.hpp:51-60     (body similarity_matrix.cpp:295-433)
 * called from divide_cluster (spectral_clustering.cpp:336-356). The entry points below are what a
 * host-side shim defining those two symbols binds (secedo_b200/host/secedo_b200_shim.cpp, INTEGRATION.md): plain
 * pointers and sizes, no C++ or torch types. One context drives ONE GPU; multi-GPU runs use one
 * process (and one context) per GPU and sum the count matrices between sgpu_counts_accumulate and
 * sgpu_similarity_finalize with a single NCCL reduction (secedo_b200/dist.py).
 *
 * Pileup layout (replaces std::vector<std::vector<PosData>>, sequenced_data.hpp:11-47):
 *   chr_ptr[n_chr+1]    u64  locus offsets per chromosome
 *   row_ptr[n_loci+1]   u64  entry offsets per locus
 *   position[n_loci]    u32  strictly increasing inside a chromosome
 *   read_id[n_entries]  u32  unique inside a chromosome (0xFFFFFFFF is reserved)
 *   gid_base[n_entries] u16  group id << 2 | base  (PosData::group_ids_bases)
 *
 * Every function returns 0 on success or a negative SGPU_E_* code; sgpu_last_error() gives the
 * text. There is no CPU fallback: without a usable CUDA device sgpu_init fails.
 */
#ifndef SECEDO_B200_H
#define SECEDO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SGPU_NO_POS 16383u   /* util/is_significant.hpp:11 */
#define SGPU_MAX_CLASS 64    /* overlap classes x_s, x_d < 64 are supported */
#define SGPU_MAX_PEERS 16    /* GPUs whose count planes one epilogue kernel can sum (sgpu_slab_raw) */
#define SGPU_IPC_HANDLE_BYTES 64

enum {
    SGPU_OK = 0,
    SGPU_E_CUDA = -1,          /* CUDA runtime error (text in sgpu_last_error) */
    SGPU_E_ARG = -2,           /* invalid argument (e.g. unknown normalization: the reference throws
                                  std::logic_error, similarity_matrix.cpp:264) */
    SGPU_E_CELL_RANGE = -3,    /* group id >= n_groups or mapped cell >= num_cells (mat.hpp:119 assert) */
    SGPU_E_FRAGMENT_SPAN = -4, /* a read id chained over >= max_fragment_length, only with SECEDO_B200_STRICT_SPAN=1 (by
                                  default such a chain is split into reads the way the reference's retirement does) */
    SGPU_E_CLASS_RANGE = -5,   /* a read pair overlaps in a class (x_s, x_d) without a log-likelihood: x_s or x_d >=
                                  SGPU_MAX_CLASS or >= L, or x_s + x_d >= min(max(L, 2), 132), the length of the
                                  reference's power tables (L = max_fragment_length) */
    SGPU_E_POSITIONS = -6,     /* loci not strictly increasing inside a chromosome */
    SGPU_E_COUNT_RANGE = -7,   /* internal int8/int32 range exceeded */
    SGPU_E_CONVERGENCE = -8    /* eigen-solver did not reach the tolerance (sgpu_spectral_embedding) */
};

/* similarity_matrix.hpp:9-17 */
enum { SGPU_NORM_ADD_MIN = 0, SGPU_NORM_EXPONENTIATE = 1, SGPU_NORM_SCALE_MAX_1 = 2 };

/* how the first-order same/different read-pair counts are produced */
enum {
    SGPU_PATH_AUTO = 0,    /* chosen from measured density (DESIGN.md) */
    SGPU_PATH_SCATTER = 1, /* per-locus cross-cell pair scatter, int32 atomics */
    SGPU_PATH_GEMM = 2     /* int8 tcgen05/TMEM GEMM on Hadamard-transformed per-base count planes */
};

typedef struct sgpu_ctx sgpu_ctx;
typedef struct sgpu_pileup sgpu_pileup; /* device-resident CSR pileup */
typedef struct sgpu_counts sgpu_counts; /* device-resident integer read-pair count matrices */

typedef struct sgpu_stats {
    uint64_t n_loci;            /* loci processed */
    uint64_t n_entries;         /* pileup entries processed */
    uint64_t n_reads;           /* distinct reads (fragments) */
    uint64_t n_dropped_entries; /* entries removed by the paired-end mate rule (similarity_matrix.cpp:387-395) */
    uint64_t n_multi_reads;     /* reads that keep >= 2 loci */
    uint64_t n_tail_reads;      /* reads with index >= K (never the first read of a pair, SURVEY F2) */
    uint64_t n_pairs_first;     /* cross-cell (read pair, shared locus) incidences counted */
    uint64_t n_pairs_multi;     /* read pairs overlapping at >= 2 loci */
    int32_t path_used;          /* SGPU_PATH_SCATTER or SGPU_PATH_GEMM */
    int32_t n_span_splits;      /* reads opened because a read id was chained over >= max_fragment_length (the reference
                                   retires a read once start + L <= position and starts a new one at the next entry with its
                                   id, similarity_matrix.cpp:348-372,379-382; 0 on ordinary pileups) */
    float ms_link;              /* device time: read linking + mate rule + cutoff K */
    float ms_first_order;       /* device time: scatter or staging + GEMM */
    float ms_multi;             /* device time: multi-locus correction */
    float ms_epilogue;          /* device time: log-likelihood transform + normalisation */
    float ms_stage;             /* GEMM path: count staging + Hadamard transform kernels */
    float ms_gemm;              /* GEMM path: the tcgen05 kernels that finished during the call (see sgpu_tensor_times) */
    uint64_t gemm_launches;     /* GEMM path: number of those kernels */
} sgpu_stats;

/* parameters of the device-side synthetic pileup generator (bench / large tests), DESIGN.md */
typedef struct sgpu_synth_params {
    uint32_t n_cells, n_chr, loci_per_chr, n_clones, spacing, reserved;
    float coverage, frac_somatic, frac_germline, theta, p_multi, p_mate, p_mate_mismatch, reserved2;
    uint64_t seed;
} sgpu_synth_params;

/* ---- context ---------------------------------------------------------------------------- */
int sgpu_init(int device, sgpu_ctx **ctx);
void sgpu_shutdown(sgpu_ctx *ctx);
const char *sgpu_last_error(const sgpu_ctx *ctx);
/* Run all work of this context on an existing CUDA stream (cudaStream_t); NULL restores the
 * context's own stream. */
int sgpu_set_stream(sgpu_ctx *ctx, void *cuda_stream);
int sgpu_synchronize(sgpu_ctx *ctx);
/* number of CUDA kernels this context has launched so far */
uint64_t sgpu_launch_count(const sgpu_ctx *ctx);
/* The first-order tensor kernel of sgpu_counts_accumulate runs on a stream of its own and the call returns without
 * waiting for it, so that the filter / read-linking / staging kernels of the caller's NEXT batch run beside it
 * (SECEDO_B200_ASYNC_GEMM=0 switches that off). Every call that reads or writes the count planes is ordered behind it;
 * sgpu_synchronize waits for it. sgpu_stats.ms_gemm / gemm_launches therefore cover the tensor kernels that FINISHED
 * during the call (usually the one of the batch before). This call waits for the kernels still in flight and returns
 * (and resets) the time and number of the kernels no sgpu_stats has reported yet. */
int sgpu_tensor_times(sgpu_ctx *ctx, float *ms, uint64_t *launches);
/* Scheduling knobs of a context (their defaults come from the environment variables of the same meaning, read by sgpu_init;
 * the results never depend on them). Waits for the context's work first. Names:
 *   "async_gemm"     1: the first-order tensor kernel runs on its own stream beside the next batch and is issued behind the
 *                    next batch's dense read-linking kernel (SECEDO_B200_ASYNC_GEMM)
 *   "prefer_shared"  1: device-wide cudaFuncCachePreferShared around the window in which kernels run beside a deferred
 *                    tensor kernel, 0: never switched; other values fail with SGPU_E_ARG (SECEDO_B200_PREFER_SHARED;
 *                    default: on when async_gemm is on at sgpu_init) */
int sgpu_set_option(sgpu_ctx *ctx, const char *name, int value);

/* ---- pileup staging (replaces the host vector<vector<PosData>>) --------------------------- */
int sgpu_pileup_upload(sgpu_ctx *ctx, uint32_t n_chr, const uint64_t *chr_ptr, const uint64_t *row_ptr,
                       const uint32_t *position, const uint32_t *read_id, const uint16_t *gid_base,
                       sgpu_pileup **out);
/* The same without waiting for the copies: they run on the context's copy stream, so that the upload
 * of the next batch of chromosomes overlaps the kernels of the current one (the host arrays must stay
 * valid, and should be pinned, until the pileup is first used or sgpu_synchronize returns). Every
 * function that takes the pileup waits for its copies on the device. */
int sgpu_pileup_upload_async(sgpu_ctx *ctx, uint32_t n_chr, const uint64_t *chr_ptr, const uint64_t *row_ptr,
                             const uint32_t *position, const uint32_t *read_id, const uint16_t *gid_base,
                             sgpu_pileup **out);
/* The same, but the read ids (4 of the 6 bytes per entry) are NOT copied: they stay in the caller's page-locked,
 * mapped host memory (cudaHostAlloc / cudaHostRegister; must stay valid while the pileup lives). sgpu_filter then
 * pulls the read ids of the loci it KEEPS straight over PCIe while compacting, so the read ids of rejected loci never
 * travel (Filter::filter only looks at the bases, util/is_significant.cpp:163-175). Any other consumer of the read
 * ids (sgpu_counts_accumulate or sgpu_pileup_download on the unfiltered pileup) copies them all first. */
int sgpu_pileup_upload_lazy_async(sgpu_ctx *ctx, uint32_t n_chr, const uint64_t *chr_ptr, const uint64_t *row_ptr,
                                  const uint32_t *position, const uint32_t *read_id, const uint16_t *gid_base,
                                  sgpu_pileup **out);
/* Direct ingestion of SECEDO's binary pileup files (replaces read_pileup_bin, util/pileup_reader.cpp:139-257,
 * and the flattening of its vector<PosData>): one buffer per chromosome holding the bytes of the `.bin` file
 *     u32 position | u16 coverage | u32 read_id[coverage] | u16 (cell_id << 2 | base)[coverage]   per locus.
 * The host only walks the records; the bytes are copied to the device as they are and unpacked there with
 * id_to_group applied (get_grouping, :273). Loci with coverage > max_coverage are skipped (:195-197); if
 * positions is not NULL, positions[c] (ascending, n_positions[c] values, may be empty = no filter) selects the
 * loci of chromosome c (:199-210). A cell id >= n_ids is an error (the reference exits). n_cells / n_groups
 * receive max cell id + 1 / max group id + 1 (:232-233); max_fragment_length is 1000 as for the reference
 * without --compute_read_stats (:256). */
int sgpu_pileup_from_bin(sgpu_ctx *ctx, uint32_t n_chr, const void *const *file_bytes, const uint64_t *file_sizes,
                         const uint16_t *id_to_group, uint32_t n_ids, uint32_t max_coverage,
                         const uint32_t *const *positions, const uint64_t *n_positions, sgpu_pileup **out,
                         uint32_t *n_cells, uint32_t *n_groups);
/* Wide pileups: group ids beyond the reference's 14 bits (sequenced_data.hpp:29-36 packs the id into 14 bits of a
 * uint16; 20 000 cells, BASELINE config 5, do not fit). gid_base32[e] = group id << 2 | base with 30-bit ids; in
 * id_to_pos / group_id_to_pos "not in the cluster" is 0xFFFFFFFF instead of SGPU_NO_POS. sgpu_filter,
 * sgpu_counts_accumulate(_range), sgpu_chromosome_cutoff, sgpu_similarity and the epilogues accept them (the kernels
 * that read the entries are templates over the entry width); the .bin ingestion, lazy uploads and
 * sgpu_expectation_maximization stay 14-bit like the reference's file format and return SGPU_E_ARG. The GEMM path
 * takes up to 26 360 cells (the scatter path has no such limit). sgpu_synth_pileup produces a wide pileup when
 * n_cells > 16 383. */
#define SGPU_NO_POS_WIDE 0xFFFFFFFFu
int sgpu_pileup_upload_wide(sgpu_ctx *ctx, uint32_t n_chr, const uint64_t *chr_ptr, const uint64_t *row_ptr,
                            const uint32_t *position, const uint32_t *read_id, const uint32_t *gid_base32,
                            sgpu_pileup **out);
int sgpu_pileup_upload_wide_async(sgpu_ctx *ctx, uint32_t n_chr, const uint64_t *chr_ptr, const uint64_t *row_ptr,
                                  const uint32_t *position, const uint32_t *read_id, const uint32_t *gid_base32,
                                  sgpu_pileup **out); /* like sgpu_pileup_upload_async */
int sgpu_pileup_download_wide(sgpu_ctx *ctx, const sgpu_pileup *p, uint64_t *chr_ptr, uint64_t *row_ptr,
                              uint32_t *position, uint32_t *read_id, uint32_t *gid_base32);
int sgpu_pileup_is_wide(const sgpu_pileup *p);
/* Adopt arrays that already live on this context's device (not copied, not freed). */
int sgpu_pileup_wrap_device(sgpu_ctx *ctx, uint32_t n_chr, const uint64_t *host_chr_ptr,
                            const uint64_t *dev_row_ptr, const uint32_t *dev_position,
                            const uint32_t *dev_read_id, const uint16_t *dev_gid_base, sgpu_pileup **out);
int sgpu_pileup_dims(const sgpu_pileup *p, uint32_t *n_chr, uint64_t *n_loci, uint64_t *n_entries);
int sgpu_pileup_download(sgpu_ctx *ctx, const sgpu_pileup *p, uint64_t *chr_ptr, uint64_t *row_ptr,
                         uint32_t *position, uint32_t *read_id, uint16_t *gid_base);
void sgpu_pileup_free(sgpu_ctx *ctx, sgpu_pileup *p);
/* Deterministic synthetic pileup generated directly in HBM (counter-based: every entry is a pure
 * function of seed, locus and slot, so any sub-range can be downloaded and replayed on the CPU). */
int sgpu_synth_pileup(sgpu_ctx *ctx, const sgpu_synth_params *params, sgpu_pileup **out);

/* ---- Filter (util/is_significant.cpp) -------------------------------------------------------- */
/* Filter::is_significant(std::array<uint16_t,4>&) on n count tuples, evaluated on the GPU. */
int sgpu_is_significant(sgpu_ctx *ctx, const uint16_t *counts4, uint64_t n, double theta,
                        int cell_proportion, uint8_t *out);
/* Filter::filter: keeps the entries whose group is in the sub-cluster (id_to_pos[gid] != NO_POS)
 * at the loci that pass is_significant; result stays on the device. avg_coverage is accumulated in
 * 64 bits (the reference wraps at 2^32, util/is_significant.cpp:156,187).
 * When every group is in the sub-cluster (the root of the recursion) the read ids are not copied: the result reads them
 * through a view of `in` until it is downloaded or freed. sgpu_pileup_free(in) before that is fine (the library keeps the
 * ids alive); device arrays that the CALLER owns (sgpu_pileup_wrap_device) must outlive the result. */
int sgpu_filter(sgpu_ctx *ctx, const sgpu_pileup *in, const uint32_t *id_to_pos, uint32_t n_groups,
                double theta, int cell_proportion, sgpu_pileup **filtered, double *avg_coverage);

/* ---- similarity matrix (similarity_matrix.cpp) ------------------------------------------------ */
/* One call = computeSimilarityMatrix on one GPU; out is caller-owned host memory, num_cells^2
 * doubles, row-major. num_threads only selects the reference's tail cutoff K (SURVEY F2). */
int sgpu_similarity(sgpu_ctx *ctx, const sgpu_pileup *filtered, uint32_t num_cells,
                    uint32_t max_fragment_length, const uint32_t *group_id_to_pos, uint32_t n_groups,
                    double mutation_rate, double homozygous_rate, double seq_error_rate,
                    uint32_t num_threads, int normalization, int path, double *out, sgpu_stats *stats);

/* The same in three steps, so that several GPUs / several batches of chromosomes can share one
 * result: create -> accumulate (any number of times) -> [sum the buffers over ranks] -> finalize. */
int sgpu_counts_create(sgpu_ctx *ctx, uint32_t num_cells, sgpu_counts **out);
int sgpu_counts_zero(sgpu_ctx *ctx, sgpu_counts *c);
void sgpu_counts_free(sgpu_ctx *ctx, sgpu_counts *c);
/* A failed accumulation (also _range) either leaves the counts object exactly as it was (an error found before any
 * count was issued, such as SGPU_E_COUNT_RANGE of the GEMM path's first panel), or leaves a partial sum in it (e.g.
 * SGPU_E_CLASS_RANGE): then every accumulation fails with SGPU_E_ARG until sgpu_counts_zero. */
int sgpu_counts_accumulate(sgpu_ctx *ctx, sgpu_counts *c, const sgpu_pileup *filtered,
                           uint32_t max_fragment_length, const uint32_t *group_id_to_pos,
                           uint32_t n_groups, double mutation_rate, double homozygous_rate,
                           double seq_error_rate, uint32_t num_threads, int path, sgpu_stats *stats);
/* ---- pieces of chromosomes: locus ranges with a halo (SURVEY 8(e)) -----------------------------------------------
 * A chromosome may be accumulated in pieces — by different GPUs, or one after the other on the same GPU. A piece is a
 * filtered pileup that holds, for each of its chromosomes, the loci it OWNS (positions in [own_pos_begin[c],
 * own_pos_end[c])) and a read-only halo: every filtered locus of that chromosome less than max_fragment_length bp
 * before the first owned position and less than max_fragment_length bp after the last one (more does no harm). The
 * owned ranges of the pieces must tile the chromosome. Each piece then adds exactly its share: first-order counts of
 * its owned loci, and the read pairs that overlap at >= 2 loci whose FIRST common locus it owns; the halo only serves
 * to see the reads of the owned loci completely (cell of the first entry, mate rule, all loci). The sums over the
 * pieces equal the counts of the whole chromosome bit for bit.
 * The reference's tail cutoff K (SURVEY F2) is a property of the whole chromosome; it is decided from the chromosome's
 * END by sgpu_chromosome_cutoff and handed to every piece as tail_position[c]: reads created at positions >=
 * tail_position[c] are never the first read of a pair (0xFFFFFFFF: none).
 *
 * sgpu_chromosome_cutoff: `ends` holds, per chromosome, either the whole filtered chromosome (whole[c] != 0) or its
 * last loci (a suffix). resolved[c] = 1: tail_position[c] is the cutoff of the whole chromosome; 0: the suffix was
 * too short to decide (no batch trigger that fires whatever happened before it lies inside its exact part, i.e. more
 * than max_fragment_length bp behind its first locus): call again with a longer suffix. On dense pileups (>= 4 *
 * num_threads new reads per locus) a suffix of a few max_fragment_length always suffices. */
#define SGPU_TAIL_NONE 0xFFFFFFFFu /* tail_position: no read of this chromosome is a tail read for this piece */
#define SGPU_TAIL_AUTO 0xFFFFFFFEu /* tail_position: the piece holds the END of the chromosome: decide the cutoff from the piece
                                      itself with num_threads (SGPU_E_ARG if the piece is too short for that) */
int sgpu_chromosome_cutoff(sgpu_ctx *ctx, const sgpu_pileup *ends, uint32_t max_fragment_length, uint32_t num_threads,
                           const uint8_t *whole, uint32_t *tail_position, uint8_t *resolved);
int sgpu_counts_accumulate_range(sgpu_ctx *ctx, sgpu_counts *c, const sgpu_pileup *piece, uint32_t max_fragment_length,
                                 const uint32_t *group_id_to_pos, uint32_t n_groups, double mutation_rate,
                                 double homozygous_rate, double seq_error_rate, uint32_t num_threads /* only for SGPU_TAIL_AUTO */,
                                 const uint32_t *own_pos_begin, const uint32_t *own_pos_end, const uint32_t *tail_position,
                                 int path, sgpu_stats *stats);
/* Device buffers to be summed element-wise across ranks before finalize:
 *   i32     int32 [n_i32]  planes of num_cells^2: S, D (first order), then, when read pairs that
 *                          overlap at >= 2 loci occurred, the class planes (2,0) (1,1) (0,2)
 *                          (3,0) (2,1) (1,2) (0,3); only the upper triangle i < j is meaningful
 *   f64     double [n_f64] num_cells^2, present only if a pair overlapped at >= 4 loci: sum of
 *                          G(x_s,x_d) = F(x_s,x_d) - x_s F(1,0) - x_d F(0,1) over those pairs
 *   hist    uint64 [SGPU_MAX_CLASS^2] global histogram of overlap classes with x_s + x_d >= 2
 * Ranks must agree on the layout before reducing: exchange (n_i32, n_f64), take the maximum and
 * call sgpu_counts_set_layout (buffers may move), then fetch the pointers again. */
int sgpu_counts_buffers(sgpu_counts *c, int32_t **i32, uint64_t *n_i32, double **f64, uint64_t *n_f64,
                        uint64_t **hist, uint64_t *n_hist);
int sgpu_counts_set_layout(sgpu_ctx *ctx, sgpu_counts *c, int planes_used /* 2, 5 or 9 */, int want_spill);
/* Half the bytes for the cross-rank reduction: the upper triangles (i < j) of the int32 planes in use,
 * packed row by row into one contiguous device buffer owned by the counts object
 * (n = planes * num_cells (num_cells - 1) / 2). Agree on the layout first; reduce the packed buffer;
 * sgpu_counts_unpack on the destination rank writes the sums back into the planes. */
int sgpu_counts_pack(sgpu_ctx *ctx, sgpu_counts *c, int32_t **packed, uint64_t *n);
int sgpu_counts_unpack(sgpu_ctx *ctx, sgpu_counts *c);
/* The same for planes [first_plane, first_plane + n_planes) only. */
int sgpu_counts_pack_range(sgpu_ctx *ctx, sgpu_counts *c, int first_plane, int n_planes, int32_t **packed, uint64_t *n);
int sgpu_counts_unpack_range(sgpu_ctx *ctx, sgpu_counts *c, int first_plane, int n_planes);
/* The planes beyond S and D count read pairs that overlap at >= 2 loci and are almost empty on real pileups: their
 * non-zeros (upper triangle) as a list of (idx, val), idx = position relative to plane `first_plane`
 * (plane * num_cells^2 + i * num_cells + j, 32 bits), in device buffers owned by the counts object. The order of the
 * list is row by row (plane, i, j ascending). sgpu_counts_sparse_add adds such a list (e.g. another rank's) into the planes; indices of one
 * list must be distinct. With these the cross-rank reduction sends S and D densely and the rest as lists. */
int sgpu_counts_sparse_pack(sgpu_ctx *ctx, sgpu_counts *c, int first_plane, uint32_t **idx, int32_t **val, uint64_t *nnz);
int sgpu_counts_sparse_add(sgpu_ctx *ctx, sgpu_counts *c, int first_plane, const uint32_t *idx, const int32_t *val,
                           uint64_t nnz);
/* Symmetric per-cell-pair integers for bit-exact checks (any pointer may be NULL):
 *   S1, D1  num_cells^2 int32: incidences (read pair, shared locus) with equal / different base
 *   H       3*num_cells^2 int32: read pairs in overlap class (2,0), (1,1), (0,2)
 *   hist    SGPU_MAX_CLASS^2 uint64: read pairs per class (x_s, x_d) with x_s + x_d >= 2 */
int sgpu_counts_download(sgpu_ctx *ctx, sgpu_counts *c, int32_t *S1, int32_t *D1, int32_t *H, uint64_t *hist);
/* Log-likelihood transform (LS/LD of similarity_matrix.cpp:117-170) + normalisation (:271-293). */
int sgpu_similarity_finalize(sgpu_ctx *ctx, sgpu_counts *c, uint32_t max_fragment_length,
                             double mutation_rate, double homozygous_rate, double seq_error_rate,
                             int normalization, double *out, sgpu_stats *stats);
/* The same without waiting for the download: the matrix is copied to `out` (page-locked host memory) on a stream of
 * its own, so that the kernels of the next batch start at once; sgpu_output_wait returns when `out` is complete. At
 * most one download is in flight per context (a second call first waits for the first). */
int sgpu_similarity_finalize_async(sgpu_ctx *ctx, sgpu_counts *c, uint32_t max_fragment_length,
                                   double mutation_rate, double homozygous_rate, double seq_error_rate,
                                   int normalization, double *out);
int sgpu_output_wait(sgpu_ctx *ctx);
/* ---- multi-GPU epilogue over peer memory: reduce-scatter + transform in one kernel --------------------------------
 * The count planes of the GPUs are NOT summed into one of them. The 32 x 32 tiles of the upper triangle are dealt out
 * in n_slabs equal contiguous shares; the GPU that owns share `slab` reads, for its tiles, the planes of ALL GPUs
 * (peer_planes[0 .. n_peers): device pointers valid on this GPU — its own planes, peers of the same process after
 * cudaDeviceEnablePeerAccess, or other processes' planes mapped with sgpu_ipc_open), adds the integers and applies
 * the log-likelihood transform in the same kernel (sgpu_slab_raw). The order of the peers does not matter (integer
 * sums) and the floating-point expression is the single-GPU epilogue's, so the values are bit-identical to a
 * reduction onto one GPU followed by sgpu_similarity_finalize. extrema receives a device pointer to two doubles
 * {-min, max} of this share's raw values: the caller takes the element-wise MAX over the GPUs in place (one tiny
 * all-reduce, which is also the barrier after which no GPU reads another's planes any more), then sgpu_slab_finalize
 * normalises this share and writes its tiles and their mirror images into `out`: an n x n row-major matrix in device
 * memory or in mapped page-locked host memory (sgpu_host_register; every GPU then writes its share of the matrix over
 * its own PCIe link), or, with out = NULL, into an n x n device matrix owned by the counts object of which only this
 * share is written (returned in *device_out). All ranks must have agreed on the layout (sgpu_counts_set_layout) and
 * finished accumulating before any of them calls sgpu_slab_raw. peer_spill: the fp64 spill planes of the GPUs (read
 * pairs that overlap at >= 4 loci; sgpu_counts_set_layout with want_spill on every rank once one of them has one), or
 * NULL when no GPU holds one; they are added in the order of the array (fp64: agrees with one GPU to rounding). Entries
 * of GPUs without a spill plane may be NULL. Like sgpu_similarity_finalize, it fails with SGPU_E_ARG when c holds a
 * spill plane and the likelihood parameters differ from those c was accumulated with. */
int sgpu_slab_raw(sgpu_ctx *ctx, sgpu_counts *c, const int32_t *const *peer_planes, const double *const *peer_spill,
                  uint32_t n_peers, uint32_t slab, uint32_t n_slabs, uint32_t max_fragment_length, double mutation_rate,
                  double homozygous_rate, double seq_error_rate, double **extrema);
int sgpu_slab_finalize(sgpu_ctx *ctx, sgpu_counts *c, int normalization, double *out, double **device_out);
/* first and one-past-last tile of the share of the last sgpu_slab_raw call (tiles numbered row by row over bj >= bi) */
int sgpu_slab_range(const sgpu_counts *c, uint64_t *tile0, uint64_t *tile1);
/* CUDA IPC: handle (SGPU_IPC_HANDLE_BYTES bytes) of this counts object's int32 planes for another PROCESS on the same
 * node; sgpu_ipc_open maps such a handle (the returned pointer is valid on ctx's device, peer access over NVLink is
 * enabled by the driver), sgpu_ipc_close unmaps it. */
int sgpu_counts_ipc_handle(sgpu_ctx *ctx, sgpu_counts *c, int which /* 0: int32 planes, 1: fp64 spill plane */, void *handle);
int sgpu_ipc_open(sgpu_ctx *ctx, const void *handle, void **device_ptr);
int sgpu_ipc_close(sgpu_ctx *ctx, void *device_ptr);
/* Page-lock and map existing host memory (e.g. a shared-memory segment that several processes write their shares of
 * the matrix into); *device_alias is the pointer kernels of ctx's device use. */
int sgpu_host_register(sgpu_ctx *ctx, void *host, uint64_t bytes, void **device_alias);
int sgpu_host_unregister(sgpu_ctx *ctx, void *host);
/* order-independent 64-bit checksum of the upper triangles (i < j) of the int32 planes in use: sum over elements of
 * value * weight(position), wrapping; linear, so the checksums of the ranks add up to the checksum of the summed planes.
 * n_peers > 1: checksum of the element-wise sum of the peers' planes restricted to tiles [tile0, tile1) of share
 * `slab`; the shares of all GPUs add up to the checksum of the whole sum. */
int sgpu_counts_checksum(sgpu_ctx *ctx, sgpu_counts *c, const int32_t *const *peer_planes, uint32_t n_peers, uint32_t slab,
                         uint32_t n_slabs, uint64_t *checksum);

/* ---- several GPUs behind one call (single process; SURVEY 8(b): sgpu_init(devices, n_dev)) --------------------------
 * For host programs that are not a multi-process job — SECEDO's divide_cluster through the C++ shim. devices = NULL
 * takes every visible GPU. sgpu_multi_similarity is computeSimilarityMatrix (similarity_matrix.cpp:295-433) on a
 * FILTERED host pileup (the five CSR arrays of the header comment): the loci are cut into one piece per GPU inside the
 * chromosomes (halos of max_fragment_length bp, SURVEY 8(e)), every GPU uploads and accumulates its piece on a host
 * thread of its own, then the epilogue over peer memory (sgpu_slab_raw / sgpu_slab_finalize with peer access enabled
 * between the GPUs) writes each GPU's share of the matrix; out = num_cells^2 doubles, row-major, caller-owned host
 * memory. Same result as sgpu_similarity on one GPU: integer counts bit for bit, the matrix bit for bit unless read
 * pairs overlap at >= 4 loci (fp64 spill planes are added in GPU order: agrees to rounding). */
typedef struct sgpu_multi sgpu_multi;
int sgpu_multi_init(const int *devices, int n_devices, sgpu_multi **out);
void sgpu_multi_shutdown(sgpu_multi *m);
const char *sgpu_multi_last_error(const sgpu_multi *m);
int sgpu_multi_size(const sgpu_multi *m);
sgpu_ctx *sgpu_multi_ctx(sgpu_multi *m, int i); /* the context of the i-th GPU (e.g. for sgpu_filter on GPU 0) */
int sgpu_multi_similarity(sgpu_multi *m, uint32_t n_chr, const uint64_t *chr_ptr, const uint64_t *row_ptr,
                          const uint32_t *position, const uint32_t *read_id, const uint16_t *gid_base, uint32_t num_cells,
                          uint32_t max_fragment_length, const uint32_t *group_id_to_pos, uint32_t n_groups,
                          double mutation_rate, double homozygous_rate, double seq_error_rate, uint32_t num_threads,
                          int normalization, int path, double *out, sgpu_stats *stats);

/* LS / LD tables as evaluated on the device, n*n row-major (parity with similarity_matrix.cpp:117-170). */
int sgpu_log_probs(sgpu_ctx *ctx, double mutation_rate, double homozygous_rate, double seq_error_rate,
                   uint32_t max_fragment_length, uint32_t n, double *ls, double *ld);

/* ---- expectation maximisation (expectation_maximization.cpp) --------------------------------------- */
/* expectation_maximization() (expectation_maximization.hpp:27-31, body expectation_maximization.cpp:131-160) on a
 * filtered pileup that already lives on the device: prob_cluster_b (n_cells doubles on the host) holds the probability
 * of every cell to belong to the second cluster and is refined in place until no entry moves by 1e-2 or more
 * (max_iterations = 0) or for at most max_iterations rounds. As in the reference the probability of an entry's cell is
 * looked up with the group id itself and the log likelihood is accumulated at id_to_pos[group id]
 * (expectation_maximization.cpp:24 vs :88-89) and the log likelihoods keep accumulating over the iterations
 * (:136-137). A group id or id_to_pos[group id] >= n_cells (out-of-range read / std::out_of_range in the reference)
 * is SGPU_E_CELL_RANGE. The sums over a cell's entries are formed in 2^-32 fixed point (order independent:
 * results are bit-reproducible); against the reference's sequential fp64 sums the probabilities agree to 1e-6. */
int sgpu_expectation_maximization(sgpu_ctx *ctx, const sgpu_pileup *filtered, const uint32_t *id_to_pos, uint32_t n_groups,
                                  double theta, double *prob_cluster_b, uint32_t n_cells, uint32_t max_iterations,
                                  uint32_t *iterations, float *ms);

/* ---- Laplacian and its leading eigenpairs (spectral_clustering.cpp) ------------------------------- */
typedef struct sgpu_spectral_stats {
    uint32_t outer_iterations; /* Rayleigh-Ritz steps */
    uint32_t block;            /* vectors iterated together */
    uint64_t matvec_columns;   /* columns multiplied by the N x N matrix in total */
    uint64_t matvec_launches;  /* launches of the block product kernel */
    uint64_t launches;         /* all kernels of the call */
    double max_residual;       /* largest |M x - theta x| of the returned pairs */
    double lower_bound;        /* Lanczos bound of the spectrum that the filter damps */
    float ms_laplacian;        /* degrees + scaling */
    float ms_solver;           /* subspace iteration */
    float ms_matvec;           /* the block product kernel alone (sum over launches) */
    uint32_t reserved;
} sgpu_spectral_stats;
/* laplacian() (spectral_clustering.cpp:33-52): out = I - D^-1/2 A D^-1/2, n x n row-major host matrices. */
int sgpu_laplacian(sgpu_ctx *ctx, const double *similarity, uint32_t n, double *out);
/* What spectral_clustering() takes from arma::eig_sym(laplacian(similarity)) (spectral_clustering.cpp:127-138,
 * :166-171, :218, :236): the k smallest eigenvalues (ascending) and their eigenvectors, eigenvectors[i * n + r] =
 * component r of eigenvector i (Armadillo's column-major layout), unit norm, the component of largest magnitude
 * positive (LAPACK's sign is arbitrary). Residuals |L v - lambda v| <= tol (0 selects 1e-10). 1 <= k <= 32,
 * n >= 2 * block (block = 16 for k <= 8, 32 for k <= 16, else 64); similarities must be non-negative. All n
 * eigenvalues (the reference's sim_mat_eigenvalues CSV) come from sgpu_laplacian_eigenvalues. */
int sgpu_spectral_embedding(sgpu_ctx *ctx, const double *similarity, uint32_t n, uint32_t k, double tol,
                            double *eigenvalues, double *eigenvectors, sgpu_spectral_stats *stats);
/* sgpu_similarity_finalize followed by sgpu_spectral_embedding without the matrix leaving the device
 * (out may be NULL: the n x n matrix is then not downloaded at all). */
int sgpu_similarity_finalize_spectral(sgpu_ctx *ctx, sgpu_counts *c, uint32_t max_fragment_length,
                                      double mutation_rate, double homozygous_rate, double seq_error_rate,
                                      int normalization, double *out, uint32_t k, double tol, double *eigenvalues,
                                      double *eigenvectors, sgpu_stats *stats, sgpu_spectral_stats *spectral_stats);
/* ---- every eigenvalue of the Laplacian (the sim_mat_eigenvalues CSV of spectral_clustering.cpp:141-143) ---------- */
typedef struct sgpu_eigenvalue_stats {
    uint64_t launches;     /* all kernels of the call */
    float ms_laplacian;    /* degrees + scaling */
    float ms_tridiagonal;  /* blocked Householder reduction to tridiagonal form */
    float ms_bisection;    /* Sturm bisection of the tridiagonal matrix */
    uint64_t bytes_matvec; /* bytes the symmetric matrix-vector products must read: one triangle of the trailing
                              matrix per column, 8 (n-1) n (n+1) / 6 */
    uint32_t reserved;
} sgpu_eigenvalue_stats;
/* All n eigenvalues of laplacian(similarity) = I - D^-1/2 A D^-1/2, ascending, as arma::eig_sym returns them
 * (spectral_clustering.cpp:127-138), computed on the device in fp64: B = D^-1/2 A D^-1/2 is reduced to tridiagonal
 * form by blocked Householder reflections (LAPACK DSYTRD) and the eigenvalues of B are found by bisection on Sturm
 * counts (DSTEBZ); eigenvalues[i] = 1 - (the i-th largest of B). similarity: host n x n, symmetric, non-negative
 * (a negative or NaN degree is SGPU_E_ARG); a cell of degree 0 has eigenvalue 1, an all-zero matrix n ones. The
 * device holds 8 ld^2 bytes of working copy (ld = n rounded up to 64). Bit-reproducible. */
int sgpu_laplacian_eigenvalues(sgpu_ctx *ctx, const double *similarity, uint32_t n, double *eigenvalues,
                               sgpu_eigenvalue_stats *stats);
/* sgpu_similarity_finalize followed by sgpu_laplacian_eigenvalues without the matrix leaving the device (out may be
 * NULL: the n x n matrix is then not downloaded). Refuses, like sgpu_similarity_finalize, likelihood parameters other
 * than the accumulation's when c holds a spill plane. */
int sgpu_similarity_finalize_eigenvalues(sgpu_ctx *ctx, sgpu_counts *c, uint32_t max_fragment_length,
                                         double mutation_rate, double homozygous_rate, double seq_error_rate,
                                         int normalization, double *out, double *eigenvalues, sgpu_stats *stats,
                                         sgpu_eigenvalue_stats *eig_stats);
/* test hook of the block product kernel: out = alpha M X + beta X + gamma W, M n x n symmetric, blocks n x width
 * row-major (width 8, 16, 32 or 64), all on the host */
int sgpu_spectral_matvec(sgpu_ctx *ctx, const double *M, uint32_t n, int width, const double *X, const double *W,
                         double alpha, double beta, double gamma, double *out);

#ifdef __cplusplus
}
#endif
#endif
