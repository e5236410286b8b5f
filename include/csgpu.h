/* csgpu.h -- C ABI of libcsgpu.so, the B200 (sm_100a) implementation of the
 * Configurable-Spectrograms data-parallel batch path.
 *
 * The reference (ev-hansen/Configurable-Spectrograms) has no FFI of its own; its
 * operator surface on this path is a set of numpy / matplotlib call sites inside
 * Python functions (SURVEY.md section 8a/8b).  Every entry point below names the
 * reference call site(s) it replaces ("CS/" = src/configurable_spectrograms/).
 * INTEGRATION.md shows the ctypes stubs a maintainer would add.
 *
 * Conventions
 *   - plain C, no C++/torch types; every function returns a csg_status (0 = OK)
 *     except constructors/accessors; csg_last_error() returns the message.
 *   - all pointers named d_* are DEVICE pointers, h_* are HOST pointers.
 *   - one csg_ctx per GPU, not thread-safe; all work is enqueued on the context's
 *     stream (own stream, or an external cudaStream_t handed to csg_create()).
 *   - dtype: CSG_F32 / CSG_F64 is the dtype D of the counts cube; sums,
 *     percentiles and normalisation are computed in D exactly like numpy /
 *     matplotlib do (SURVEY.md Appendix B).
 *   - there is NO CPU fallback: without a CUDA device every compute call fails.
 */
#ifndef CSGPU_H
#define CSGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CSG_ABI_VERSION 26

#if defined(__GNUC__)
#define CSG_API __attribute__((visibility("default")))
#else
#define CSG_API
#endif

typedef enum {
  CSG_OK = 0,
  CSG_ERR_CUDA = 1,   /* a CUDA runtime call failed (message has the CUDA error) */
  CSG_ERR_ARG = 2,    /* invalid argument */
  CSG_ERR_NOMEM = 3,  /* allocation failed */
  CSG_ERR_NODEV = 4,  /* no usable CUDA device */
  CSG_ERR_IO = 5      /* a file could not be written (csg_png_write_files: per-file errno in csg_png_file.status) */
} csg_status;

enum { CSG_F32 = 0, CSG_F64 = 1 };
/* memory order of a counts cube */
enum {
  CSG_LAYOUT_TPE = 0, /* C-contiguous (time, pitch, energy): np.nansum(axis=1) is an ascending-p chain  */
  CSG_LAYOUT_TEP = 1  /* stored (time, energy, pitch), collapsed through the transposed view of
                         CS/cdf_utils.py:254-255: numpy's 8-accumulator pairwise order                 */
};
#define CSG_MAX_GROUPS 7 /* pitch-angle groups per file besides the unmasked total */

typedef struct csg_ctx csg_ctx;

/* ------------------------------------------------------------------ context */
CSG_API int csg_abi_version(void);
CSG_API int csg_device_count(void);
/* external_stream: a cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream) or NULL for an own stream */
CSG_API csg_ctx* csg_create(int device, void* external_stream);
/* A second context on the same device with its own (optionally highest-priority) stream: work
 * that is independent of the main stream's next kernels (the K2b digit loop and its exchanges
 * next to K2a / K3) overlaps them.  csg_wait_for: everything enqueued on `signal` so far
 * happens before whatever is enqueued on `waiter` from now on. */
CSG_API csg_ctx* csg_create_side(int device, int high_priority);
/* a context with its own stream at priority `level` steps above the device's least urgent level (0 = what
 * csg_create gives; clamped to the most urgent).  The directory driver runs its planner's kernels (K2a / K3,
 * short) one step above the K4 encoder's (long), and the extrema chain on the most urgent stream. */
CSG_API csg_ctx* csg_create_with_priority(int device, int level);
CSG_API int csg_wait_for(csg_ctx* waiter, csg_ctx* signal);
CSG_API void csg_destroy(csg_ctx* ctx);
CSG_API const char* csg_last_error(csg_ctx* ctx); /* ctx may be NULL: error of a failed csg_create() */
CSG_API int csg_sync(csg_ctx* ctx);
/* the cudaStream_t every call of this context is enqueued on (for ordering external work, e.g. NCCL) */
CSG_API void* csg_stream_handle(csg_ctx* ctx);
/* "NVIDIA B200", SM count, total memory bytes */
CSG_API int csg_device_info(csg_ctx* ctx, char* name, int name_len, int* sm_count, size_t* total_mem);

/* ------------------------------------------------------------------- memory */
/* Device blocks come from a per-device cache: csg_dev_free parks the block (fenced with an event on every
   stream of every live context, so nobody gets it back before all work enqueued so far is over) and
   csg_dev_alloc reuses a parked block of the same size class (4 classes per power of two) whose fences have
   passed -- a block still fenced is skipped, never waited for -- a directory run
   allocates per-chunk tables at a rate at which cudaMalloc / cudaFree (device-wide synchronisation, ms each)
   showed up as half the wall time.  CSG_POOL=0 restores plain cudaMalloc / cudaFree; CSG_POOL_MAX_MB caps the
   parked bytes (default 32768).  An allocation the driver refuses is retried after the cache is emptied. */
CSG_API int csg_dev_alloc(csg_ctx* ctx, size_t bytes, void** d_ptr);
CSG_API int csg_dev_free(csg_ctx* ctx, void* d_ptr);
/* return every parked block of the context's device to the driver; released_bytes may be NULL */
CSG_API int csg_dev_trim(csg_ctx* ctx, size_t* released_bytes);
/* bytes parked in the cache / bytes handed out and not yet freed (either pointer may be NULL) */
CSG_API int csg_dev_cached(csg_ctx* ctx, size_t* idle_bytes, size_t* live_bytes);
CSG_API int csg_host_alloc(csg_ctx* ctx, size_t bytes, void** h_ptr); /* pinned */
CSG_API int csg_host_free(csg_ctx* ctx, void* h_ptr);
CSG_API int csg_host_register(csg_ctx* ctx, void* h_ptr, size_t bytes); /* pin caller memory (cdflib arrays) */
CSG_API int csg_host_unregister(csg_ctx* ctx, void* h_ptr);
CSG_API int csg_h2d(csg_ctx* ctx, void* d_dst, const void* h_src, size_t bytes); /* async on the ctx stream */
CSG_API int csg_d2h(csg_ctx* ctx, void* h_dst, const void* d_src, size_t bytes); /* async on the ctx stream */
CSG_API int csg_d2d(csg_ctx* ctx, void* d_dst, const void* d_src, size_t bytes); /* async on the ctx stream */
CSG_API int csg_memset(csg_ctx* ctx, void* d_dst, int byte_value, size_t bytes);
/* Result read-back on the context's copy-out stream: ordered after everything enqueued on the
 * ctx stream so far, but later ctx-stream work (the next shard's uploads and kernels) does not
 * wait for it -- PCIe is full duplex.  csg_side_join makes the ctx stream wait for the copies
 * (call it before the source buffer is overwritten); csg_side_sync makes the host wait. */
CSG_API int csg_d2h_side(csg_ctx* ctx, void* h_dst, const void* d_src, size_t bytes);
CSG_API int csg_side_join(csg_ctx* ctx);
CSG_API int csg_side_sync(csg_ctx* ctx);

/* ------------------------------------------------------------------- timing */
/* CUDA-event stopwatch slots (0..31) on the ctx stream. */
CSG_API int csg_timer_start(csg_ctx* ctx, int slot);
CSG_API int csg_timer_stop(csg_ctx* ctx, int slot);
CSG_API int csg_timer_ms(csg_ctx* ctx, int slot, float* ms); /* synchronises on the stop event */
/* number of kernels this context has launched since creation */
CSG_API int64_t csg_launch_count(csg_ctx* ctx);
/* Event slots (0..31): record on the ctx stream, wait on the host for that point only (later
 * work keeps running) -- used to read small results back while the next kernels execute. */
CSG_API int csg_event_record(csg_ctx* ctx, int slot);
CSG_API int csg_event_sync(csg_ctx* ctx, int slot);

/* ------------------------------------------------------------- K1: collapse */
/* One counts cube.  Replaces COLLAPSE_FUNCTION = np.nansum(cube, axis=1)
 * (CS/constants.py:12) at CS/plotting.py:188, CS/fast/plotting.py:128,278,
 * CS/fast/extrema.py:259, together with the pitch-angle gather
 * data[:, mask, :] (CS/fast/plotting.py:121-127) and the zoom test
 * np.any(~np.isnan(cube[window])) (CS/plotting.py:597-603). */
typedef struct {
  const void* d_cube; /* device cube, dtype D, layout as given to csg_collapse()         */
  int64_t sums_off;   /* element offset in d_sums of this file's [(G+1)][E][Tp] block (multiple of 4) */
  int64_t flags_off;  /* byte offset in d_row_flags of this file's [T] flag bytes       */
  int32_t T, P, E;
  int32_t bits_off;    /* byte offset in d_pa_bits of this file's [P] membership bytes   */
  int32_t first_block; /* exclusive prefix sum of csg_collapse_blocks() over the files   */
  int32_t reserved[3]; /* STREAM kernel: [0] index of the file's first triple in d_runs, [1] number of
                          runs, [2] alias mask (csg_pitch_runs); ignored by the other kernels      */
} csg_file_desc; /* 56 bytes */

/* Which kernel collapses a file: the stream kernel (16-row tiles, loop bodies specialised per
 * run of constant group membership, coalesced transposed output) needs a 16-byte aligned
 * C-contiguous (T,P,E) cube with E / (16 bytes / sizeof D) in {16,24,32,48,64}; everything else
 * takes the generic kernel.  A csg_collapse() call handles files of ONE kernel, and every file of
 * a STREAM table has the same E (= max_E). */
enum { CSG_K1_GENERIC = 0, CSG_K1_STREAM = 1 };
CSG_API int csg_collapse_kernel(int32_t T, int32_t P, int32_t E, int dtype, int layout, const void* d_cube);
/* The same choice when the number of pitch-angle groups is known: a stored (T,E,P) view with no
 * groups, 8 <= P <= 128 and P % 8 == 0 takes the row kernel (CSG_K1_STREAM for layout TEP). */
CSG_API int csg_collapse_kernel_for(int32_t T, int32_t P, int32_t E, int dtype, int layout, const void* d_cube,
                            int n_groups);
/* Host helper: runs of constant group membership along the pitch axis as {p0, p1, mask} int32
 * triples (at most P of them) for csg_file_desc.reserved[0..1]; *alias (-> reserved[2]) = groups
 * that contain every bin -- their bits are cleared from the masks, the kernel copies the total. */
CSG_API int csg_pitch_runs(const uint8_t* h_pa_bits, int P, int n_groups, int32_t* h_runs, int32_t* alias);
/* thread blocks csg_collapse() uses for one (T,P,E) file (for first_block) */
CSG_API int32_t csg_collapse_blocks(int32_t T, int32_t P, int32_t E, int dtype, int layout, int kernel);
/* elements of one file's sums block: (n_groups+1) * E * Tp, Tp = T rounded up to a multiple of 4 */
CSG_API int64_t csg_sums_elems(int32_t T, int32_t E, int n_groups);

/* sums are ENERGY-MAJOR -- the orientation of matrix_plot = collapsed.T (CS/plotting.py:236):
 * sums[file][g][e][t] at sums_off + (g*E + e)*Tp + t; g = 0 is the sum over every pitch bin,
 * g = 1+k the sum over bins p with (d_pa_bits[bits_off+p] >> k) & 1 (cells t >= T of a row
 * are padding and never read).  NaN counts as +0, fill values and +-inf are summed as-is,
 * result dtype = D, summation order bit-identical to numpy's (SURVEY.md Appendix B).
 * d_row_flags[flags_off+t] bit 0 / bit 1+k: some non-NaN cell exists in time row t among
 * all / group-k pitch bins (any energy); zero it before the call.
 * All files of one call share dtype, layout, kernel and n_groups. */
CSG_API int csg_collapse(csg_ctx* ctx, const csg_file_desc* d_files, int n_files, int total_blocks,
                 const uint8_t* d_pa_bits, const int32_t* d_runs, int n_groups, int max_P, int max_E,
                 int dtype, int layout, int kernel, void* d_sums, uint8_t* d_row_flags);

/* zoom_needed = np.any(~np.isnan(cube[window])) (CS/plotting.py:597-603) from the row flags:
 * d_out[w] = 1 iff some row of window w has bit `bit` set.  Rows are [t0, t0+nt) when
 * rows_off < 0, else d_index_pool[rows_off .. rows_off+nt). */
typedef struct {
  int64_t flags_off; /* byte offset of the file's flags in d_row_flags */
  int32_t t0, nt, rows_off, bit;
} csg_flag_window; /* 24 bytes */
CSG_API int csg_window_any(csg_ctx* ctx, const uint8_t* d_row_flags, const csg_flag_window* d_windows, int n_windows,
                   const int32_t* d_index_pool, uint8_t* d_out);

/* Host-buffer convenience for one cube: the drop-in for COLLAPSE_FUNCTION(array, axis=1).
 * h_pa_bits may be NULL when n_groups == 0.  h_sums receives [(G+1)][T][E] of dtype D,
 * h_row_flags (may be NULL) [T]. */
CSG_API int csg_collapse_host(csg_ctx* ctx, const void* h_cube, int32_t T, int32_t P, int32_t E, int dtype,
                      int layout, const uint8_t* h_pa_bits, int n_groups, void* h_sums,
                      uint8_t* h_row_flags);

/* ------------------------------------------- K2a: region stats + percentiles */
/* A region is the cell set of one energy-time matrix slice after the reference's
 * masks (CS/plotting.py:191-219, CS/fast/plotting.py:116-118,129-130,279-281):
 * output row j (energy, after the descending flip) = energy row d_index_pool[cols_off+j]
 * of the energy-major [E][ld] matrix, output column i = time step t0+i (rows_off < 0) or
 * d_index_pool[rows_off+i]. */
typedef struct {
  int64_t mat_off; /* element offset of the [E][ld] matrix in d_mats              */
  int32_t ld;      /* elements between consecutive energy rows (= Tp)             */
  int32_t t0, nt;
  int32_t rows_off; /* -1: contiguous rows [t0, t0+nt)                             */
  int32_t cols_off;
  int32_t ne;
  int32_t want_pct; /* 0: reductions only, 1: reductions + percentiles, 2: geometry only (no stats) */
  int32_t reserved;
  double p_lo, p_hi; /* percentiles (0..100), e.g. 1 and 99                         */
} csg_region;        /* 56 bytes */

/* np.nanpercentile(matrix, p) twice (CS/percentile_utils.py:87-88), plus the
 * reductions of CS/plotting.py:261-262 (safe_vmin) and :313-315 (nanmin/nanmax). */
typedef struct {
  double p_lo, p_hi;       /* linear-interpolation percentiles in D arithmetic; NaN if no valid cell */
  double min_pos;          /* min over finite cells > 0; +inf when none                               */
  double fin_min, fin_max; /* min / max over finite cells; +inf / -inf when none                      */
  int64_t n_valid;         /* non-NaN cells                                                           */
  int32_t n_nan, n_neginf, n_posinf, n_pos; /* n_pos = finite cells > 0                               */
} csg_region_stats;                         /* 64 bytes */

CSG_API int csg_region_stats_run(csg_ctx* ctx, const void* d_mats, int dtype, const csg_region* d_regions,
                         int n_regions, const int32_t* d_index_pool, csg_region_stats* d_out);
/* Diagnostics: regions of the last run whose percentile ranks escaped the sampled brackets and
 * were redone by the exact radix select (synchronises the stream). */
CSG_API int csg_region_stats_fallbacks(csg_ctx* ctx, int n_regions, int* count);
/* Test knob: on != 0 makes every later csg_region_stats_run() of this context resolve ALL percentile
 * regions with the exact multi-pass radix select (the path a rank escaping its sampled bracket takes),
 * so that path can be compared with np.nanpercentile on ordinary inputs.  Results are identical either
 * way; only the route differs. */
CSG_API int csg_region_stats_force_exact(csg_ctx* ctx, int on);

/* ------------------------------------------------------ K3: norm + colormap */
/* One imshow panel (CS/plotting.py:276-287 log, :308-324 linear). */
typedef struct {
  int32_t region;      /* cells to draw (geometry)                                         */
  int32_t pct_region;  /* stats entry whose p_lo/p_hi stand in for z bounds that are NaN   */
  int32_t log_scale;   /* 1: LogNorm branch, 0: linear branch                              */
  int32_t first_block; /* exclusive prefix sum of csg_raster_blocks(ne, nt)                */
  double z_min, z_max; /* explicit bounds (reference z_axis_min / z_axis_max); NaN = None  */
  int64_t out_off;     /* pixel offset of this panel in d_rgba / d_index (ne rows x nt)    */
  int32_t stat_region; /* stats entry giving safe_vmin / the linear fallback: a region with
                          the same cell SET as `region` (order-independent), or -1 = region */
  int32_t reserved;
  int32_t zmin_slot, zmax_slot; /* >= 0: take the bound from d_zvals[slot] instead of z_min / z_max
                                   (bounds that depend on this step's global extrema); -1: literal */
} csg_panel;           /* 56 bytes */

enum {
  CSG_NORM_OK = 0,
  CSG_NORM_VMIN_GT_VMAX = 1, /* matplotlib: ValueError("vmin must be less or equal to vmax") */
  CSG_NORM_INVALID = 2       /* matplotlib LogNorm: ValueError("Invalid vmin or vmax")       */
};
typedef struct {
  double vmin, vmax;       /* bounds handed to LogNorm(vmin,vmax) / imshow(vmin=,vmax=)            */
  double fill_lo, fill_hi; /* substitutes written into the matrix (already rounded to D)          */
  double t_vmin, t_range;  /* log: log10(vmin), log10(vmax)-log10(vmin); linear: vmin, vmax-vmin  */
  int32_t status;          /* CSG_NORM_*                                                          */
  int32_t degenerate;      /* 1: vmin == vmax -> every cell maps to index 0; 2: NaN bound, or log10(vmin) == log10(vmax) -> all "bad";
                               3: linear, vmax - vmin = inf -> index 0, "bad" where v - vmin is inf */
  float c0, c1;            /* rasteriser's first-guess coefficients (internal)                    */
} csg_panel_norm;          /* 64 bytes */

CSG_API int32_t csg_raster_blocks(int32_t ne, int32_t nt);

/* bytes of the per-panel threshold table csg_panel_prepare() fills (257 values of dtype D
 * per panel, padded): value -> index is a monotone step function, so the rasteriser only
 * counts thresholds <= value; the thresholds themselves come from the direct formula. */
CSG_API size_t csg_threshold_bytes(int n_panels, int dtype);

/* Resolve every panel's normalisation (and its index thresholds) on the device from the
 * region stats.  d_zvals (may be NULL when no panel uses a slot): double[], NaN = None. */
CSG_API int csg_panel_prepare(csg_ctx* ctx, const csg_panel* d_panels, int n_panels,
                      const csg_region* d_regions, const csg_region_stats* d_stats, int dtype,
                      const double* d_zvals, csg_panel_norm* d_norms, void* d_thresholds);

/* Launches blocks [block_offset, block_offset + total_blocks) of the panel table's block space
 * (a table can be rasterised in several launches, e.g. the panels whose bounds are known first).
 * d_block_panel (required): panel index of every thread block, i.e. panel p repeated
 * csg_raster_blocks(ne_p, nt_p) times.
 * Clamp -> normalise -> 256-entry LUT index -> RGBA8.  d_lut: 259 x 4 bytes (256 colours,
 * under, over, bad).  d_index (uint16, may be NULL) receives Colormap indices 0..255 and
 * 256/257/258 for under/over/bad; d_rgba (may be NULL) the colours.  Row 0 of a panel is
 * the lowest energy (imshow origin="lower"). */
CSG_API int csg_rasterise(csg_ctx* ctx, const void* d_mats, int dtype, const csg_region* d_regions,
                  const int32_t* d_index_pool, const csg_panel* d_panels,
                  const csg_panel_norm* d_norms, const void* d_thresholds, int n_panels,
                  int total_blocks, int block_offset, const int32_t* d_block_panel, const uint8_t* d_lut,
                  uint8_t* d_rgba, uint16_t* d_index);
/* K3 runs persistent blocks, as many as fit an SM (3 for float32: 1536 threads, 61 K registers, 199 KB shared).
 * A full house leaves no room for ANY other block, so kernels on a concurrent high-priority stream -- the
 * global-extrema digit loop and its peer exchanges (K2b) -- stall until K3 ends.  While such a chain is in
 * flight the batch step caps K3 at 2 blocks per SM (0 restores the default): K3 loses a little occupancy, the
 * chain keeps moving.  Applies to the following csg_rasterise calls of this context. */
CSG_API int csg_rasterise_blocks_per_sm(csg_ctx* ctx, int blocks_per_sm);

/* ---------------------------------------------- K2b: global extrema (pooled) */
/* The pooled finite-positive samples of CS/fast/extrema.py:259-267 are never
 * materialised: each file's collapsed total matrix is histogrammed by radix digit
 * of the float key, the histograms are prefix-scanned along the ascending-orbit
 * file sequence of each instrument, and order statistics of every prefix pool
 * (the reference recomputes nanpercentile(concat(blocks so far)) per step,
 * :280-285) are located digit by digit. */
typedef struct {
  int64_t mat_off; /* element offset of the file's total [E][Tp] matrix in d_mats (group 0)     */
  int32_t T;       /* time steps; row pitch Tp = T rounded up to a multiple of 4                 */
  int32_t E;
  int32_t inst; /* instrument slot 0..n_inst-1                                                 */
  int32_t pos;  /* position of this file in its instrument's ascending-orbit sequence          */
} csg_pool_item; /* 24 bytes */

/* Level-0 pass: d_hist[inst][pos][0][bin] (uint32, bins = 1<<bits, top `bits` bits of the
 * positive-float key), d_counts[item][E] (int32: finite-positive cells per energy column,
 * CS/fast/extrema.py:260-264), d_npos[item] (int32).  hist_stride_pos = slots*bins. */
CSG_API int csg_pool_hist_first(csg_ctx* ctx, const void* d_mats, int dtype, const csg_pool_item* d_items,
                        int n_items, int max_pos, int bits, int max_E, uint32_t* d_hist,
                        int32_t* d_counts, int32_t* d_npos, uint32_t* d_ehist);
/* d_ehist (may be NULL; zeroed by the caller) [inst][pos][max_E]: the same per-energy counts keyed
 * by (instrument, position) -- csg_pool_scan_cols() turns them into the per-energy totals of
 * every prefix pool, the input of csg_pool_energy_candidates(). */
/* Refinement pass: cells whose key >> prefix_shift equals d_slot_prefix[inst][s] are counted
 * in d_hist[inst][pos][s][(key >> shift) & (bins-1)].  d_slot_prefix is sorted ascending per
 * instrument, padded with UINT64_MAX, n_slots entries per instrument. */
CSG_API int csg_pool_hist_refine(csg_ctx* ctx, const void* d_mats, int dtype, const csg_pool_item* d_items,
                         int n_items, int max_pos, int n_slots, const uint64_t* d_slot_prefix,
                         int prefix_shift, int shift, int bits, uint32_t* d_hist);
/* In-place inclusive scan of d_hist along pos for every (inst, slot, bin); d_totals (may be
 * NULL) receives the last row [inst][slot][bin] (this rank's bucket totals, the payload of
 * the histogram-merge all-gather).  d_slot_table (may be NULL) [inst][n_slots]: slots holding
 * the UINT64_MAX padding are skipped (their totals are 0). */
CSG_API int csg_pool_scan(csg_ctx* ctx, uint32_t* d_hist, int n_inst, int max_pos, const int32_t* d_inst_len,
                  int n_slots, int bits, const uint64_t* d_slot_table, uint32_t* d_totals);
/* The same scan over an arbitrary number of columns per (inst, pos) row (the per-energy counts). */
CSG_API int csg_pool_scan_cols(csg_ctx* ctx, uint32_t* d_hist, int n_inst, int max_pos, const int32_t* d_inst_len,
                       int cols, uint32_t* d_totals);
/* One query = (inst, pos, slot, rank): find the bin of the scanned row where the cumulative
 * count first exceeds rank; writes bin and the residual rank inside that bin.  d_base (may be
 * NULL) [inst][slot][bin]: counts held by lower ranks, added to every row on the fly. */
typedef struct {
  int32_t inst, pos, slot, bin; /* bin: output */
  int64_t rank;                 /* in: rank within the slot's population; out: residual */
  int64_t row_total;            /* out: population of the slot row (level 0: pool size n_k) */
} csg_pool_query;               /* 32 bytes */
CSG_API int csg_pool_locate(csg_ctx* ctx, const uint32_t* d_hist, int max_pos, int n_slots, int bits,
                    const uint32_t* d_base, csg_pool_query* d_queries, int n_queries);

/* ------------------------------- K2b, device-resident selection (no host round trips) */
/* The digit loop above driven on the GPU: one dense table entry per (request, pos) follows the
 * two neighbour ranks of numpy's linear interpolation through the digits; prefixes that cannot
 * hold the running maximum (CS/fast/extrema.py:287-300) are dropped between digits and the
 * distinct surviving key prefixes form the slot table of the next csg_pool_hist_refine(). */
typedef struct {
  int32_t inst;
  int32_t mode; /* 0: max over every prefix pool of its percentile (the reference's max-merge);
                   1: percentile of the whole pool (compute_mins, CS/fast/extrema.py:302-309) */
  double p;     /* percentile 0..100 */
} csg_pool_request; /* 16 bytes */
typedef struct {
  int32_t inst, pos, req, active;
  int32_t slot[2];    /* slot of the lo / hi neighbour's prefix in the current refine table   */
  int64_t rank[2];    /* rank inside the current bucket                                       */
  uint64_t prefix[2]; /* key bits resolved so far                                             */
  double gamma;       /* numpy's interpolation weight, computed in D                          */
} csg_pool_sel;       /* 64 bytes */
/* d_flags: int32[4], zeroed by the caller; bit set on: [0] a rank fell outside its row,
 * [1] more than n_slots distinct prefixes survived (fall back to the host-driven loop),
 * [2] a target's prefix is missing from the slot table. */

/* n_after[inst][pos] = population of prefix pool pos (scanned level-0 row + lower ranks' d_base,
 * may be NULL); d_below[inst] = population held by lower ranks. */
CSG_API int csg_pool_row_totals(csg_ctx* ctx, const uint32_t* d_hist, int n_inst, int max_pos, int bits,
                        const uint32_t* d_base, int64_t* d_n_after, int64_t* d_below);
/* Fill d_sel[n_req][max_pos]: active entries + numpy's (n-1)*q rank arithmetic in D.
 * d_above[inst] (may be NULL): positives held by higher ranks. */
CSG_API int csg_pool_sel_init(csg_ctx* ctx, int dtype, const csg_pool_request* d_requests, int n_req,
                      const int32_t* d_inst_len, int max_pos, const int64_t* d_n_after,
                      const int64_t* d_below, const int64_t* d_above, csg_pool_sel* d_sel);
CSG_API int csg_pool_sel_locate(csg_ctx* ctx, const uint32_t* d_hist, int max_pos, int n_slots, int bits,
                        const uint32_t* d_base, csg_pool_sel* d_sel, int n_req, int32_t* d_flags);
/* d_best[n_req] (int64 key bits, -1 = none): this rank's best lower bound per running-max request;
 * all-reduce(max) it across ranks before csg_pool_sel_slots(). */
CSG_API int csg_pool_sel_bounds(csg_ctx* ctx, const csg_pool_sel* d_sel, const csg_pool_request* d_requests,
                        int n_req, int max_pos, int shift, int64_t* d_best);
/* Prune against d_best, then d_local_slots[inst][n_slots] = ascending distinct prefixes still
 * followed on this rank (padded with UINT64_MAX); all-gather it before csg_pool_sel_assign(). */
CSG_API int csg_pool_sel_slots(csg_ctx* ctx, csg_pool_sel* d_sel, const csg_pool_request* d_requests, int n_req,
                       int max_pos, int shift, const int64_t* d_best, int n_inst, int n_slots,
                       uint64_t* d_local_slots, int32_t* d_flags);
/* One exchange per digit carries both the bounds and the slot lists: every rank's payload is
 * [64 x int64 bounds (csg_pool_sel_bounds output, d_best) | n_inst x n_slots uint64 slot lists
 * (csg_pool_sel_slots output, pruned with the LOCAL bounds)], csg_pool_slot_payload_bytes() in
 * all.  d_gathered holds n_ranks payloads, rank_stride_bytes apart (n_ranks = 1: the local
 * payload itself).  The kernel takes the maximum bound over the ranks, drops the prefixes
 * below it, merges the lists into d_table[inst][n_slots] and gives every target its slot. */
CSG_API int csg_pool_sel_assign(csg_ctx* ctx, csg_pool_sel* d_sel, const csg_pool_request* d_requests, int n_req,
                        int max_pos, int shift, const void* d_gathered, size_t rank_stride_bytes, int n_ranks,
                        int n_inst, int n_slots, uint64_t* d_table, int32_t* d_flags);
CSG_API size_t csg_pool_slot_payload_bytes(int n_inst, int n_slots);
/* d_values[n_req] (double; -inf when no entry survived on this rank), d_has[n_req]. */
CSG_API int csg_pool_sel_finish(csg_ctx* ctx, int dtype, const csg_pool_sel* d_sel, int n_req, int max_pos,
                        double* d_values, int32_t* d_has);
/* From the all-gathered bucket totals (rank r's [inst][cols_per_inst] block starts at
 * d_gathered + r * rank_stride uint32 elements): d_base = sum over lower ranks; d_above[inst]
 * (may be NULL) = cells held by higher ranks. */
CSG_API int csg_pool_base(csg_ctx* ctx, const uint32_t* d_gathered, size_t rank_stride, int n_ranks, int rank,
                  int n_inst, size_t cols_per_inst, uint32_t* d_base, int64_t* d_above);

/* y extrema on the device: the 99 %-coverage energy (CS/fast/extrema.py:270-278) of every prefix
 * pool, max-merged per instrument.  d_ehist: scanned per-energy counts [inst][pos][max_E];
 * d_order[inst][max_E]: energy columns in ascending-energy order; d_keys[inst][max_E]: those
 * energies (float64, distinct, no NaN); d_n_keys[inst]; d_limit[inst]: positions < limit take
 * part (the reference stops an instrument's chain at its `complete` step, :315-319);
 * d_gathered_etot (+ r * rank_stride uint32 elements): rank r's per-energy totals [inst][max_E]
 * (may be NULL on rank 0).  d_ycand[inst]: order-preserving int64 key of the largest candidate
 * (decoded by csg_pool_pack_results; "none" when no position took part). */
CSG_API int csg_pool_energy_candidates(csg_ctx* ctx, const uint32_t* d_ehist, int n_inst, int max_pos, int max_E,
                               const int32_t* d_order, const double* d_keys, const int32_t* d_n_keys,
                               const int32_t* d_limit, const uint32_t* d_gathered_etot, size_t rank_stride,
                               int rank, int64_t* d_ycand);
/* d_out[n_out >= n_req + n_inst + 5] (double) = [values | y candidates (-inf: none; d_ycand may be
 * NULL) | the 4 selection flags | *d_peer_error (may be NULL) | zero padding]: one payload, so one
 * last exchange + csg_pool_reduce_max() finishes the step on every rank. */
CSG_API int csg_pool_pack_results(csg_ctx* ctx, const double* d_values, int n_req, const int64_t* d_ycand, int n_inst,
                          const int32_t* d_flags, const void* d_peer_error, double* d_out, int n_out);
CSG_API int csg_pool_reduce_max(csg_ctx* ctx, const double* d_gathered, int n_ranks, int n, double* d_out);

/* ------------------------------------------- peer exchange (NVLink / NVSwitch stores) */
/* The exchange step of the global extrema (SURVEY.md section 8e) without library collectives:
 * every rank owns a mailbox in its HBM; an all-gather is one kernel that stores the payload
 * into every peer's mailbox, publishes an epoch flag (release, system scope) and waits for every
 * rank's flag (acquire).  See csrc/peer.cu. */
typedef struct csg_peer csg_peer;
/* slot_bytes: largest payload of one rank.  ipc_handle_64 (may be NULL): receives the 64-byte
 * cudaIpcMemHandle_t of this rank's mailbox (zeros when the platform has no IPC). */
CSG_API int csg_peer_create(csg_ctx* ctx, int rank, int n_ranks, size_t slot_bytes, csg_peer** out, void* ipc_handle_64);
CSG_API void* csg_peer_mailbox(csg_peer* peer);
/* all_handles: n_ranks x 64 bytes, rank order (one process per GPU). */
CSG_API int csg_peer_connect_ipc(csg_ctx* ctx, csg_peer* peer, const void* all_handles);
/* mailboxes[n_ranks]: csg_peer_mailbox() of every rank (ranks living in one process). */
CSG_API int csg_peer_connect_ptrs(csg_ctx* ctx, csg_peer* peer, void* const* mailboxes);
/* nbytes: multiple of 16, <= slot_bytes; *d_gathered: n_ranks payloads, nbytes apart, valid until
 * the third following exchange. */
CSG_API int csg_peer_allgather(csg_ctx* ctx, csg_peer* peer, const void* d_src, size_t nbytes, void** d_gathered);
/* int32 on the device: 0, or 1 + the rank whose flag did not arrive within the timeout (20 s, or
 * CSG_PEER_TIMEOUT_S: a rank may arrive seconds late -- first-step planning, lazy module loads). */
CSG_API void* csg_peer_error_word(csg_peer* peer);
/* Time the last `last_n` (<= 64) all-gathers spent waiting for the other ranks' epochs, in microseconds:
 * rank skew + link latency, measured inside the exchange kernel with clock64 (synchronises the stream). */
CSG_API int csg_peer_wait_stats(csg_ctx* ctx, csg_peer* peer, int last_n, double* mean_us, double* max_us);
/* Timeline of the last `last_n` (<= 64) exchanges, oldest first: ns3[3k + {0,1,2}] = %globaltimer nanoseconds at
 * which exchange k's kernel started, published its epoch to the peers, and saw every peer's epoch; *n_written =
 * how many exchanges were written.  The gap between "saw" of one exchange and "started" of the next is the
 * consumer / producer kernels in between. */
CSG_API int csg_peer_trace(csg_ctx* ctx, csg_peer* peer, int last_n, uint64_t* ns3, int* n_written);
CSG_API int csg_peer_clear_error(csg_ctx* ctx, csg_peer* peer); /* on the ctx stream */
/* Unmap the other ranks' mailboxes (every rank does this, then a barrier, before any rank destroys its
 * own mailbox: an exporter must not free memory an importer still has open). */
CSG_API int csg_peer_disconnect(csg_ctx* ctx, csg_peer* peer);
CSG_API int csg_peer_destroy(csg_ctx* ctx, csg_peer* peer);

/* --------------------------------------------- K4: figure mosaics -> DEFLATE (PNG hand-off) */
/* Replaces fig.savefig() of CS/fast/process_orbit.py:98-117 / CS/generic_batch.py:108-113 for figures
 * whose panels are K3 rasters in HBM.  A canvas is a list of tiles; every tile is a source raster
 * resampled nearest-neighbour into its rectangle on the canvas -- a K3 panel filling its axes box the way
 * imshow(aspect="auto") does at display resolution (CS/plotting.py:280-287,606-611; 4800 x 2400 pixels
 * for the FAST grids, CS/fast/process_orbit.py:110), or a host-drawn annotation sprite (text, tick marks,
 * frames, colour bars) from the overlay atlas at its own size.  The mosaic
 * (figure.SpectrogramFigure.compose is its host oracle) is evaluated per scanline inside the encoder and
 * written as Huffman-coded DEFLATE blocks, one per segment (<= 1024 pixels of one scanline), each closed
 * by an empty stored block so that segments concatenate bytewise.  Only scanlines with new content are
 * encoded (d_rows lists them per canvas); runs of repeated lines are constants the host splices in.
 * See csrc/png.cu. */
typedef struct {
  int64_t rgba_off;  /* pixel offset of the [ne][nt] source raster in d_rgba (flags bit 0 clear) or d_overlay */
  int32_t ne, nt;    /* source rows x columns                                                               */
  int32_t x, y;      /* top-left corner on the canvas                                                        */
  int32_t w, h;      /* size on the canvas: source index = floor((d + 0.5) * n_src / n_dst), float32         */
  int32_t vline_first, vline_count; /* cusp lines burnt into this tile (d_vlines)                            */
  int32_t flags;     /* bit 0: source in the overlay atlas; bit 1: source row 0 is the TOP row (a K3 raster
                        stores the lowest energy first and is flipped: imshow origin="lower"); bit 2
                        (TILE_ROW_MAP): canvas row r shows storage row d_row_maps[row_map + (r - y)], clamped
                        to [0, ne-1], instead of the nearest row and the flip (a panel on a log energy axis)  */
  int32_t row_map;   /* with bit 2: offset of the tile's h-entry map in d_row_maps                           */
} csg_png_tile; /* 48 bytes */
typedef struct {
  int32_t col, half; /* canvas columns col-half .. col+half, relative to the tile's left edge              */
  uint32_t rgba;
  int32_t pad;
} csg_png_vline; /* 16 bytes */
typedef struct {
  int32_t W, H;
  int32_t tile_first, tile_count; /* first matching tile wins: list annotations before what they cover      */
  uint32_t background;
  int32_t seg_first;    /* id of the canvas' first segment; segments are numbered listed row by listed row */
  int32_t segs_per_row; /* ceil(W / 1024)                                                                  */
  int32_t row_first;    /* index in d_rows of the canvas' first listed scanline                            */
} csg_png_canvas; /* 32 bytes */
/* A segment whose filtered bytes are all zero (it repeats the line above: most segments of a scanline on
 * which only one colour bar or one label moved on) is a constant of its length n_raw = 4 * pixels (+ 1 with
 * the filter byte, which is 2): the host supplies the byte-aligned DEFLATE piece ready made (png.py:
 * zlib's encoding), the encoder copies it instead of forming tokens. */
typedef struct {
  int32_t n_raw; /* filtered bytes of the segment                     */
  int32_t len;   /* bytes of the piece (<= 56)                        */
  uint8_t bytes[56];
} csg_png_zero_segment; /* 64 bytes */

/* The DEFLATE code of a batch of figures.  Codes are bit-reversed (ready for the LSB-first stream);
 * len_code[n] / dist_code[k] = the Huffman code of a match of 4n bytes / at distance 4k bytes followed
 * by its extra bits; *_len = total bits; *_sym = the symbol (for csg_png_count).  Literal / length
 * codes may use at most 9 bits, distance codes at most 7.  header = the block header every segment
 * starts with, BFINAL/BTYPE included: 3 bits for the fixed code, BTYPE=10 + code lengths for a custom
 * one (png.py builds it from the counts of csg_png_count). */
typedef struct {
  uint16_t lit_code[256];
  uint8_t lit_len[256];
  uint32_t len_code[65];
  uint32_t dist_code[129];
  uint16_t len_sym[65];
  uint8_t len_len[65];
  uint8_t dist_len[129];
  uint8_t dist_sym[129];
  uint8_t eob_len;
  uint16_t eob_code;
  int32_t header_bits;
  uint32_t header[40];
} csg_png_tables;
CSG_API int csg_png_fixed_tables(csg_png_tables* out);                        /* RFC 1951 fixed code    */
CSG_API int csg_png_set_tables(csg_ctx* ctx, const csg_png_tables* tables);  /* NULL: the fixed code   */
/* Symbol statistics of every stride-th segment: d_counts[286 + 30] (uint32, zeroed by the caller) +=
 * literal / length symbol counts, then distance symbol counts.  Nothing is encoded.  d_row_maps as for
 * csg_png_encode (the counts must see the pixels the encode pass will encode). */
CSG_API int csg_png_count(csg_ctx* ctx, const uint8_t* d_rgba, const uint8_t* d_overlay, const csg_png_canvas* d_canvases,
                  int n_canvases, const csg_png_tile* d_tiles, const csg_png_vline* d_vlines, const int32_t* d_rows,
                  int n_segments, int stride, uint32_t* d_counts, const csg_png_zero_segment* d_zero, int n_zero,
                  const int32_t* d_row_maps);
CSG_API int32_t csg_png_slot_bytes(void);                    /* capacity of one segment's output slot        */
CSG_API int32_t csg_png_segments(int32_t W, int32_t n_rows); /* segments of n_rows listed scanlines of width W */
CSG_API int32_t csg_png_max_segment_tiles(void);             /* tiles one segment may intersect               */
/* d_rows: ascending scanline numbers with new content, canvas after canvas (csg_png_canvas.row_first).
 * d_slots[n_segments][slot_bytes]: the encoded segments; d_sizes[n_segments]: their byte counts;
 * d_adler[n_segments][2]: (sum of bytes, sum of (n - t) * byte_t) mod 65521 of the filtered bytes;
 * d_error (int32, may be NULL, zeroed by the caller): 1 + the canvas in which more than
 * csg_png_max_segment_tiles() tiles met in one segment, or -(1 + the canvas) in which a TILE_ROW_MAP tile
 * met a NULL d_row_maps (either way its output is wrong: the host raises).
 * d_row_maps (int32, may be NULL when no tile sets TILE_ROW_MAP): the row maps of the tiles that do. */
CSG_API int csg_png_encode(csg_ctx* ctx, const uint8_t* d_rgba, const uint8_t* d_overlay, const csg_png_canvas* d_canvases,
                   int n_canvases, const csg_png_tile* d_tiles, const csg_png_vline* d_vlines, const int32_t* d_rows,
                   int n_segments, uint8_t* d_slots, int32_t* d_sizes, uint32_t* d_adler, int32_t* d_error,
                   const csg_png_zero_segment* d_zero, int n_zero, /* d_zero may be NULL */
                   const int32_t* d_row_maps);
/* d_packed + d_offsets[s] <- slot s (d_offsets: exclusive prefix sum of d_sizes, from the host). */
CSG_API int csg_png_compact(csg_ctx* ctx, const uint8_t* d_slots, const int32_t* d_sizes, const int64_t* d_offsets,
                    int n_segments, uint8_t* d_packed);

/* Host half of K4: frame + write.  One PNG file per entry, built in place from the read-back buffer (no
 * copy: one CRC-32 pass, then writev) on `n_threads` native threads, outside the interpreter lock:
 *   signature, IHDR, ONE IDAT = zlib header + for every content row its `segs_per_row` device pieces
 *   (packed[offsets[s] .. offsets[s+1]), s from seg_first) + after a row followed by g repeated scanlines a
 *   constant "g x (filter Up + 4*width zero bytes)" DEFLATE piece + final empty block + Adler-32 (combined
 *   from adler[s][2], the device's per-piece partial sums), IEND.
 * Replaces the host side of fig.savefig (CS/fast/process_orbit.py:98-117: Agg's PNG writer).  `rows`: the
 * content scanlines of every canvas (csg_png_encode's d_rows, host copy).  Returns CSG_ERR_IO when any file
 * failed (status = errno per file), CSG_OK otherwise. */
typedef struct csg_png_file {
  const char* path;     /* destination (created or truncated) */
  int64_t row_first;    /* index of the canvas' first content row in rows[] */
  int64_t seg_first;    /* index of its first segment in offsets[] / adler[] */
  int64_t file_bytes;   /* out: size of the file written */
  int32_t width, height;
  int32_t n_rows;       /* content rows */
  int32_t segs_per_row; /* ceil(width / 1024) */
  int32_t status;       /* out: 0 or errno */
  int32_t pad;
} csg_png_file; /* 56 bytes */
CSG_API int csg_png_write_files(csg_png_file* files, int n_files, const int32_t* rows, const uint8_t* packed,
                                const int64_t* offsets, const uint32_t* adler, int n_threads);

/* ------------------------------------------------ ingest: native CDF v3 reader (host only) */
/* Replaces the four cdflib `varget` calls of load_fast_cdf_dataset (CS/cdf_utils.py:247-251) for the
 * batch path: the file is memory-mapped once, the variable index (zVDR / rVDR -> VXR -> VVR / CVVR)
 * is walked and only the records asked for are copied or inflated (gzip) into caller memory -- a
 * pinned staging slot -- in host byte order, row-major.  `energy[0,0,:]` and `pitch_angle[0,:,0]`
 * (CS/cdf_utils.py:252-253) need record 0 only, not the data-sized variables the reference decodes.
 * Thread-safe per handle (one handle per thread); errors: csg_cdf_last_error() (thread-local).
 * See csrc/cdf.cpp for the supported subset (IEEE encodings, row-major, plain / gzip). */
#define CSG_CDF_MAX_DIMS 8
typedef struct csg_cdf csg_cdf;
typedef struct {
  char name[260];
  int32_t data_type;  /* CDF data type code: 21/44 REAL4/FLOAT, 22/45 REAL8/DOUBLE, 31 EPOCH, 33 TT2000, 4 INT4 ... */
  int32_t elem_bytes; /* bytes of one value; 0 = unsupported type                                            */
  int32_t n_dims;     /* varying dimensions of one record                                                    */
  int32_t dims[CSG_CDF_MAX_DIMS];
  int32_t rec_vary, compressed, row_major;
  int64_t n_records;         /* records written (MaxRec + 1)                                                 */
  int64_t values_per_record; /* product of dims                                                              */
} csg_cdf_var;               /* 336 bytes */
CSG_API int csg_cdf_open(const char* path, csg_cdf** out);
CSG_API void csg_cdf_close(csg_cdf* cdf);
CSG_API int csg_cdf_var_count(csg_cdf* cdf);
/* by name, or by index when name is NULL */
CSG_API int csg_cdf_var_info(csg_cdf* cdf, const char* name, int index, csg_cdf_var* info);
/* records [rec0, rec0 + n_rec) of the variable -> h_dst (n_rec * values_per_record * elem_bytes bytes) */
CSG_API int csg_cdf_read(csg_cdf* cdf, const char* name, int64_t rec0, int64_t n_rec, void* h_dst, size_t dst_bytes);
CSG_API const char* csg_cdf_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* CSGPU_H */
