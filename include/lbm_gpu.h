/*
 * lbm_gpu.h -- C-ABI of the B200 d2q9-bgk timestep loop (liblbm_b200.so).
 *
 * The reference (ChuyueL/advanced-hpc-lbm, one C99 file) has no plugin or FFI layer:
 * the hot path is the plain C call
 *
 *     av_vels[tt] = timestep_new2(params, cells, tmp_cells, obstacles);   d2q9-bgk.c:182
 *     swap(&cells, &tmp_cells);                                           d2q9-bgk.c:190
 *
 * inside `for (tt = 0; tt < params.maxIters; tt++)` (d2q9-bgk.c:180-201).  A per-step
 * boundary would force one host synchronisation per step, so this ABI replaces the
 * WHOLE loop: the lattice lives in HBM between calls and lbm_gpu_run() executes any
 * number of steps without touching the host.  Every entry point takes plain pointers
 * and sizes; none of them calls exit() -- they return 0 on success and a non-zero
 * code on failure, with the text available from lbm_gpu_last_error() so that a C host
 * can print it in the reference's die() format (d2q9-bgk.c:3001-3007).
 *
 * Layouts at the boundary are the reference's own:
 *   cells      array-of-structs t_speed{float speeds[9]} (d2q9-bgk.c:76-79), cell
 *              (ii,jj) at index ii + jj*nx, i.e. 9 consecutive floats per cell;
 *   obstacles  one int per cell, 0 = fluid, non-zero = blocked (d2q9-bgk.c:2797);
 *   av_vels    one float per step (d2q9-bgk.c:2866).
 * Inside the library the lattice is structure-of-arrays, double-buffered, with a
 * bit-packed mask (DESIGN.md section 3).
 *
 * Speeds: 0 rest, 1 E, 2 N, 3 W, 4 S, 5 NE, 6 NW, 7 SW, 8 SE (d2q9-bgk.c:7-13).
 */
#ifndef LBM_GPU_H
#define LBM_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Same members, order and types as the reference's t_param (d2q9-bgk.c:64-73). */
typedef struct {
  int   nx;            /* no. of cells in x-direction */
  int   ny;            /* no. of cells in y-direction */
  int   maxIters;      /* no. of iterations (informational for the library) */
  int   reynolds_dim;  /* dimension for Reynolds number */
  float density;       /* density per link */
  float accel;         /* density redistribution */
  float omega;         /* relaxation parameter */
} lbm_param;

/* Double-precision twin, used only by the validation build of the kernel that
 * reproduces the reference's (double precision) golden files in check/. */
typedef struct {
  int    nx, ny, maxIters, reynolds_dim;
  double density, accel, omega;
} lbm_param_f64;

typedef struct lbm_gpu lbm_gpu;   /* opaque handle: one lattice on one or more GPUs */

/* lbm_gpu_create flags.  At most one LBM_GPU_KERNEL_* flag: a create that forces two is refused. */
#define LBM_GPU_DEFAULT        0u
#define LBM_GPU_STRICT         1u  /* source operation order, no FMA contraction: bit-exact
                                      against a -O2 -ffp-contract=off build of the reference */
#define LBM_GPU_OBST_BITS      2u  /* `obstacles` is bit-packed: uint32 words, bit (ii & 31) of
                                      word [jj * ((nx + 31) / 32) + ii / 32]; for grids whose
                                      int mask does not fit in host memory */
#define LBM_GPU_KERNEL_SCALAR  4u  /* force the one-cell-per-thread kernel (any nx) */
#define LBM_GPU_KERNEL_TMA     8u  /* force the TMA-staged kernel (fp32; measured equal/slower than
                                      VEC4, kept as the comparison point) */
#define LBM_GPU_KERNEL_VEC4   16u  /* force the 128-bit direct-load kernel (one launch per timestep) */
#define LBM_GPU_KERNEL_PERSISTENT 64u /* force the persistent cooperative kernel (all steps of a run
                                      in one launch; single GPU).  Chosen by default
                                      for grids small enough to live in L2 */
#define LBM_GPU_KERNEL_CLUSTER 256u /* force the thread-block-cluster kernel: the lattice lives in the
                                      distributed shared memory of one cluster for the whole run (single
                                      GPU, fp32, at most ~48 k cells).  Measured no faster than the persistent kernel, never
                                      chosen by default */
#define LBM_GPU_POOL         128u  /* take the lattice from the device's stream-ordered memory pool and
                                      leave it there on destroy: a host that creates many lattices in
                                      one process (sweeps) skips cudaMalloc/cudaFree of ~20 GB each time */
#define LBM_GPU_SYNC_FLAGS    32u  /* lbm_gpu_create with n_gpus > 1: insist on the device-side flag
                                      protocol between the slabs (the default whenever every slab has a
                                      GPU of its own; an error if two slabs share one) */
#define LBM_GPU_KERNEL_TB2   512u  /* force the two-timesteps-per-pass kernel (temporal blocking: each
                                      distribution crosses HBM once per TWO timesteps).  The default for
                                      fp32 grids beyond L2 with nx a multiple of 4, nx >= 32 and at least
                                      8 rows per GPU; an odd step of a run is done by the one-step kernel */
#define LBM_GPU_KERNEL_PAIRS 2048u  /* force the small-grid persistent kernel that meets at a grid barrier once
                                      per TWO timesteps (single GPU, fp32, nx a multiple of 4 and <= 256); the
                                      default for such grids */
#define LBM_GPU_KERNEL_TB3  4096u  /* force the three-timesteps-per-pass kernel (each distribution crosses
                                      HBM once per THREE timesteps; fp32, nx a multiple of 4 and >= 32, the
                                      whole grid on one GPU, at least 12 rows).  The default for such grids
                                      that are large enough (otherwise LBM_GPU_KERNEL_TB2 is); the last one
                                      or two steps of a run are done by the one- or two-step kernel */
#define LBM_GPU_SYNC_EVENTS 1024u  /* lbm_gpu_create with n_gpus > 1: order the slabs with CUDA events
                                      (host-recorded, no device-side waiting) even when every slab has its
                                      own GPU; always used when slabs share a GPU */
/* Shifted binary16 lattice storage: half the bytes per cell (larger grids, fewer bytes per update)
 * for some accuracy.  With c_k the rest-state value of speed k computed in fp32 as for the rest
 * state (density*4/9, density/9, density/36), the lattice holds s_k = __float2half_rn(f_k - c_k)
 * (one fp32 subtract, round to nearest even) and is read as f_k = __half2float(s_k) + c_k (one fp32
 * add).  A timestep decodes, runs the ordinary fp32 step (accelerate row ny-2, pull, rebound or
 * collide), and encodes.  Not rounded: the accelerated values of row ny-2 within a step, and the |u|
 * that goes into av_vels (taken from the fp32 results before they are encoded).  The rest state
 * encodes to zeros; download / final_fields / av_velocity / lbm_gpu_digest see the decoded fp32
 * values; upload and create with cells_aos encode (and so round).  With LBM_GPU_STRICT the result is
 * bit-exact against the fp32 reference arithmetic with the same encode/decode between steps.
 * lbm_gpu_create only, fp32, n_gpus == 1; the only kernels that may be forced are
 * LBM_GPU_KERNEL_VEC4 (one step per pass) and LBM_GPU_KERNEL_TB2 (two steps per pass, nx a multiple
 * of 8 and >= 32, at least 8 rows; the default where it applies).  The accuracy of the shipped
 * inputs is in INTEGRATION.md. */
#define LBM_GPU_STORE_F16   8192u

/* Information about a handle (lbm_gpu_get_info). */
typedef struct {
  int       nx, ny;
  int       n_gpus;            /* slabs held by THIS process */
  int       is_f64;
  int       kernel;            /* LBM_GPU_KERNEL_* that runs the next lbm_gpu_run (chosen at create,
                                  again at lbm_gpu_ipc_connect / _connect_all) */
  int       pitch;             /* elements per stored lattice row */
  long long free_cells;        /* non-obstacle cells of the WHOLE grid (if known) or of the local rows */
  long long local_free_cells;  /* non-obstacle cells of the rows held by this process */
  long long local_row0;        /* first global row held by this process */
  long long local_rows;        /* number of rows held by this process */
  long long steps_done;        /* timesteps executed since creation */
  long long kernel_launches;   /* CUDA kernels this handle has launched since creation */
  double    last_run_device_ms;/* device time of the last lbm_gpu_run (CUDA events, max over local GPUs) */
  double    last_step_kernel_ms;/* mean duration of the step kernel in the last run (same events) */
  size_t    device_bytes;      /* device memory held per GPU (largest slab) */
} lbm_gpu_info;

/* Number of CUDA devices visible; <0 on error. */
int lbm_gpu_device_count(void);

/*
 * Replaces the tail of initialise() (d2q9-bgk.c:2787-2857: allocate + fill + obstacle
 * array) for the device side: copies the caller's arrays into HBM (AoS -> SoA planes,
 * int mask -> bits) and splits the rows into `n_gpus` contiguous slabs on devices
 * device_ids[0..n_gpus) (NULL = 0,1,2,...).  The caller keeps ownership of its arrays.
 *   cells_aos == NULL  =>  the reference's rest state (d2q9-bgk.c:2802-2823) is
 *                          generated on the device; mandatory for grids whose AoS
 *                          copy does not fit in host memory.
 *   obstacles == NULL  =>  no blocked cells.
 * Requirements: nx >= 1, ny >= 2 (the reference accelerates row ny-2, d2q9-bgk.c:240),
 * ny >= n_gpus.
 */
int lbm_gpu_create(const lbm_param* params, const float* cells_aos, const void* obstacles,
                   int n_gpus, const int* device_ids, unsigned flags, lbm_gpu** out);
int lbm_gpu_create_f64(const lbm_param_f64* params, const double* cells_aos, const void* obstacles,
                       int n_gpus, const int* device_ids, unsigned flags, lbm_gpu** out);

/*
 * One-process-per-GPU form (torchrun / MPI style launch): this process holds global
 * rows [row0, row0 + nrows) of an nx x ny grid on `device`.  cells_aos / obstacles
 * describe ONLY those rows (nrows * nx cells).  After creating, every rank must
 *   1. lbm_gpu_ipc_export() its descriptor,
 *   2. exchange descriptors with the ranks holding the rows below (row0-1, periodic)
 *      and above (row0+nrows, periodic) by any host-side means,
 *   3. lbm_gpu_ipc_connect() with those two descriptors -- or, better, all-gather the
 *      descriptors of ALL ranks and call lbm_gpu_ipc_connect_all(): the library then finds
 *      its two neighbours itself, learns the whole grid's free-cell count (so lbm_gpu_run
 *      returns true averages without lbm_gpu_set_global_free_cells) and, knowing every
 *      slab's height, selects the two-timesteps-per-pass kernel where every rank can run
 *      it, a decision all ranks must share.  Otherwise, and always with the two-descriptor
 *      form, a ring runs the one-step kernel (unless another was forced), also on a slab
 *      that holds the whole grid and took a multi-step kernel at create,
 *   4. pass a host barrier over all ranks, then lbm_gpu_ipc_prepare(), then a second
 *      host barrier -- after which lbm_gpu_run() may be called (same n_steps on
 *      every rank).
 * The ghost rows are written straight into the neighbours' HBM by the step kernel
 * (peer stores over NVLink) and ordered by device-side flags: no collective, no host
 * synchronisation per step.
 *
 * Failure and teardown.  lbm_gpu_run() returns only after both neighbours have completed
 * the same number of kernel passes (a bounded device-side wait at the end of the run), so
 * on return nothing is in flight towards this rank's window any more: destroying,
 * uploading or re-creating needs no host barrier.  Every device-side wait for a neighbour
 * is bounded (LBM_GPU_SYNC_TIMEOUT_MS, default 10000): if a neighbour never arrives -- its
 * process died, or it was asked for a different n_steps -- the waiting rank gives up, raises
 * an abort word in its neighbours so that the whole ring drains, and lbm_gpu_run() returns
 * non-zero with the reason in lbm_gpu_last_error() (the reference's die() convention,
 * d2q9-bgk.c:3001-3007).  The lattice of an abandoned run is void; further runs are refused.
 */
#define LBM_GPU_IPC_DESC_BYTES 256
int lbm_gpu_create_slab(const lbm_param* params, long long row0, long long nrows, int device,
                        const float* cells_aos_rows, const void* obstacles_rows,
                        unsigned flags, lbm_gpu** out);
int lbm_gpu_ipc_export(lbm_gpu* h, void* desc /* LBM_GPU_IPC_DESC_BYTES */);
int lbm_gpu_ipc_connect(lbm_gpu* h, const void* desc_below, const void* desc_above);
int lbm_gpu_ipc_connect_all(lbm_gpu* h, const void* descs /* n x LBM_GPU_IPC_DESC_BYTES */, int n);
int lbm_gpu_ipc_prepare(lbm_gpu* h);

/*
 * Replaces the loop `for (tt...) { av_vels[tt] = timestep_new2(...); swap(...); }`
 * (d2q9-bgk.c:180-201).  Runs n_steps timesteps back to back on the device(s); blocks
 * until they are finished (so a gettimeofday() pair around it is an honest compute
 * time).  av_vels_out (n_steps floats, may be NULL) receives each step's average
 * velocity = sum of |u| over non-obstacle cells / number of such cells
 * (d2q9-bgk.c:1103-1130,:1811), accumulated exactly on the device and reduced once
 * at the end.  For a slab handle (one process per GPU) av_vels_out receives this
 * process's share sum|u|/free_cells_of_the_whole_grid only if the whole-grid count was
 * given with lbm_gpu_set_global_free_cells(); use lbm_gpu_run_sums() otherwise.
 */
int lbm_gpu_run(lbm_gpu* h, int n_steps, float* av_vels_out);
int lbm_gpu_run_f64(lbm_gpu* h, int n_steps, double* av_vels_out);

/* Same, but returns the raw per-step sums of |u| over the rows held by this process
 * as doubles (sums_out[n_steps]); a multi-process caller adds them across ranks and
 * divides by the global free-cell count. */
int lbm_gpu_run_sums(lbm_gpu* h, int n_steps, double* sums_out);
int lbm_gpu_set_global_free_cells(lbm_gpu* h, long long free_cells);

/*
 * Parameter sweeps: advance n independent lattices by n_steps each, together on one GPU.
 * Same result, bit for bit, as calling lbm_gpu_run(handles[i], n_steps, av_vels_out + i*n_steps)
 * for i = 0..n-1 in turn; a small lattice leaves most of the GPU idle, so running many in
 * one kernel costs little more than running one.  av_vels_out: n * n_steps floats,
 * member-major, may be NULL.
 * Members are ordinary handles from lbm_gpu_create.  They must share the device, nx, ny and
 * the LBM_GPU_STRICT setting, and each must be fp32, a single slab, not failed, and run
 * LBM_GPU_KERNEL_PAIRS (the default for fp32 grids with nx a multiple of 4 and <= 256).
 * They may differ in density, accel, omega, obstacles, contents and history (steps done).
 * Otherwise the call is refused before anything runs (no handle changes), as it is for
 * n < 1, a NULL or duplicate handle, or n_steps < 0.  Afterwards each member is exactly
 * where lbm_gpu_run would have left it; its last_run_device_ms is the whole batch's time.
 */
int lbm_gpu_run_batch(lbm_gpu* const* handles, int n, int n_steps, float* av_vels_out);

/*
 * The reference keeps the lattice on the host, so calc_reynolds (d2q9-bgk.c:2893) and
 * write_values (d2q9-bgk.c:2918) read it directly.  Here the host asks for it:
 *   download        whole local lattice, AoS like t_speed (9 floats per cell)
 *   download_rows   global rows [row0,row0+nrows) only (must be held by this process)
 *   final_fields    u_x, u_y, |u|, pressure per cell exactly as write_values computes
 *                   them (d2q9-bgk.c:2937-2976; obstacle cells: 0,0,0,density/3), for a
 *                   row range, so a writer can stream huge grids slab by slab.  Any of
 *                   the four output pointers may be NULL.
 *   av_velocity     av_velocity() of the current lattice (d2q9-bgk.c:2665-2714) for
 *                   the Reynolds number line; sum over local rows / free cells.  NaN when
 *                   a fluid cell's |u| is NaN (a NaN or zero-density cell) or not below 2,
 *                   as lbm_gpu_run reports such a step.
 * For download_rows and final_fields, nrows = 0 succeeds and writes nothing; a negative
 * nrows, or rows not held by this process, is refused before anything is written.
 */
int lbm_gpu_download(lbm_gpu* h, float* cells_aos_out);
int lbm_gpu_download_rows(lbm_gpu* h, long long row0, long long nrows, float* cells_aos_out);
int lbm_gpu_final_fields(lbm_gpu* h, long long row0, long long nrows,
                         float* u_x, float* u_y, float* u, float* pressure);
int lbm_gpu_av_velocity(lbm_gpu* h, float* av_out);

/*
 * Block-averaged fields, computed on the device so that only the coarse picture crosses PCIe
 * (a snapshot of a grid too large to read out cell by cell, or a time series of one).
 * The grid is cut into factor x factor blocks from cell (0,0): ncx = ceil(nx/factor) blocks per
 * coarse row, ceil(ny/factor) coarse rows; coarse row J covers global rows [J*factor,
 * min(J*factor + factor, ny)), and the blocks at the right and top edges are smaller.  Each
 * non-NULL output receives ncrows x ncx values, row-major, of coarse rows [crow0, crow0+ncrows).
 *
 * The value of a block is the mean over ALL its cells (obstacle cells included, with the
 * 0, 0, 0, density/3 that final_fields reports for them) of lbm_gpu_final_fields' per-cell values,
 * bit for bit; for u_x and u_y that is the superficial (volume-averaged) velocity, so the coarse
 * field carries the flux of the fine one.  The arithmetic is exact and the same for any slab
 * split: each cell value v adds round_half_even(v * 2^32) to an int64 sum S, and the mean is
 * (float)((double)S * 2^-32 / cells), computed in double and rounded once to fp32.  A block in
 * which a value is NaN, infinite or of magnitude 2^15 or more reports NaN for that field (below
 * that bound the sum of a 256 x 256 block stays under 2^63).
 *
 *   LBM_GPU_FIELDS_F32  float outputs: the mean.
 *   LBM_GPU_FIELDS_F16  binary16 outputs (uint16_t bit patterns), half the bytes: u_x, u_y and |u|
 *                       hold __float2half_rn(mean); pressure is shifted, as the lattice is under
 *                       LBM_GPU_STORE_F16, because it varies by ~1e-4 relative around density/3
 *                       and binary16 keeps 11 bits: it holds __float2half_rn(mean - p0), the
 *                       subtraction in fp32, with p0 = (float)density * (1.0f/3.0f) the obstacle
 *                       pressure of final_fields.  Decode it as __half2float(h) + p0.
 * factor == 1:  with F16 each cell's own values are converted (pressure shifted): the
 * full-resolution read-out at half the size, with no fixed-point step; with F32 the call is
 * lbm_gpu_final_fields.
 *
 * factor 1..256.  A handle with several slabs in this process adds the integer sums of a
 * coarse row cut by a slab boundary on the host, so the result equals one slab's bit for bit.
 * A slab handle (one process per GPU) serves the coarse rows whose fine rows it holds entirely;
 * a request for any other coarse row is refused with a message that names it.  Refused before
 * anything is enqueued or written: factor out of range, an unknown format, ncrows < 0, coarse
 * rows beyond the grid or not held, and double-precision handles (use
 * lbm_gpu_final_fields_f64).  ncrows = 0 succeeds and writes nothing.  The lattice, steps_done
 * and the kernel choice are not touched, so run(a); coarse_fields; run(b) equals run(a+b).
 */
#define LBM_GPU_FIELDS_F32 0u
#define LBM_GPU_FIELDS_F16 1u
int lbm_gpu_coarse_fields(lbm_gpu* h, int factor, unsigned format, long long crow0, long long ncrows,
                          void* u_x, void* u_y, void* u, void* pressure);

int lbm_gpu_download_f64(lbm_gpu* h, double* cells_aos_out);
int lbm_gpu_final_fields_f64(lbm_gpu* h, long long row0, long long nrows,
                             double* u_x, double* u_y, double* u, double* pressure);
int lbm_gpu_av_velocity_f64(lbm_gpu* h, double* av_out);

/*
 * Exact digest of the rows held by this process, computed on the device:
 *   total_density  the reference's total_density() (d2q9-bgk.c:2900-2916; its -DDEBUG mass
 *                  conservation check), summed in 2^-32 fixed point;
 *   checksum       wrapping 64-bit sum of bit_pattern(speed) * odd_weight(global cell, k).
 * Both are integer sums: independent of summation order and additive over slabs and
 * ranks, so two runs hold the same lattice iff their checksums agree -- the way to
 * compare lattices too large to download (16384 x 131072 is 77 GB).  Either may be NULL.
 * A speed that is NaN, infinite or of magnitude 2^31 or more has no fixed-point value:
 * total_density is then NaN, as the reference's sum would be; the checksum is unaffected.
 */
int lbm_gpu_digest(lbm_gpu* h, double* total_density, unsigned long long* checksum);

/*
 * Force on obstacles by momentum exchange, computed on the device: the drag (x) and lift (y) on
 * the solid cells inside each of n_boxes boxes, for a time series of a flow past obstacles without
 * moving the lattice across PCIe.
 *
 * At state t (after t steps):
 *   f~    the values step t+1 streams: the stored lattice values, except that on row ny-2 speeds
 *         1, 3, 5, 6, 7 and 8 hold their values after accelerate_flow (the side row);
 *   S     the obstacle cells;  c_k the speed vectors (order above, +y = towards row ny-1);
 *   x +- c_k wraps periodically in x and y.
 * The force exerted on the solid cells of box B during step t+1 is
 *
 *   F_B(t) = sum over x_s in S and B of [   sum_{k=1..8, x_s - c_k not in S} c_k f~_k(x_s - c_k)
 *                                         - sum_{k=1..8, x_s + c_k not in S} c_k f~_k(x_s)       ]
 *
 * the momentum streaming into the solid minus the momentum it sends back (the values it holds
 * after its previous rebound).  Collision conserves momentum, so summed over all solid cells
 * P_fluid(t+1) = P~_fluid(t) - F_all(t) up to the collision's rounding (P~: fluid momentum of f~).
 * +x is the direction accelerate_flow pushes: F_x is the drag.
 *
 * Arithmetic: exact, and the same for any split of the rows over slabs.  Each value v that enters
 * becomes the signed integer round_half_even(v * 2^32) (the digest's conversion); the signed sums
 * S_B are exact integers in 128 bits.  Each integer is below 2^63 in magnitude and a solid cell
 * adds at most 12 of them per component, so |S_B| < 12 * 2^63 * cells < 2^127 for any grid of fewer
 * than 2^60 cells (18 EiB even as binary16): no sum the library can form wraps.  The output is the
 * correctly rounded double of S_B * 2^-32 (for the
 * binary16 lattice the values are the decoded fp32 ones).  A box with a contributing value that is
 * NaN, infinite or of magnitude 2^31 or more reports NaN for both components; other boxes are
 * unaffected.
 *
 *   boxes      n_boxes x {x0, y0, x1, y1}: half-open global cell ranges [x0, x1) x [y0, y1),
 *              0 <= x0 <= x1 <= nx, 0 <= y0 <= y1 <= ny.  They may overlap or be empty; a solid cell
 *              counts in every box that holds it.  NULL with n_boxes == 1: the whole grid.
 *   force_out  n_boxes x {fx, fy}.
 * n_boxes 1..256.  Works for fp32, fp64 and binary16 handles after any kernel.  The lattice,
 * steps_done and the kernel choice are not touched, so run(a); obstacle_force; run(b) equals
 * run(a+b).  A handle with several slabs in this process adds their integer sums before the
 * conversion.  A slab handle (lbm_gpu_create_slab) returns the share of the solid cells in its
 * rows (their links may reach the neighbours' rows): add the shares across ranks in double, one
 * rounding per rank, as with lbm_gpu_run_sums.
 * Refused before anything is enqueued or written, with a message that starts with
 * "lbm_gpu_obstacle_force:" and names the cause: n_boxes out of range, a NULL force_out, NULL boxes
 * with n_boxes != 1, a malformed box (named by its index), a handle whose earlier run was
 * abandoned, a slab handle that is not connected to its neighbours yet, and a slab handle that
 * loaded rows and has not called lbm_gpu_ipc_prepare yet (its ghost rows are stale, as for
 * lbm_gpu_run).  A box costs its own area: the mask words it covers and its boundary cells.
 */
int lbm_gpu_obstacle_force(lbm_gpu* h, int n_boxes, const int* boxes, double* force_out);

/* Replace the device lattice by the caller's (whole local rows, AoS). */
int lbm_gpu_upload(lbm_gpu* h, const float* cells_aos);
int lbm_gpu_upload_f64(lbm_gpu* h, const double* cells_aos);

/*
 * Checkpoint and restart: global rows [row0, row0 + nrows) of the STORED lattice, in the handle's
 * own storage type, nothing decoded or rounded.  Cell (ii, jj) is record ii + (jj - row0) * nx; a
 * record is the cell's 9 stored elements in speed order 0..8:
 *   fp32 handle                 float                                       36 bytes per cell
 *   fp64 handle (create_f64)    double                                      72 bytes per cell
 *   LBM_GPU_STORE_F16           uint16_t bit pattern of s_k = __float2half_rn(f_k - c_k)
 *                               (the stored shifted value, see LBM_GPU_STORE_F16)   18 bytes per cell
 * For fp32 and fp64 that is the t_speed AoS of lbm_gpu_download_rows / lbm_gpu_download_f64, byte for
 * byte.  For binary16 it is the stored bits themselves, at half the bytes of lbm_gpu_download:
 * download then upload decodes and re-encodes in fp32, which does not return every stored bit
 * pattern (at density 10, 8195 of the finite binary16 values change, though each decodes to the
 * same fp32 value as before), so a binary16 lattice is checkpointed with these two calls.
 *
 * After lbm_gpu_load_rows the handle behaves as if those rows had been computed into it: the side
 * row of row ny-2 and the ghost rows its kernel needs are rebuilt; run(a); save; [any process, any
 * slab layout] load; run(b) gives the bits of run(a + b).  steps_done, the kernel choice and the
 * obstacle mask are not touched (loading changes contents, not geometry).  Load between runs only.
 * A slab handle (lbm_gpu_create_slab) saves and loads the rows it holds; one that holds part of the
 * grid cannot rebuild its neighbours' ghost rows itself, so after loading, every rank passes a host
 * barrier, calls lbm_gpu_ipc_prepare, and passes a second barrier, as after creation; until its
 * lbm_gpu_ipc_prepare, lbm_gpu_run on that handle is refused.
 * Refused before anything is enqueued or written, with the call named in the message: a NULL
 * pointer with nrows > 0, nrows < 0, rows beyond the grid or not held by this process, a handle
 * whose earlier run was abandoned.  nrows = 0 succeeds and does nothing.
 */
int lbm_gpu_save_rows(lbm_gpu* h, long long row0, long long nrows, void* out);
int lbm_gpu_load_rows(lbm_gpu* h, long long row0, long long nrows, const void* in);

int lbm_gpu_get_info(lbm_gpu* h, lbm_gpu_info* info);

/* Page-locked host memory for the caller's input/output arrays (the reference uses
 * malloc, d2q9-bgk.c:2787-2866; pinned pages make the one-off copies run at full
 * PCIe speed).  Optional: every entry point also accepts ordinary malloc'ed memory. */
int lbm_gpu_host_alloc(size_t bytes, void** out);
void lbm_gpu_host_free(void* p);

/* Replaces the device part of finalise() (d2q9-bgk.c:2871-2890). */
void lbm_gpu_destroy(lbm_gpu* h);

/* Text of the last error on this thread ("" if none). */
const char* lbm_gpu_last_error(void);

/* ABI version of this header (2: lbm_gpu_ipc_connect_all, LBM_GPU_KERNEL_TB2, LBM_GPU_SYNC_EVENTS). */
int lbm_gpu_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* LBM_GPU_H */
