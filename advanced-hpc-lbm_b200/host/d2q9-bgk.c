/*
 * d2q9-bgk.c -- host program of the B200 build: same command line, same output files
 * and same stdout block as the reference's main() (d2q9-bgk.c:146-226 there), with the
 * timestep loop (d2q9-bgk.c:180-201) handed to liblbm_b200.so through the C-ABI of
 * include/lbm_gpu.h.  Plain C99; no CUDA in this file.
 *
 *   ./d2q9-bgk <paramfile> <obstaclefile>      -> final_state.dat, av_vels.dat in CWD
 *
 * The command line takes exactly two arguments like the reference (argc check
 * d2q9-bgk.c:159); everything else is an environment variable:
 *   LBM_GPUS=N             split the rows over N GPUs (default 1)
 *   LBM_PRECISION=f64      run the double-precision validation kernel (the golden files
 *                          in check/ were produced by a double build of the reference)
 *   LBM_PRECISION=f16      keep the lattice as shifted binary16 (LBM_GPU_STORE_F16: half the
 *                          device memory, fp32 arithmetic, less accurate; single GPU only)
 *   LBM_STRICT=1           source operation order, no FMA contraction
 *   LBM_KERNEL=scalar|vec4|persistent|tma|cluster|tb2|tb3|pairs   force a kernel variant
 *   LBM_SKIP_FINAL_STATE=1 do not write final_state.dat (huge synthetic grids: 16384^2
 *                          would be 24 GB of text)
 *   LBM_REPORT=1           print MLUPS / GB/s / device time after the contract lines
 *                          (LBM_REPORT=json: the same as one JSON line)
 *   LBM_DEBUG=1            the reference's -DDEBUG output (d2q9-bgk.c:196-200): after every
 *                          timestep print its number, average velocity and total density
 *                          (one lbm_gpu_run + lbm_gpu_digest per step: slow, for eyeballing
 *                          mass conservation)
 *   LBM_CHECKPOINT=path    after the last step, before final_state.dat, write a checkpoint
 *                          (stored lattice bit for bit, av_vels so far; format in lbm_io.h) to
 *                          path.tmp, then fsync and rename it to path
 *   LBM_CHECKPOINT_EVERY=k also write one after every k steps (step counts that are multiples
 *                          of k): the run is cut into lbm_gpu_run calls of k steps, which changes
 *                          no output bit
 *   LBM_RESTART=path       continue from a checkpoint of the same parameter file (maxIters may be
 *                          larger), obstacle file, LBM_PRECISION and LBM_STRICT; LBM_GPUS may
 *                          differ.  The header is checked before the GPU is touched; av_vels.dat
 *                          then holds all maxIters lines and both files equal an uninterrupted run's
 *   LBM_FORCE_EVERY=k      write forces.dat: the momentum-exchange force on the obstacles
 *                          (lbm_gpu_obstacle_force) at every state t = k, 2k, ... <= maxIters, one
 *                          line "t fx fy [fx fy ...]" (tab-separated, %.12E).  The run is cut into
 *                          lbm_gpu_run calls at multiples of k, which changes no output bit; after
 *                          LBM_RESTART the file holds the samples after the restart step
 *   LBM_FORCE_BOXES="x0,y0,x1,y1;..."   the boxes of the force (half-open global cell ranges; a
 *                          solid cell counts in every box that holds it); default: the whole grid
 */
#define _POSIX_C_SOURCE 200809L
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/time.h>

#include "lbm_gpu.h"
#include "lbm_io.h"

#define FINALSTATEFILE "final_state.dat"
#define AVVELSFILE "av_vels.dat"
#define FORCESFILE "forces.dat"

static void usage(const char* exe)
{
  fprintf(stderr, "Usage: %s <paramfile> <obstaclefile>\n", exe);
  exit(EXIT_FAILURE);
}

static double wtime(void)
{
  struct timeval t;
  gettimeofday(&t, NULL);
  return t.tv_sec + (t.tv_usec / 1000000.0);
}

#define GPU(call)                                                       \
  do {                                                                  \
    if ((call) != 0) die(lbm_gpu_last_error(), __LINE__, __FILE__);     \
  } while (0)

/* the lattice side of a checkpoint (lbm_io.c streams the file a block of rows at a time) */
static void save_rows_cb(void* gpu, long long row0, long long nrows, void* buf)
{
  GPU(lbm_gpu_save_rows((lbm_gpu*)gpu, row0, nrows, buf));
}

static void load_rows_cb(void* gpu, long long row0, long long nrows, void* buf)
{
  GPU(lbm_gpu_load_rows((lbm_gpu*)gpu, row0, nrows, buf));
}

/* one block of checkpoint rows, page-locked where the library can give it */
static void* ckpt_buffer(const lbm_ckpt_header* h, int* pinned)
{
  const size_t rec = h->kind == LBM_CKPT_F64 ? 72 : h->kind == LBM_CKPT_F16 ? 18 : 36;
  const size_t bytes = (size_t)lbm_ckpt_block_rows(h) * (size_t)h->nx * rec;
  void* p = NULL;
  *pinned = lbm_gpu_host_alloc(bytes, &p) == 0;
  if (!*pinned) p = malloc(bytes);
  if (p == NULL) die("cannot allocate memory for checkpoint rows", __LINE__, __FILE__);
  return p;
}

static void write_checkpoint(const char* path, lbm_gpu* gpu, lbm_ckpt_header* h, int steps_done, const void* av_vels)
{
  unsigned long long checksum = 0;
  GPU(lbm_gpu_digest(gpu, NULL, &checksum));
  h->steps_done = steps_done;
  h->checksum = checksum;
  int pinned;
  void* buf = ckpt_buffer(h, &pinned);
  lbm_write_checkpoint(path, h, av_vels, save_rows_cb, gpu, buf);
  if (pinned) lbm_gpu_host_free(buf);
  else free(buf);
}

/* one line of forces.dat: the force on each box at state t */
static void sample_force(lbm_gpu* gpu, FILE* fp, long long t, int n_boxes, const int* boxes, double* force)
{
  GPU(lbm_gpu_obstacle_force(gpu, n_boxes, boxes, force));
  lbm_write_force_line(fp, t, n_boxes, force);
}

static int env_flag(const char* name)
{
  const char* v = getenv(name);
  return v != NULL && v[0] != '\0' && strcmp(v, "0") != 0;
}

int main(int argc, char* argv[])
{
  if (argc != 3) usage(argv[0]);
  const char* paramfile = argv[1];
  const char* obstaclefile = argv[2];

  const int f64 = getenv("LBM_PRECISION") != NULL && strcmp(getenv("LBM_PRECISION"), "f64") == 0;
  const int n_gpus = getenv("LBM_GPUS") ? atoi(getenv("LBM_GPUS")) : 1;
  unsigned flags = LBM_GPU_OBST_BITS;
  if (getenv("LBM_PRECISION") != NULL && strcmp(getenv("LBM_PRECISION"), "f16") == 0) flags |= LBM_GPU_STORE_F16;
  if (env_flag("LBM_STRICT")) flags |= LBM_GPU_STRICT;
  const char* kv = getenv("LBM_KERNEL");
  if (kv != NULL) {
    if (strcmp(kv, "scalar") == 0) flags |= LBM_GPU_KERNEL_SCALAR;
    else if (strcmp(kv, "vec4") == 0) flags |= LBM_GPU_KERNEL_VEC4;
    else if (strcmp(kv, "persistent") == 0) flags |= LBM_GPU_KERNEL_PERSISTENT;
    else if (strcmp(kv, "tma") == 0) flags |= LBM_GPU_KERNEL_TMA;
    else if (strcmp(kv, "cluster") == 0) flags |= LBM_GPU_KERNEL_CLUSTER;
    else if (strcmp(kv, "tb2") == 0) flags |= LBM_GPU_KERNEL_TB2;
    else if (strcmp(kv, "tb3") == 0) flags |= LBM_GPU_KERNEL_TB3;
    else if (strcmp(kv, "pairs") == 0) flags |= LBM_GPU_KERNEL_PAIRS;
    else die("LBM_KERNEL must be scalar, vec4, persistent, tma, cluster, tb2, tb3 or pairs", __LINE__, __FILE__);
  }

  const char* ckpt_path = getenv("LBM_CHECKPOINT");
  const char* restart_path = getenv("LBM_RESTART");
  if (ckpt_path != NULL && ckpt_path[0] == '\0') ckpt_path = NULL;
  if (restart_path != NULL && restart_path[0] == '\0') restart_path = NULL;
  long long every = 0;
  if (getenv("LBM_CHECKPOINT_EVERY") != NULL) {
    char* end = NULL;
    every = strtoll(getenv("LBM_CHECKPOINT_EVERY"), &end, 10);
    if (end == getenv("LBM_CHECKPOINT_EVERY") || *end != '\0' || every < 1)
      die("LBM_CHECKPOINT_EVERY must be a positive number of steps", __LINE__, __FILE__);
    if (ckpt_path == NULL) die("LBM_CHECKPOINT_EVERY needs LBM_CHECKPOINT=<path>", __LINE__, __FILE__);
  }
  const long long force_every = getenv("LBM_FORCE_EVERY") != NULL ? lbm_parse_force_every(getenv("LBM_FORCE_EVERY")) : 0;
  if (getenv("LBM_FORCE_BOXES") != NULL && force_every == 0)
    die("LBM_FORCE_BOXES needs LBM_FORCE_EVERY=<k>", __LINE__, __FILE__);

  /* Total/init time starts here: load values from file, build the device lattice */
  const double tot_tic = wtime();
  const double init_tic = tot_tic;

  lbm_param params;
  lbm_param_f64 params_d;
  lbm_read_params(paramfile, &params, &params_d);
  const int nx = params.nx, ny = params.ny, iters = params.maxIters;
  uint32_t* obstacle_bits = lbm_read_obstacle_bits(obstaclefile, nx, ny);

  /* the boxes of the force time series: the whole grid unless LBM_FORCE_BOXES names them */
  static int force_boxes[4 * LBM_FORCE_MAX_BOXES];
  static double force[2 * LBM_FORCE_MAX_BOXES];
  int n_boxes = 1;
  force_boxes[2] = nx;
  force_boxes[3] = ny;
  if (getenv("LBM_FORCE_BOXES") != NULL) n_boxes = lbm_parse_force_boxes(getenv("LBM_FORCE_BOXES"), nx, ny, force_boxes);

  /* a record of the av. velocity computed for each timestep (d2q9-bgk.c:2866) */
  double* av_vels = (double*)malloc(sizeof(double) * (size_t)(iters > 0 ? iters : 1));
  float* av_vels_f = (float*)malloc(sizeof(float) * (size_t)(iters > 0 ? iters : 1));
  if (av_vels == NULL || av_vels_f == NULL) die("cannot allocate memory for av_vels", __LINE__, __FILE__);

  /* a checkpoint is checked against this run's inputs before the GPU is touched */
  lbm_ckpt_header ckpt;
  FILE* restart_fp = NULL;
  lbm_ckpt_header restart_hdr;
  int t0 = 0;
  if (ckpt_path != NULL || restart_path != NULL) {
    const uint32_t kind = f64 ? LBM_CKPT_F64 : (flags & LBM_GPU_STORE_F16) ? LBM_CKPT_F16 : LBM_CKPT_F32;
    lbm_ckpt_header_init(&ckpt, kind, (flags & LBM_GPU_STRICT) != 0, &params, &params_d,
                         lbm_obstacle_hash(obstacle_bits, nx, ny));
  }
  if (restart_path != NULL) {
    restart_fp = lbm_open_checkpoint(restart_path, &ckpt, iters, &restart_hdr);
    t0 = (int)restart_hdr.steps_done;
  }

  /* the rest-state lattice (d2q9-bgk.c:2802-2823) is generated on the device */
  lbm_gpu* gpu = NULL;
  if (f64) GPU(lbm_gpu_create_f64(&params_d, NULL, obstacle_bits, n_gpus, NULL, flags, &gpu));
  else GPU(lbm_gpu_create(&params, NULL, obstacle_bits, n_gpus, NULL, flags, &gpu));
  if (restart_fp != NULL) {      /* ... or the checkpoint's lattice and av_vels replace it */
    int pinned;
    void* buf = ckpt_buffer(&restart_hdr, &pinned);
    lbm_read_checkpoint(restart_fp, &restart_hdr, f64 ? (void*)av_vels : (void*)av_vels_f, load_rows_cb, gpu, buf);
    if (pinned) lbm_gpu_host_free(buf);
    else free(buf);
    if (!f64)
      for (int t = 0; t < t0; t++) av_vels[t] = av_vels_f[t];
    unsigned long long checksum = 0;
    GPU(lbm_gpu_digest(gpu, NULL, &checksum));
    if (checksum != restart_hdr.checksum)
      die("checkpoint lattice checksum differs from the one in its header: the file is corrupt", __LINE__, __FILE__);
  }

  /* Init time stops here, compute time starts */
  const double init_toc = wtime();
  const double comp_tic = init_toc;

  double ckpt_secs = 0.0;        /* checkpoint writes and force samples, not counted as compute time */
  FILE* forces_fp = NULL;
  if (force_every > 0) {
    forces_fp = fopen(FORCESFILE, "w");
    if (forces_fp == NULL) die("could not open file " FORCESFILE, __LINE__, __FILE__);
  }
  if (env_flag("LBM_DEBUG")) {
    for (int tt = t0; tt < iters; tt++) {
      double density;
      if (f64) {
        GPU(lbm_gpu_run_f64(gpu, 1, &av_vels[tt]));
      } else {
        GPU(lbm_gpu_run(gpu, 1, &av_vels_f[tt]));
        av_vels[tt] = av_vels_f[tt];
      }
      GPU(lbm_gpu_digest(gpu, &density, NULL));
      printf("==timestep: %d==\n", tt);
      printf("av velocity: %.12E\n", av_vels[tt]);
      printf("tot density: %.12E\n", density);
      if (force_every > 0 && (tt + 1) % force_every == 0) sample_force(gpu, forces_fp, tt + 1, n_boxes, force_boxes, force);
    }
  } else {
    /* steps [t0, iters), cut at the multiples of LBM_CHECKPOINT_EVERY and of LBM_FORCE_EVERY */
    for (int t = t0; t < iters;) {
      long long next = iters;
      if (every > 0 && ((long long)t / every + 1) * every < next) next = ((long long)t / every + 1) * every;
      if (force_every > 0 && ((long long)t / force_every + 1) * force_every < next)
        next = ((long long)t / force_every + 1) * force_every;
      if (f64) GPU(lbm_gpu_run_f64(gpu, (int)next - t, av_vels + t));
      else GPU(lbm_gpu_run(gpu, (int)next - t, av_vels_f + t));
      t = (int)next;
      if (force_every > 0 && t % force_every == 0) {
        const double tic = wtime();
        sample_force(gpu, forces_fp, t, n_boxes, force_boxes, force);
        ckpt_secs += wtime() - tic;
      }
      if (every > 0 && t < iters && t % every == 0) {
        const double tic = wtime();
        write_checkpoint(ckpt_path, gpu, &ckpt, t, f64 ? (const void*)av_vels : (const void*)av_vels_f);
        ckpt_secs += wtime() - tic;
      }
    }
    if (!f64)
      for (int t = 0; t < iters; t++) av_vels[t] = av_vels_f[t];
  }

  /* Compute time stops here (lbm_gpu_run returns with the device idle), collate time
   * starts: bring the results of all GPUs back to the host */
  const double comp_end = wtime();
  const double comp_toc = comp_end - ckpt_secs;
  const double col_tic = comp_end;

  double reynolds;
  if (f64) {
    double av;
    GPU(lbm_gpu_av_velocity_f64(gpu, &av));
    const double viscosity = 1.0 / 6.0 * (2.0 / params_d.omega - 1.0);
    reynolds = av * params_d.reynolds_dim / viscosity;
  } else {
    float av;
    GPU(lbm_gpu_av_velocity(gpu, &av));
    const float viscosity = 1.f / 6.f * (2.f / params.omega - 1.f);      /* d2q9-bgk.c:2895 */
    reynolds = av * params.reynolds_dim / viscosity;
  }

  const double col_toc = wtime();
  const double tot_toc = col_toc - ckpt_secs;

  /* write final values and free memory */
  printf("==done==\n");
  printf("Reynolds number:\t\t%.12E\n", reynolds);
  printf("Elapsed Init time:\t\t\t%.6lf (s)\n", init_toc - init_tic);
  printf("Elapsed Compute time:\t\t\t%.6lf (s)\n", comp_toc - comp_tic);
  printf("Elapsed Collate time:\t\t\t%.6lf (s)\n", col_toc - col_tic);
  printf("Elapsed Total time:\t\t\t%.6lf (s)\n", tot_toc - tot_tic);

  if (env_flag("LBM_REPORT") && strcmp(getenv("LBM_REPORT"), "json") == 0) {
    lbm_gpu_info info;
    GPU(lbm_gpu_get_info(gpu, &info));
    const double updates = (double)nx * (double)ny * (double)iters;
    const double dev_s = info.last_run_device_ms * 1e-3;
    printf("{\"nx\": %d, \"ny\": %d, \"steps\": %d, \"gpus\": %d, \"precision\": \"%s\", \"kernel\": %d, "
           "\"init_s\": %.6f, \"compute_s\": %.6f, \"collate_s\": %.6f, \"device_compute_s\": %.6f, "
           "\"mlups_device\": %.1f, \"gbs_72B\": %.1f, \"free_cells\": %lld, \"kernel_launches\": %lld}\n",
           nx, ny, iters, n_gpus, f64 ? "f64" : (flags & LBM_GPU_STORE_F16) ? "f16" : "f32", info.kernel, init_toc - init_tic, comp_toc - comp_tic,
           col_toc - col_tic, dev_s, dev_s > 0 ? updates / dev_s / 1e6 : 0.0, dev_s > 0 ? updates * 72.0 / dev_s / 1e9 : 0.0,
           info.free_cells, info.kernel_launches);
  } else if (env_flag("LBM_REPORT")) {
    lbm_gpu_info info;
    GPU(lbm_gpu_get_info(gpu, &info));
    const double updates = (double)nx * (double)ny * (double)iters;
    const double dev_s = info.last_run_device_ms * 1e-3;
    printf("GPUs:\t\t\t\t\t%d\n", n_gpus);
    printf("Device compute time:\t\t\t%.6lf (s)\n", dev_s);
    if (dev_s > 0.0) {
      printf("MLUPS (device time):\t\t\t%.1f\n", updates / dev_s / 1e6);
      printf("Algorithmic GB/s (72 B/update):\t\t%.1f\n", updates * 72.0 / dev_s / 1e9);
    }
    printf("MLUPS (wall compute time):\t\t%.1f\n", updates / (comp_toc - comp_tic) / 1e6);
  }

  if (ckpt_path != NULL) {
    const double tic = wtime();
    write_checkpoint(ckpt_path, gpu, &ckpt, iters, f64 ? (const void*)av_vels : (const void*)av_vels_f);
    ckpt_secs += wtime() - tic;
    printf("Elapsed Checkpoint time:\t\t%.6lf (s)\n", ckpt_secs);
  }

  /* write_values (d2q9-bgk.c:2918-2999): the per-cell fields are computed on the GPU
   * and streamed back a block of rows at a time */
  if (!env_flag("LBM_SKIP_FINAL_STATE")) {
    FILE* fp = fopen(FINALSTATEFILE, "w");
    if (fp == NULL) die("could not open file output file", __LINE__, __FILE__);
    static char big[1 << 22];
    setvbuf(fp, big, _IOFBF, sizeof big);
    long long chunk = (2LL << 20) / nx;       /* rows per block: about 2 M cells (~200 MB of text) */
    if (chunk < 1) chunk = 1;
    if (chunk > ny) chunk = ny;
    const size_t n = (size_t)chunk * (size_t)nx;
    double* d[4];
    float* f[4];
    for (int i = 0; i < 4; i++) {
      d[i] = (double*)malloc(n * sizeof(double));
      f[i] = (float*)malloc(n * sizeof(float));
      if (d[i] == NULL || f[i] == NULL) die("cannot allocate memory for output rows", __LINE__, __FILE__);
    }
    for (long long r0 = 0; r0 < ny; r0 += chunk) {
      const long long nr = (r0 + chunk <= ny) ? chunk : ny - r0;
      if (f64) {
        GPU(lbm_gpu_final_fields_f64(gpu, r0, nr, d[0], d[1], d[2], d[3]));
      } else {
        GPU(lbm_gpu_final_fields(gpu, r0, nr, f[0], f[1], f[2], f[3]));
        for (int i = 0; i < 4; i++)
          for (size_t k = 0; k < (size_t)nr * (size_t)nx; k++) d[i][k] = f[i][k];
      }
      lbm_write_final_state_rows(fp, nx, r0, nr, d[0], d[1], d[2], d[3], obstacle_bits);
    }
    for (int i = 0; i < 4; i++) { free(d[i]); free(f[i]); }
    fclose(fp);
  }
  lbm_write_av_vels(AVVELSFILE, iters, av_vels);
  if (forces_fp != NULL && fclose(forces_fp) != 0) die("could not write " FORCESFILE, __LINE__, __FILE__);

  lbm_gpu_destroy(gpu);
  free(av_vels);
  free(av_vels_f);
  free(obstacle_bits);
  return EXIT_SUCCESS;
}
