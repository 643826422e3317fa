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
 */
#define _POSIX_C_SOURCE 200809L
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/time.h>

#include "lbm_gpu.h"
#include "lbm_io.h"

#define FINALSTATEFILE "final_state.dat"
#define AVVELSFILE "av_vels.dat"

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

  /* Total/init time starts here: load values from file, build the device lattice */
  const double tot_tic = wtime();
  const double init_tic = tot_tic;

  lbm_param params;
  lbm_param_f64 params_d;
  lbm_read_params(paramfile, &params, &params_d);
  const int nx = params.nx, ny = params.ny, iters = params.maxIters;
  uint32_t* obstacle_bits = lbm_read_obstacle_bits(obstaclefile, nx, ny);

  /* a record of the av. velocity computed for each timestep (d2q9-bgk.c:2866) */
  double* av_vels = (double*)malloc(sizeof(double) * (size_t)(iters > 0 ? iters : 1));
  float* av_vels_f = (float*)malloc(sizeof(float) * (size_t)(iters > 0 ? iters : 1));
  if (av_vels == NULL || av_vels_f == NULL) die("cannot allocate memory for av_vels", __LINE__, __FILE__);

  /* the rest-state lattice (d2q9-bgk.c:2802-2823) is generated on the device */
  lbm_gpu* gpu = NULL;
  if (f64) GPU(lbm_gpu_create_f64(&params_d, NULL, obstacle_bits, n_gpus, NULL, flags, &gpu));
  else GPU(lbm_gpu_create(&params, NULL, obstacle_bits, n_gpus, NULL, flags, &gpu));

  /* Init time stops here, compute time starts */
  const double init_toc = wtime();
  const double comp_tic = init_toc;

  if (env_flag("LBM_DEBUG")) {
    for (int tt = 0; tt < iters; tt++) {
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
    }
  } else if (f64) {
    GPU(lbm_gpu_run_f64(gpu, iters, av_vels));
  } else {
    GPU(lbm_gpu_run(gpu, iters, av_vels_f));
    for (int t = 0; t < iters; t++) av_vels[t] = av_vels_f[t];
  }

  /* Compute time stops here (lbm_gpu_run returns with the device idle), collate time
   * starts: bring the results of all GPUs back to the host */
  const double comp_toc = wtime();
  const double col_tic = comp_toc;

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
  const double tot_toc = col_toc;

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

  lbm_gpu_destroy(gpu);
  free(av_vels);
  free(av_vels_f);
  free(obstacle_bits);
  return EXIT_SUCCESS;
}
