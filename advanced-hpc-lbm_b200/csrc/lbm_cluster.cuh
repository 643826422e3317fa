// lbm_cluster.cuh -- K6: the whole run of a tiny lattice inside ONE thread-block cluster.
//
// The reference's two smallest shipped inputs (128x128, 128x256: 0.6 / 1.2 MB per buffer)
// fit, double-buffered, in the shared memory of 16 SMs.  K6 keeps the lattice there for all
// timesteps: every CTA of the cluster owns a band of rows in its shared memory, pulls its
// neighbours' edge rows through distributed shared memory (DSMEM), and ONE cluster barrier
// per step replaces K5's L2 round trips and grid barrier.  One launch per lbm_gpu_run.
//
// Step t inside the kernel (same per-cell arithmetic as every other kernel -- cell_update,
// cell_accelerate -- so the results are bit-identical):
//   every thread pulls the nine values of each of its cells (default build: of each of its
//   x-aligned quads of cells) from buffer `cur` (own band, or the band of the CTA
//   below/above via DSMEM), collides, adds |u| to the step's sum and
//   stores the result into its own band of buffer `cur ^ 1`; row ny-2 is stored WITH the
//   next step's accelerate_flow applied (d2q9-bgk.c:229-260), except after the last step;
//   cluster barrier; the buffers swap roles.
// Before the first step the band is loaded from the global lattice (row ny-2 accelerated on
// the way in); after the last one it is written to the other global buffer.
#pragma once
#include <cooperative_groups.h>

#include "lbm_kernels.cuh"

namespace lbm {

namespace cg = cooperative_groups;

#define LBM_CLUSTER_THREADS 1024

struct ClusterArgs {
  const float* src;            // global lattice buffer holding the current state
  float* dst;                  // global lattice buffer that receives the final state
  const uint32_t* mask;
  unsigned long long* av;      // n_steps x (LBM_AV_STRIDE * LBM_AV_SLOTS) words
  long long plane_stride;
  int nx, ny, pitch, mask_pitch;
  int rows_per_cta;            // band height (the last CTAs may hold fewer rows, or none)
  int n_steps;
  float omega, aw1, aw2;
};

template <bool STRICT>
__global__ void __launch_bounds__(LBM_CLUSTER_THREADS, 1)
lbm_steps_cluster(const __grid_constant__ ClusterArgs a) {
  extern __shared__ __align__(16) float band[];          // [2 buffers][9 planes][rows_per_cta][nx]
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int tid = threadIdx.x;
  const int nx = a.nx, ny = a.ny, R = a.rows_per_cta;
  const int y0 = rank * R;
  const int my_rows = max(0, min(R, ny - y0));
  const int my_cells = my_rows * nx;
  const int plane = R * nx;                              // floats per plane in shared memory
  const int buffer = 9 * plane;                          // floats per buffer
  const int accel_y = ny - 2;

  // neighbour bands: the CTAs that hold row y0-1 and row y0+my_rows (periodic in y)
  const int y_below = (y0 == 0) ? ny - 1 : y0 - 1;
  const int y_above = (y0 + my_rows >= ny) ? 0 : y0 + my_rows;
  const int rank_below = min(y_below / R, (int)cluster.num_blocks() - 1);
  const int rank_above = min(y_above / R, (int)cluster.num_blocks() - 1);
  const float* below = cluster.map_shared_rank(band, (unsigned)rank_below) + (y_below - rank_below * R) * nx;
  const float* above = cluster.map_shared_rank(band, (unsigned)rank_above) + (y_above - rank_above * R) * nx;

  // ---- load the band into buffer 0 (row ny-2 gets the first step's accelerate on the way in)
  for (int c = tid; c < my_cells; c += LBM_CLUSTER_THREADS) {
    const int yl = c / nx, x = c - yl * nx, y = y0 + yl;
    const bool obst = (a.mask[(long long)y * a.mask_pitch + (x >> 5)] >> (x & 31)) & 1u;
    float f[9];
#pragma unroll
    for (int k = 0; k < 9; k++) f[k] = a.src[k * a.plane_stride + (long long)y * a.pitch + x];
    if (y == accel_y && a.n_steps > 0)
      cell_accelerate<float, true>(f[1], f[3], f[5], f[6], f[7], f[8], obst, a.aw1, a.aw2);
#pragma unroll
    for (int k = 0; k < 9; k++) band[k * plane + c] = f[k];
  }
  cluster.sync();

  int cur = 0;
  for (int t = 0; t < a.n_steps; t++) {
    const float* rd = band + cur * buffer;
    float* wr = band + (cur ^ 1) * buffer;
    const float* rd_below = below + cur * buffer;
    const float* rd_above = above + cur * buffer;
    unsigned long long* av_step = a.av + (size_t)t * (LBM_AV_STRIDE * LBM_AV_SLOTS);
    const bool last_step = (t == a.n_steps - 1);
    // one cell: collide, store into buffer `wr`, return |u| (0 for an obstacle cell)
    auto update = [&](const int yl, const int x) -> float {
      const int c = yl * nx + x, y = y0 + yl;
      const int xw = (x == 0) ? nx - 1 : x - 1;
      const int xe = (x + 1 == nx) ? 0 : x + 1;
      const float* c_row = rd + yl * nx;
      const float* s_row = (yl == 0) ? rd_below : rd + (yl - 1) * nx;
      const float* n_row = (yl == my_rows - 1) ? rd_above : rd + (yl + 1) * nx;
      const bool obst = (a.mask[(long long)y * a.mask_pitch + (x >> 5)] >> (x & 31)) & 1u;
      float p[9], o[9];
      p[0] = c_row[0 * plane + x];
      p[1] = c_row[1 * plane + xw];
      p[3] = c_row[3 * plane + xe];
      p[2] = s_row[2 * plane + x];
      p[5] = s_row[5 * plane + xw];
      p[6] = s_row[6 * plane + xe];
      p[4] = n_row[4 * plane + x];
      p[7] = n_row[7 * plane + xe];
      p[8] = n_row[8 * plane + xw];
      const float s = cell_update<float, STRICT>(p, obst, a.omega, o);
      if (y == accel_y && !last_step)
        cell_accelerate<float, true>(o[1], o[3], o[5], o[6], o[7], o[8], obst, a.aw1, a.aw2);
#pragma unroll
      for (int k = 0; k < 9; k++) wr[k * plane + c] = o[k];
      return s;
    };
    unsigned long long q = 0ULL;
    bool bad = false;
    if (STRICT) {
      for (int c = tid; c < my_cells; c += LBM_CLUSTER_THREADS) {
        const int yl = c / nx;
        const float s = update(yl, c - yl * nx);
        q += to_fixed(s);
        bad |= !(s < (float)LBM_SPEED_LIMIT);
      }
    } else {
      // the default build adds |u| over the x-aligned quads of the other kernels, in their
      // float order (quad_sum_fixed), so that every kernel gives the same av_vels bits
      const int quads_x = (nx + 3) / 4;
      for (int i = tid; i < my_rows * quads_x; i += LBM_CLUSTER_THREADS) {
        const int yl = i / quads_x, x0 = 4 * (i - yl * quads_x);
        float s[4];
#pragma unroll
        for (int j = 0; j < 4; j++) s[j] = (x0 + j < nx) ? update(yl, x0 + j) : 0.0f;
        bool b;
        q += quad_sum_fixed<float>(s[0], s[1], s[2], s[3], b);
        bad |= b;
      }
    }
    if (bad) atomicOr(av_step + 1, LBM_NONFINITE_MARK);
    block_accumulate(q, av_step);
    cluster.sync();
    cur ^= 1;
  }

  // ---- write the final (un-accelerated) state to the other global buffer ---------------------
  if (a.n_steps > 0) {
    const float* rd = band + cur * buffer;
    for (int c = tid; c < my_cells; c += LBM_CLUSTER_THREADS) {
      const int yl = c / nx, x = c - yl * nx, y = y0 + yl;
#pragma unroll
      for (int k = 0; k < 9; k++) a.dst[k * a.plane_stride + (long long)y * a.pitch + x] = rd[k * plane + c];
    }
  }
}

}  // namespace lbm
