// lbm_pairs.cuh -- K9: the whole run of a SMALL lattice in one cooperative launch, two
// timesteps per grid barrier (fp32, single GPU, nx a multiple of 4 and <= 256).
//
// The reference's smallest shipped inputs (128x128, 128x256, 256x256) occupy a fraction of
// one SM's worth of work per timestep: what a step costs is latency -- one grid barrier
// (two L2 round trips) plus one dependent chain of L2 loads, arithmetic and stores.  The
// persistent kernel K5 pays that per TIMESTEP.  K9 pays it per PAIR of timesteps:
//
//   a block owns `tile_rows` consecutive rows over the full width; thread row ty works on
//   lattice row R0 - 1 + ty (periodic), so the block holds its rows plus one on each side:
//     phase 1  every thread row pulls its quad's nine values straight from L2 (the loads of
//              K1a/K5: vec4_pull), collides, and leaves the result of sub-step 1 in shared
//              memory -- with the next step's accelerate_flow applied if the row is ny-2
//              (d2q9-bgk.c:229-260: accelerate, then stream);
//     phase 2  the block's own rows pull sub-step 1 from shared memory (periodic in x inside
//              the row), collide and store sub-step 2 to the other lattice buffer, keeping
//              the side row and the ghost rows up to date exactly like K1a;
//   then the grid barrier, and the buffers swap roles.  The halo rows of sub-step 1 are
//   computed twice (by the two blocks that need them): on a grid this small arithmetic is
//   free, round trips are not.
//
// An odd last timestep is left to K1a (the lattice, side row and ghost rows are in the
// state every other kernel expects).  Same per-cell arithmetic as every other kernel.
#pragma once
#include "lbm_kernels.cuh"

namespace lbm {

#define LBM_PAIRS_MAX_NX 256
#define LBM_PAIRS_MAX_TILE_ROWS 4
#define LBM_PAIRS_MAX_THREADS ((LBM_PAIRS_MAX_NX / 4) * (LBM_PAIRS_MAX_TILE_ROWS + 2))

struct PairsArgs {
  StepArgs<float> s;           // geometry and constants; the per-pass pointers are set inside the kernel
  float* lattice[2];
  float* side[2];
  float* window;               // own window: ghost rows at ghost_offset(pitch, parity, direction)
  unsigned long long* av;      // 2 x n_pairs steps x LBM_AV_SLOTS x LBM_AV_STRIDE words
  unsigned long long* barrier; // zeroed before the launch
  int first_parity;            // buffer index read by the first pair
  int n_pairs;
  int tile_rows;               // rows owned by a block; blockDim = (round_up(nx / 4, 32), tile_rows + 2)
};

template <bool STRICT>
__global__ void __launch_bounds__(LBM_PAIRS_MAX_THREADS, 1)
lbm_steps_pairs(const __grid_constant__ PairsArgs pa) {
  extern __shared__ __align__(16) float pairs_tile[];     // [tile_rows + 2][9][nx]: sub-step 1 of the block's rows
  StepArgs<float> a = pa.s;
  const int nx = a.nx, pitch = a.pitch, H = pa.tile_rows;
  const int ty = threadIdx.y;
  const int x0 = 4 * (int)threadIdx.x;
  const bool col_ok = x0 < nx;
  const int xc = col_ok ? x0 : 0;
  const int R0 = (int)blockIdx.x * H;
  int r = R0 - 1 + ty;                                    // the lattice row of this thread row, periodic in y
  if (r < 0) r += a.rows;
  if (r >= a.rows) r -= a.rows;
  const bool own = col_ok && ty >= 1 && ty <= H && (R0 + ty - 1 < a.rows);   // a row this block stores
  const QuadConsts<float, STRICT> qc(a.omega);
  float* mine = pairs_tile + (size_t)(ty * 9) * nx;
  const long long PS = a.plane_stride;

  for (int p = 0; p < pa.n_pairs; p++) {
    const int src = (pa.first_parity + p) & 1, dst = src ^ 1;
    a.src = pa.lattice[src];
    a.dst = pa.lattice[dst];
    a.side_src = pa.side[src];
    a.side_dst = pa.side[dst];
    a.ghost_s = pa.window + ghost_offset(pitch, src, 0);
    a.ghost_n = pa.window + ghost_offset(pitch, src, 1);
    a.push_up = pa.window + ghost_offset(pitch, dst, 0);
    a.push_dn = pa.window + ghost_offset(pitch, dst, 1);
    unsigned long long* av1 = pa.av + (size_t)(2 * p) * (LBM_AV_STRIDE * LBM_AV_SLOTS);
    unsigned long long* av2 = av1 + LBM_AV_STRIDE * LBM_AV_SLOTS;

    // ---- phase 1: sub-step 1 of row r into shared memory --------------------------------
    float in[4][9], out[4][9];
    uint32_t mbits, obits;
    vec4_pull<float, true>(a, r, xc, in, mbits, obits);
    bool bad;
    unsigned long long q1 = quad_update<float, STRICT>(in, obits, qc, out, bad);
    if (!own) q1 = 0ULL;
    if (own && bad) atomicOr(av1 + 1, LBM_NONFINITE_MARK);
    if (r == a.accel_row) {
#pragma unroll
      for (int j = 0; j < 4; j++)
        cell_accelerate<float, STRICT>(out[j][1], out[j][3], out[j][5], out[j][6], out[j][7], out[j][8],
                                       (mbits >> j) & 1u, a.aw1, a.aw2);
    }
    if (col_ok) {
#pragma unroll
      for (int k = 0; k < 9; k++)
        *reinterpret_cast<float4*>(mine + k * nx + x0) = make_float4(out[0][k], out[1][k], out[2][k], out[3][k]);
    }
    __syncthreads();

    // ---- phase 2: sub-step 2 of the block's own rows, pulled from shared memory ------------
    unsigned long long q2 = 0ULL;
    if (own) {
      const float* c = mine;                 // row r
      const float* s = mine - 9 * nx;        // row r - 1
      const float* n = mine + 9 * nx;        // row r + 1
      const int xw = (x0 == 0) ? nx - 1 : x0 - 1;
      const int xe = (x0 + 4 >= nx) ? 0 : x0 + 4;
#define LBM_PAIRS_SAME(row, k)                                                                      \
  { const float4 v = *reinterpret_cast<const float4*>((row) + (k) * nx + x0);                        \
    in[0][k] = v.x; in[1][k] = v.y; in[2][k] = v.z; in[3][k] = v.w; }
#define LBM_PAIRS_WEST(row, k)                                                                      \
  { const float4 v = *reinterpret_cast<const float4*>((row) + (k) * nx + x0);                        \
    in[0][k] = (row)[(k) * nx + xw]; in[1][k] = v.x; in[2][k] = v.y; in[3][k] = v.z; }
#define LBM_PAIRS_EAST(row, k)                                                                      \
  { const float4 v = *reinterpret_cast<const float4*>((row) + (k) * nx + x0);                        \
    in[0][k] = v.y; in[1][k] = v.z; in[2][k] = v.w; in[3][k] = (row)[(k) * nx + xe]; }
      LBM_PAIRS_SAME(c, 0) LBM_PAIRS_WEST(c, 1) LBM_PAIRS_EAST(c, 3)
      LBM_PAIRS_SAME(s, 2) LBM_PAIRS_WEST(s, 5) LBM_PAIRS_EAST(s, 6)
      LBM_PAIRS_SAME(n, 4) LBM_PAIRS_EAST(n, 7) LBM_PAIRS_WEST(n, 8)
#undef LBM_PAIRS_SAME
#undef LBM_PAIRS_WEST
#undef LBM_PAIRS_EAST
      q2 = quad_update<float, STRICT>(in, obits, qc, out, bad);
      if (bad) atomicOr(av2 + 1, LBM_NONFINITE_MARK);
      float* d = a.dst + (long long)r * pitch + x0;
#pragma unroll
      for (int k = 0; k < 9; k++)
        *reinterpret_cast<float4*>(d + k * PS) = make_float4(out[0][k], out[1][k], out[2][k], out[3][k]);
      const bool first = (r == 0), last = (r == a.rows - 1), cA = (r == a.accel_row);
      if (first | last | cA) {
        if (cA) {
#pragma unroll
          for (int j = 0; j < 4; j++)
            cell_accelerate<float, STRICT>(out[j][1], out[j][3], out[j][5], out[j][6], out[j][7], out[j][8],
                                           (mbits >> j) & 1u, a.aw1, a.aw2);
          const int ks[6] = {1, 3, 5, 6, 7, 8};
#pragma unroll
          for (int i = 0; i < 6; i++)
            *reinterpret_cast<float4*>(a.side_dst + (long long)i * pitch + x0) =
                make_float4(out[0][ks[i]], out[1][ks[i]], out[2][ks[i]], out[3][ks[i]]);
        }
#define LBM_PAIRS_PUSH(dstp, k)                                                                  \
  *reinterpret_cast<float4*>((dstp) + (long long)(k) * pitch + x0) = make_float4(out[0][k], out[1][k], out[2][k], out[3][k]);
        if (first) { LBM_PAIRS_PUSH(a.push_dn, 4) LBM_PAIRS_PUSH(a.push_dn, 7) LBM_PAIRS_PUSH(a.push_dn, 8) }
        if (last) { LBM_PAIRS_PUSH(a.push_up, 2) LBM_PAIRS_PUSH(a.push_up, 5) LBM_PAIRS_PUSH(a.push_up, 6) }
#undef LBM_PAIRS_PUSH
      }
    }
    warp_accumulate(q1, av1);
    warp_accumulate(q2, av2);
    grid_barrier(pa.barrier, (unsigned long long)gridDim.x * (unsigned long long)(p + 1));
  }
}

// ------------------------------------------------------------------------------------
// K11  lbm_steps_pairs_batch: K9 for MANY independent lattices of one shape in one launch
// (parameter sweeps).  blockIdx.y is the member; its pointers and constants come from a
// table in device memory, and its blocks meet at a barrier of its own (members never wait
// for each other).  Same scheme and per-cell code as K9, so each member gets K9's bits.
//
// What differs from K9 is the block shape.  K9 gives every lattice row of a tile (plus the
// two halo rows) a thread row of its own; with its ~166 registers per thread that leaves
// two 4-row blocks per SM, i.e. ~9 members of 128^2 on the whole GPU.  Here a block has
// `thread_rows` thread rows that loop over the tile: phase 1 over its tile_rows + 2 rows,
// phase 2 over its tile_rows owned rows.  Taller tiles then put the members' residency on
// shared memory (one tile of 16 rows at nx = 128 is 83 KB) rather than on registers, and
// recompute fewer halo rows.  thread_rows = tile_rows + 2 is K9's shape.
// ------------------------------------------------------------------------------------
struct BatchMember {
  float* lattice[2];
  float* side[2];
  float* window;               // own window: ghost rows at ghost_offset(pitch, parity, direction)
  const uint32_t* mask;
  unsigned long long* av;      // 2 x n_pairs steps x LBM_AV_SLOTS x LBM_AV_STRIDE words
  unsigned long long* barrier; // zeroed before the launch; target gridDim.x x (pair + 1)
  int first_parity;            // buffer index read by the member's first pair
  float omega, aw1, aw2;
};

struct BatchArgs {
  StepArgs<float> s;              // geometry shared by every member; pointers and constants are per member
  const BatchMember* members;     // gridDim.y entries, member blockIdx.y first
  int n_pairs;
  int tile_rows;                  // rows owned by a block
};

// register budget of K11: 384 threads x 1 block = up to 168 registers (measured against
// 256 x 2 = 128 registers with a few spills in profiles/r04_batch.md)
#ifndef LBM_BATCH_MAX_THREADS
#define LBM_BATCH_MAX_THREADS LBM_PAIRS_MAX_THREADS
#endif
#ifndef LBM_BATCH_MIN_BLOCKS
#define LBM_BATCH_MIN_BLOCKS 1
#endif

template <bool STRICT>
__global__ void __launch_bounds__(LBM_BATCH_MAX_THREADS, LBM_BATCH_MIN_BLOCKS)
lbm_steps_pairs_batch(const __grid_constant__ BatchArgs ba) {
  extern __shared__ __align__(16) float pairs_tile[];     // [tile_rows + 2][9][nx]: sub-step 1 of the block's rows
  // the member's entry, read once: the acquire of every barrier drops L1, and a table read
  // from L2 after each barrier put one more round trip on every pair (measured +18 % at 128^2)
  __shared__ BatchMember m;
  if (threadIdx.x == 0 && threadIdx.y == 0) m = ba.members[blockIdx.y];
  __syncthreads();
  StepArgs<float> a = ba.s;
  a.mask = m.mask;
  a.omega = m.omega;
  a.aw1 = m.aw1;
  a.aw2 = m.aw2;
  const int nx = a.nx, pitch = a.pitch, H = ba.tile_rows, T = (int)blockDim.y;
  const int ty = threadIdx.y;
  const int x0 = 4 * (int)threadIdx.x;
  const bool col_ok = x0 < nx;
  const int xc = col_ok ? x0 : 0;
  const int R0 = (int)blockIdx.x * H;
  const QuadConsts<float, STRICT> qc(a.omega);
  const long long PS = a.plane_stride;

  for (int p = 0; p < ba.n_pairs; p++) {
    const int src = (m.first_parity + p) & 1, dst = src ^ 1;
    a.src = m.lattice[src];
    a.dst = m.lattice[dst];
    a.side_src = m.side[src];
    a.side_dst = m.side[dst];
    a.ghost_s = m.window + ghost_offset(pitch, src, 0);
    a.ghost_n = m.window + ghost_offset(pitch, src, 1);
    a.push_up = m.window + ghost_offset(pitch, dst, 0);
    a.push_dn = m.window + ghost_offset(pitch, dst, 1);
    unsigned long long* av1 = m.av + (size_t)(2 * p) * (LBM_AV_STRIDE * LBM_AV_SLOTS);
    unsigned long long* av2 = av1 + LBM_AV_STRIDE * LBM_AV_SLOTS;
    float in[4][9], out[4][9];
    uint32_t mbits, obits;
    bool bad;

    // ---- phase 1: sub-step 1 of tile rows i = ty, ty + T, ... (lattice row R0 - 1 + i) ----
    unsigned long long q1 = 0ULL;
    for (int i = ty; i < H + 2; i += T) {
      int r = R0 - 1 + i;                                  // periodic in y
      if (r < 0) r += a.rows;
      if (r >= a.rows) r -= a.rows;
      const bool own = col_ok && i >= 1 && i <= H && (R0 + i - 1 < a.rows);
      vec4_pull<float, true>(a, r, xc, in, mbits, obits);
      const unsigned long long q = quad_update<float, STRICT>(in, obits, qc, out, bad);
      if (own) q1 += q;
      if (own && bad) atomicOr(av1 + 1, LBM_NONFINITE_MARK);
      if (r == a.accel_row) {
#pragma unroll
        for (int j = 0; j < 4; j++)
          cell_accelerate<float, STRICT>(out[j][1], out[j][3], out[j][5], out[j][6], out[j][7], out[j][8],
                                         (mbits >> j) & 1u, a.aw1, a.aw2);
      }
      if (col_ok) {
        float* mine = pairs_tile + (size_t)(i * 9) * nx;
#pragma unroll
        for (int k = 0; k < 9; k++)
          *reinterpret_cast<float4*>(mine + k * nx + x0) = make_float4(out[0][k], out[1][k], out[2][k], out[3][k]);
      }
    }
    __syncthreads();

    // ---- phase 2: sub-step 2 of owned tile rows i = 1 + ty, 1 + ty + T, ..., from shared memory ----
    unsigned long long q2 = 0ULL;
    for (int i = 1 + ty; i <= H; i += T) {
      const int r = R0 + i - 1;
      if (!col_ok || r >= a.rows) break;
      // nx is a multiple of 4: every cell of the quad is a lattice cell, the mask is the whole story
      mbits = obits = (a.mask[(long long)r * a.mask_pitch + (x0 >> 5)] >> (x0 & 31)) & 0xFu;
      const float* c = pairs_tile + (size_t)(i * 9) * nx;   // row r
      const float* s = c - 9 * nx;                          // row r - 1
      const float* n = c + 9 * nx;                          // row r + 1
      const int xw = (x0 == 0) ? nx - 1 : x0 - 1;
      const int xe = (x0 + 4 >= nx) ? 0 : x0 + 4;
#define LBM_PAIRS_SAME(row, k)                                                                      \
  { const float4 v = *reinterpret_cast<const float4*>((row) + (k) * nx + x0);                        \
    in[0][k] = v.x; in[1][k] = v.y; in[2][k] = v.z; in[3][k] = v.w; }
#define LBM_PAIRS_WEST(row, k)                                                                      \
  { const float4 v = *reinterpret_cast<const float4*>((row) + (k) * nx + x0);                        \
    in[0][k] = (row)[(k) * nx + xw]; in[1][k] = v.x; in[2][k] = v.y; in[3][k] = v.z; }
#define LBM_PAIRS_EAST(row, k)                                                                      \
  { const float4 v = *reinterpret_cast<const float4*>((row) + (k) * nx + x0);                        \
    in[0][k] = v.y; in[1][k] = v.z; in[2][k] = v.w; in[3][k] = (row)[(k) * nx + xe]; }
      LBM_PAIRS_SAME(c, 0) LBM_PAIRS_WEST(c, 1) LBM_PAIRS_EAST(c, 3)
      LBM_PAIRS_SAME(s, 2) LBM_PAIRS_WEST(s, 5) LBM_PAIRS_EAST(s, 6)
      LBM_PAIRS_SAME(n, 4) LBM_PAIRS_EAST(n, 7) LBM_PAIRS_WEST(n, 8)
#undef LBM_PAIRS_SAME
#undef LBM_PAIRS_WEST
#undef LBM_PAIRS_EAST
      q2 += quad_update<float, STRICT>(in, obits, qc, out, bad);
      if (bad) atomicOr(av2 + 1, LBM_NONFINITE_MARK);
      float* d = a.dst + (long long)r * pitch + x0;
#pragma unroll
      for (int k = 0; k < 9; k++)
        *reinterpret_cast<float4*>(d + k * PS) = make_float4(out[0][k], out[1][k], out[2][k], out[3][k]);
      const bool first = (r == 0), last = (r == a.rows - 1), cA = (r == a.accel_row);
      if (first | last | cA) {
        if (cA) {
#pragma unroll
          for (int j = 0; j < 4; j++)
            cell_accelerate<float, STRICT>(out[j][1], out[j][3], out[j][5], out[j][6], out[j][7], out[j][8],
                                           (mbits >> j) & 1u, a.aw1, a.aw2);
          const int ks[6] = {1, 3, 5, 6, 7, 8};
#pragma unroll
          for (int k = 0; k < 6; k++)
            *reinterpret_cast<float4*>(a.side_dst + (long long)k * pitch + x0) =
                make_float4(out[0][ks[k]], out[1][ks[k]], out[2][ks[k]], out[3][ks[k]]);
        }
#define LBM_PAIRS_PUSH(dstp, k)                                                                  \
  *reinterpret_cast<float4*>((dstp) + (long long)(k) * pitch + x0) = make_float4(out[0][k], out[1][k], out[2][k], out[3][k]);
        if (first) { LBM_PAIRS_PUSH(a.push_dn, 4) LBM_PAIRS_PUSH(a.push_dn, 7) LBM_PAIRS_PUSH(a.push_dn, 8) }
        if (last) { LBM_PAIRS_PUSH(a.push_up, 2) LBM_PAIRS_PUSH(a.push_up, 5) LBM_PAIRS_PUSH(a.push_up, 6) }
#undef LBM_PAIRS_PUSH
      }
    }
    warp_accumulate(q1, av1);
    warp_accumulate(q2, av2);
    grid_barrier(m.barrier, (unsigned long long)gridDim.x * (unsigned long long)(p + 1));
  }
}

}  // namespace lbm
