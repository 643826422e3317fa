// lbm_tb2.cuh -- K7: TWO timesteps per pass over HBM (temporal blocking), fp32, sm_100a.
//
// The one-step kernel K1a moves exactly the algorithmic 72 B per cell update and runs at the
// HBM roofline; the only way to more updates per second on a grid beyond L2 is fewer bytes
// per update.  K7 executes two consecutive iterations of the reference's step loop
// (d2q9-bgk.c:180-201, per-cell work :961-1131) while each distribution is read from HBM
// once and written once: 36 B per update plus halo overhead.
//
// Decomposition.  A block owns a "strip" of `wout` <= 376 columns and a "segment" of
// `seg_rows` rows, and marches through the segment row by row (y is the streaming
// direction, so there is no halo recomputation in y except two rows per segment):
//
//   iteration i, row r = R0 - 1 + i:
//     1. the nine pulled plane-rows of row r (384 columns: the strip plus 4 halo columns on
//        each side) arrive in shared memory by bulk asynchronous copies (cp.async.bulk,
//        issued two rows ahead by one thread, completion on an mbarrier) -- rows 0,1,3 from
//        row r, 2,5,6 from r-1, 4,7,8 from r+1, exactly the reads of K1a, each HBM element
//        once; ghost rows and the accelerated side row are selected per plane-row;
//     2. sub-step 1: every thread updates the four cells of its quad (x shifts are one extra
//        scalar shared-memory load) and writes the result into a ring of plane-rows in
//        shared memory -- it never goes to HBM.  If r is global row ny-2 the next step's
//        accelerate_flow (d2q9-bgk.c:229-260) is applied first, which is the reference's
//        order: accelerate, then stream;
//     3. sub-step 2 on row r-1 pulls from the ring (rows r-2, r-1, r of sub-step 1) and
//        stores to the destination lattice with 128-bit stores; edge rows are also pushed
//        into the neighbours' ghost rows, row ny-2 also (accelerated) into the side row.
//
//   Sub-step 1 is valid on span columns [1, 383), sub-step 2 on [2, 382); a thread stores
//   only quads inside the owned columns [4, 4 + wout).  Each sub-step's |u| sum counts owned
//   cells of the segment's own rows only, so av_vels[t] and av_vels[t+1] are exact.
//
// Same per-cell arithmetic as every other kernel (quad_update): the strict build is
// bit-exact against the reference arithmetic, the default build bit-identical to two K1a steps.
#pragma once
#include "lbm_kernels.cuh"

namespace lbm {

#ifndef LBM_TB2_THREADS
#define LBM_TB2_THREADS 96          /* one 384-column strip per block: as fast as 128 threads at 16384^2 and up to
                                       36 % faster on mid-size grids (more, smaller blocks), profiles/r02_kernel_variants.md */
#endif
#define LBM_TB2_SPAN (LBM_TB2_THREADS * 4)            /* columns loaded per strip */
#define LBM_TB2_PAD 4                                  /* floats left and right of a staged row */
#define LBM_TB2_ROWF (LBM_TB2_SPAN + 2 * LBM_TB2_PAD) /* 392 floats = 1568 B, a multiple of 16 B */
#define LBM_TB2_MAX_WOUT (LBM_TB2_SPAN - 8)           /* owned columns per strip */
#ifndef LBM_TB2_MIN_BLOCKS
#define LBM_TB2_MIN_BLOCKS 4                           /* 4 x 54.9 KB of shared memory per SM, 12 warps */
#endif

struct Tb2Smem {
  float in[2][9][LBM_TB2_ROWF];      // two stages of pulled plane-rows (TMA destination)
  float r013[2][3][LBM_TB2_ROWF];    // sub-step-1 rows: planes 0,1,3 (read one iteration later)
  float r256[3][3][LBM_TB2_ROWF];    // planes 2,5,6 (read two iterations later)
  float r78[2][LBM_TB2_ROWF];        // planes 7,8 (read in the same iteration; plane 4 stays in registers)
  unsigned long long mbar[2];         // "stage filled" (transaction barriers of the bulk copies)
  unsigned long long mbar_free;       // "ring slots of the previous iteration have been read" (one arrival per warp)
};
static_assert(sizeof(Tb2Smem) * LBM_TB2_MIN_BLOCKS <= 225 * 1024, "LBM_TB2_MIN_BLOCKS blocks of shared memory per SM");
static_assert((LBM_TB2_ROWF * sizeof(float)) % 16 == 0, "staged rows must keep 16-byte alignment");

struct Tb2Args {
  StepArgs<float> s;               // tiles_x = strips, tiles_y = segments, edge_tiles = 1; av = sums of sub-step 1
  const uint32_t* ghost_mask;      // own window: mask words of row -1, then of row `rows`
  unsigned long long* av2;         // sums of sub-step 2
  int wout;                        // owned columns per strip (multiple of 4, <= LBM_TB2_MAX_WOUT)
  int span;                        // staged columns per strip = threads x 4 (384), or nx + 8 for a narrow grid
  int seg_rows;                    // rows per segment ...
  int n_big;                       // ... of the first n_big segments, which cover rows [0, big_rows);
  int big_rows;                    // the segments behind them are seg_rows_tail rows tall: they get the highest
  int seg_rows_tail;               // block indices, so a launch ends with short blocks and the SMs drain together
  unsigned long long* av3;         // K10 only: sums of sub-step 3
};

__device__ __forceinline__ void tb2_mbar_wait(unsigned long long* bar, const uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done = 0;
  while (!done)
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.b32 %0, 1, 0, p; }"
                 : "=r"(done) : "r"(addr), "r"(parity) : "memory");
}

__device__ __forceinline__ void tb2_bulk_load(float* dst_smem, const float* src, const uint32_t bytes,
                                              unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst_smem)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// where plane k of local row `row` of the SOURCE state lives (row in [-2, rows + 2)); PERIODIC:
// the slab is the whole grid and rows beyond its ends are its own rows (row in [-rows, 2 rows))
template <bool PERIODIC = false>
__device__ __forceinline__ const float* tb2_row_ptr(const StepArgs<float>& a, const int k, int row) {
  if (PERIODIC) {
    row = (row < 0) ? row + a.rows : (row >= a.rows) ? row - a.rows : row;
  } else {
    if (row < 0) return a.ghost_s + (long long)((-1 - row) * 9 + k) * a.pitch;
    if (row >= a.rows) return a.ghost_n + (long long)((row - a.rows) * 9 + k) * a.pitch;
  }
  if (row == a.accel_row && k != 0 && k != 2 && k != 4) {
    const int idx = (k == 1) ? 0 : (k == 3) ? 1 : k - 3;       // side row order 1,3,5,6,7,8
    return a.side_src + (long long)idx * a.pitch;
  }
  return a.src + (long long)k * a.plane_stride + (long long)row * a.pitch;
}

// Start the copies of the nine plane-rows that sub-step 1 on row r pulls from.  The work is
// spread over the block so that no warp lags behind the others: thread t < 9 (one per plane,
// in different warps first) works out where "its" plane-row lives and copies it, in as many
// pieces as the periodic wrap in x cuts the span into (up to three when the span is the
// whole width plus halo).  The bytes were announced before by tb2_expect.
template <typename Smem>
__device__ __forceinline__ void tb2_expect(Smem& sm, const int stage, const int span) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&sm.mbar[stage])),
               "r"((uint32_t)(9 * span * sizeof(float))) : "memory");
}
__device__ __forceinline__ int tb2_plane_of_thread() {
  const int nwarps = (int)blockDim.x >> 5, w = (int)threadIdx.x >> 5, lane = (int)threadIdx.x & 31;
  const int k = w + nwarps * lane;
  return (k < 9) ? k : -1;
}
template <bool PERIODIC = false, typename Smem>
__device__ __forceinline__ void tb2_issue(const StepArgs<float>& a, Smem& sm, const int stage, const int r,
                                          const int s0, const int span, const int k) {
  if (k < 0) return;
  unsigned long long* bar = &sm.mbar[stage];
  const int dy = (k == 2 || k == 5 || k == 6) ? -1 : (k == 4 || k == 7 || k == 8) ? 1 : 0;
  const float* row = tb2_row_ptr<PERIODIC>(a, k, r + dy);
  float* dst = &sm.in[stage][k][LBM_TB2_PAD];
  int col = s0, left = span;
  while (left > 0) {
    const int n = min(left, a.nx - col);
    tb2_bulk_load(dst, row + col, (uint32_t)n * 4u, bar);
    dst += n;
    left -= n;
    col = 0;
  }
}

// the four cells of a quad from a staged plane-row: as stored / shifted one column
__device__ __forceinline__ void tb2_get(const float* row, const int c0, float& v0, float& v1, float& v2, float& v3) {
  const float4 v = *reinterpret_cast<const float4*>(row + LBM_TB2_PAD + c0);
  v0 = v.x; v1 = v.y; v2 = v.z; v3 = v.w;
}
__device__ __forceinline__ void tb2_get_west(const float* row, const int c0, float& v0, float& v1, float& v2, float& v3) {
  const float4 v = *reinterpret_cast<const float4*>(row + LBM_TB2_PAD + c0);
  v0 = row[LBM_TB2_PAD + c0 - 1]; v1 = v.x; v2 = v.y; v3 = v.z;
}
__device__ __forceinline__ void tb2_get_east(const float* row, const int c0, float& v0, float& v1, float& v2, float& v3) {
  const float4 v = *reinterpret_cast<const float4*>(row + LBM_TB2_PAD + c0);
  v0 = v.y; v1 = v.z; v2 = v.w; v3 = row[LBM_TB2_PAD + c0 + 4];
}
// this warp has finished reading the ring slots of the current iteration (release: the reads
// above are performed before any thread that waits on the barrier overwrites the slots)
__device__ __forceinline__ void tb2_ring_read_done(Tb2Smem& sm) {
  __syncwarp();
  if ((threadIdx.x & 31) == 0)
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&sm.mbar_free)) : "memory");
}
__device__ __forceinline__ void tb2_put(float* row, const int c0, const float (&o)[4][9], const int k) {
  *reinterpret_cast<float4*>(row + LBM_TB2_PAD + c0) = make_float4(o[0][k], o[1][k], o[2][k], o[3][k]);
}

// a thread's quad of a finished row y goes to the destination lattice with 128-bit stores; the
// slab's two edge rows at each end are also pushed into the neighbours' ghost rows, row ny-2
// also (accelerated) into the side row.  `out` is accelerated in place on that row.
template <bool STRICT>
__device__ __forceinline__ void tb2_store_row(const StepArgs<float>& a, const int y, const int xg, float (&out)[4][9],
                                              const uint32_t mbits) {
  const long long PS = a.plane_stride;
  float* d = a.dst + (long long)y * a.pitch + xg;
#pragma unroll
  for (int k = 0; k < 9; k++)
    *reinterpret_cast<float4*>(d + k * PS) = make_float4(out[0][k], out[1][k], out[2][k], out[3][k]);
  const bool first = (y == 0), second = (y == 1), last = (y == a.rows - 1), before_last = (y == a.rows - 2);
  const bool cA = (y == a.accel_row);
  if (first | second | last | before_last | cA) {        // block-uniform
    if (cA) {
#pragma unroll
      for (int j = 0; j < 4; j++)
        cell_accelerate<float, STRICT>(out[j][1], out[j][3], out[j][5], out[j][6], out[j][7], out[j][8],
                                       (mbits >> j) & 1u, a.aw1, a.aw2);
      const int ks[6] = {1, 3, 5, 6, 7, 8};
#pragma unroll
      for (int n = 0; n < 6; n++)
        *reinterpret_cast<float4*>(a.side_dst + (long long)n * a.pitch + xg) =
            make_float4(out[0][ks[n]], out[1][ks[n]], out[2][ks[n]], out[3][ks[n]]);
    }
#define LBM_TB2_PUSH(dst, depth, k)                                                             \
  *reinterpret_cast<float4*>((dst) + (long long)((depth) * 9 + (k)) * a.pitch + xg) =          \
      make_float4(out[0][k], out[1][k], out[2][k], out[3][k]);
    if (first) {
      LBM_TB2_PUSH(a.push_dn, 0, 4) LBM_TB2_PUSH(a.push_dn, 0, 7) LBM_TB2_PUSH(a.push_dn, 0, 8)
      LBM_TB2_PUSH(a.push_dn, 0, 0) LBM_TB2_PUSH(a.push_dn, 0, 1) LBM_TB2_PUSH(a.push_dn, 0, 3)
    }
    if (last) {
      LBM_TB2_PUSH(a.push_up, 0, 2) LBM_TB2_PUSH(a.push_up, 0, 5) LBM_TB2_PUSH(a.push_up, 0, 6)
      LBM_TB2_PUSH(a.push_up, 0, 0) LBM_TB2_PUSH(a.push_up, 0, 1) LBM_TB2_PUSH(a.push_up, 0, 3)
    }
    if (second) { LBM_TB2_PUSH(a.push_dn, 1, 4) LBM_TB2_PUSH(a.push_dn, 1, 7) LBM_TB2_PUSH(a.push_dn, 1, 8) }
    if (before_last) { LBM_TB2_PUSH(a.push_up, 1, 2) LBM_TB2_PUSH(a.push_up, 1, 5) LBM_TB2_PUSH(a.push_up, 1, 6) }
#undef LBM_TB2_PUSH
  }
}

// One tile = one strip x one segment, two timesteps.  `phases` holds the parity each staging
// barrier completes next (a block that works through several tiles keeps using the barriers).
template <bool STRICT>
__device__ __forceinline__ void tb2_tile(const Tb2Args& ta, Tb2Smem& sm, const int strip, const int seg,
                                         uint32_t& phases, unsigned long long& q1, unsigned long long& q2,
                                         bool& bad1, bool& bad2) {
  const StepArgs<float>& a = ta.s;
  const int tid = threadIdx.x;
  const int X0 = strip * ta.wout;                              // first owned column
  const int S0 = (X0 >= LBM_TB2_PAD) ? X0 - LBM_TB2_PAD : X0 - LBM_TB2_PAD + a.nx;   // first staged column
  const bool big = seg < ta.n_big;
  const int R0 = big ? seg * ta.seg_rows : ta.big_rows + (seg - ta.n_big) * ta.seg_rows_tail;
  const int R1 = big ? min(R0 + ta.seg_rows, ta.big_rows) : min(R0 + ta.seg_rows_tail, a.rows);
  const int n_it = R1 - R0 + 2;                                // sub-step-1 rows R0-1 .. R1

  // the quad's column inside the span (threads beyond the span idle along on its last quad)
  const int c0 = min(4 * tid, ta.span - 4);
  int xg = S0 + c0;                                            // ... and in the grid (nx % 4 == 0: no straddling)
  while (xg >= a.nx) xg -= a.nx;
  const bool owned = (tid >= 1) && (4 * tid < ta.span) && (c0 - LBM_TB2_PAD < ta.wout) &&
                     (X0 + c0 - LBM_TB2_PAD < a.nx);

  const int my_plane = tb2_plane_of_thread();
  if (tid == 0) { tb2_expect(sm, 0, ta.span); tb2_expect(sm, 1, ta.span); }
#pragma unroll 1
  for (int k = 0; k < 2; k++) tb2_issue(a, sm, k, R0 - 1 + k, S0, ta.span, my_plane);

  const QuadConsts<float, STRICT> qc(a.omega);
  const int mword_idx = xg >> 5, mshift = xg & 31;
  auto mask_bits = [&](const int row) -> uint32_t {
    const uint32_t* m = (row < 0) ? ta.ghost_mask : (row >= a.rows) ? ta.ghost_mask + a.mask_pitch
                                                                    : a.mask + (long long)row * a.mask_pitch;
    return (m[mword_idx] >> mshift) & 0xFu;
  };
  uint32_t mbits = mask_bits(R0 - 1);        // mask of the row sub-step 1 works on
  uint32_t mbits_prev = 0u;                  // ... and of the row before it (sub-step 2's row)

#pragma unroll 1
  for (int i = 0; i < n_it; i++) {
    const int st = i & 1;
    const int r = R0 - 1 + i;
    const uint32_t mbits_next = (i + 1 < n_it) ? mask_bits(r + 1) : 0u;
    float keep4[4];
    {
      // ---------------- sub-step 1 on row r: pulled values are staged in sm.in[st] ----------
      tb2_mbar_wait(&sm.mbar[st], (phases >> st) & 1u);
      phases ^= 1u << st;
      if (tid == 0 && i + 2 < n_it) tb2_expect(sm, st, ta.span);      // the refill of this stage, issued after the barrier below
      float in[4][9], out[4][9];
      const float(*row)[LBM_TB2_ROWF] = sm.in[st];
      tb2_get(row[0], c0, in[0][0], in[1][0], in[2][0], in[3][0]);
      tb2_get(row[2], c0, in[0][2], in[1][2], in[2][2], in[3][2]);
      tb2_get(row[4], c0, in[0][4], in[1][4], in[2][4], in[3][4]);
      tb2_get_west(row[1], c0, in[0][1], in[1][1], in[2][1], in[3][1]);
      tb2_get_west(row[5], c0, in[0][5], in[1][5], in[2][5], in[3][5]);
      tb2_get_west(row[8], c0, in[0][8], in[1][8], in[2][8], in[3][8]);
      tb2_get_east(row[3], c0, in[0][3], in[1][3], in[2][3], in[3][3]);
      tb2_get_east(row[6], c0, in[0][6], in[1][6], in[2][6], in[3][6]);
      tb2_get_east(row[7], c0, in[0][7], in[1][7], in[2][7], in[3][7]);
      bool bad;
      const unsigned long long q = quad_update<float, STRICT>(in, mbits, qc, out, bad);
      if (owned && r >= R0 && r < R1) { q1 += q; bad1 |= bad; }
      if (r == a.accel_row) {              // accelerate_flow between the two steps (d2q9-bgk.c:229-260)
#pragma unroll
        for (int j = 0; j < 4; j++)
          cell_accelerate<float, STRICT>(out[j][1], out[j][3], out[j][5], out[j][6], out[j][7], out[j][8],
                                         (mbits >> j) & 1u, a.aw1, a.aw2);
      }
      // the ring slots written now were read by sub-step 2 of the previous iteration: every warp
      // has said so (mbar_free) a whole sub-step ago, so this wait is normally free -- it replaces
      // a second block barrier per row, which cost 11 % (profiles/r02_kernel_variants.md)
      if (i > 0) {
        tb2_mbar_wait(&sm.mbar_free, (phases >> 2) & 1u);
        phases ^= 4u;
      }
      tb2_put(sm.r013[i & 1][0], c0, out, 0);
      tb2_put(sm.r013[i & 1][1], c0, out, 1);
      tb2_put(sm.r013[i & 1][2], c0, out, 3);
      tb2_put(sm.r256[i % 3][0], c0, out, 2);
      tb2_put(sm.r256[i % 3][1], c0, out, 5);
      tb2_put(sm.r256[i % 3][2], c0, out, 6);
      tb2_put(sm.r78[0], c0, out, 7);
      tb2_put(sm.r78[1], c0, out, 8);
#pragma unroll
      for (int j = 0; j < 4; j++) keep4[j] = out[j][4];
    }
    __syncthreads();          // ring rows of this iteration are complete; stage `st` has been read by everyone
    if (i + 2 < n_it) tb2_issue(a, sm, st, r + 2, S0, ta.span, my_plane);

    if (i >= 2) {
      // ---------------- sub-step 2 on row y = r - 1, pulling sub-step-1 rows y-1, y, y+1 ----
      const int y = r - 1;
      float in[4][9], out[4][9];
      const float(*c)[LBM_TB2_ROWF] = sm.r013[(i - 1) & 1];    // row y
      const float(*s)[LBM_TB2_ROWF] = sm.r256[(i - 2) % 3];    // row y - 1
      tb2_get(c[0], c0, in[0][0], in[1][0], in[2][0], in[3][0]);
      tb2_get_west(c[1], c0, in[0][1], in[1][1], in[2][1], in[3][1]);
      tb2_get_east(c[2], c0, in[0][3], in[1][3], in[2][3], in[3][3]);
      tb2_get(s[0], c0, in[0][2], in[1][2], in[2][2], in[3][2]);
      tb2_get_west(s[1], c0, in[0][5], in[1][5], in[2][5], in[3][5]);
      tb2_get_east(s[2], c0, in[0][6], in[1][6], in[2][6], in[3][6]);
#pragma unroll
      for (int j = 0; j < 4; j++) in[j][4] = keep4[j];         // row y + 1 = r, this thread's own cells
      tb2_get_east(sm.r78[0], c0, in[0][7], in[1][7], in[2][7], in[3][7]);
      tb2_get_west(sm.r78[1], c0, in[0][8], in[1][8], in[2][8], in[3][8]);
      tb2_ring_read_done(sm);
      bool bad;
      const unsigned long long q = quad_update<float, STRICT>(in, mbits_prev, qc, out, bad);
      if (owned) {
        q2 += q;
        bad2 |= bad;
        tb2_store_row<STRICT>(a, y, xg, out, mbits_prev);
      }
    }
    else {
      tb2_ring_read_done(sm);   // nothing read in the first two iterations: keep one arrival per warp per iteration
    }
    mbits_prev = mbits;
    mbits = mbits_next;
  }

}

// shared memory of a block before its first tile: staging barriers, and the pads of the staged
// rows -- never written by the copies or the ring stores, read by the edge quads of the span
// (whose results are never used): keep them defined
__device__ __forceinline__ void tb2_init_smem(Tb2Smem& sm, const int span) {
  const int tid = threadIdx.x;
  for (int i = tid; i < 35 * 2 * LBM_TB2_PAD; i += blockDim.x) {
    float* row = &sm.in[0][0][0] + (size_t)(i / (2 * LBM_TB2_PAD)) * LBM_TB2_ROWF;
    const int e = i % (2 * LBM_TB2_PAD);
    row[e < LBM_TB2_PAD ? e : span + e] = 0.f;
  }
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&sm.mbar[0])) : "memory");
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&sm.mbar[1])) : "memory");
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(&sm.mbar_free)), "r"((uint32_t)(blockDim.x >> 5)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
}

// ------------------------------------------------------------------------------------
// K7  lbm_step2_tb: one launch = two timesteps of one slab (grids beyond L2, any GPU count)
// ------------------------------------------------------------------------------------
template <bool STRICT, bool MULTI>
__global__ void __launch_bounds__(LBM_TB2_THREADS, LBM_TB2_MIN_BLOCKS)
lbm_step2_tb(const __grid_constant__ Tb2Args ta) {
  extern __shared__ __align__(128) unsigned char tb2_smem_raw[];
  Tb2Smem& sm = *reinterpret_cast<Tb2Smem*>(tb2_smem_raw);
  const StepArgs<float>& a = ta.s;
  int strip, seg;
  tile_of_block(a.tiles_x, a.tiles_y, 1, strip, seg);
  const bool is_boundary = is_edge_tile(seg, a.tiles_y, 1);
  tb2_init_smem(sm, ta.span);
  cudaGridDependencySynchronize();           // PDL: the previous pass's writes are visible from here on
  __syncthreads();
  boundary_wait<float, MULTI>(a, is_boundary);
  uint32_t phases = 0u;
  unsigned long long q1 = 0ULL, q2 = 0ULL;
  bool bad1 = false, bad2 = false;
  tb2_tile<STRICT>(ta, sm, strip, seg, phases, q1, q2, bad1, bad2);
  if (bad1) atomicOr(a.av + 1, LBM_NONFINITE_MARK);
  if (bad2) atomicOr(ta.av2 + 1, LBM_NONFINITE_MARK);
  block_accumulate(q1, a.av);
  __syncthreads();            // block_accumulate's shared scratch is reused
  block_accumulate(q2, ta.av2);
  boundary_signal<float, MULTI>(a, is_boundary);
}

}  // namespace lbm
