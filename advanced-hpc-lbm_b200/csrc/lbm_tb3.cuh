// lbm_tb3.cuh -- K10: THREE timesteps per pass over HBM (temporal blocking), fp32, sm_100a.
//
// K7 (lbm_tb2.cuh) moves 36 B per update and runs at ~94 % of the copy bandwidth; the only
// large gain left on grids beyond L2 is fewer bytes per update.  K10 executes three
// consecutive iterations of the reference's step loop (d2q9-bgk.c:180-201) while each
// distribution is read from HBM once and written once: 24 B per update plus halo overhead.
//
// Scope: one slab that holds the whole grid (one GPU, periodic in y).  Rows beyond the slab's
// ends are then its own rows, so K10 reads them from the source lattice directly and needs
// no three-deep ghost zones; it still pushes K7's two-deep ghost rows, so that a K7 pass (two
// steps left) or a K1a step (one left) can follow it.  Several slabs run K7.
//
// Decomposition: K7's strips and segments, bulk-copy staging with mbarrier completion.
// Iteration i of a segment [R0, R1), source row r = R0 - 2 + i:
//   1. sub-step 1 on row r from the staged input -> ring level 1;
//   2. sub-step 2 on row r-1 from ring level 1  -> ring level 2      (i >= 2);
//   3. sub-step 3 on row r-2 from ring level 2  -> HBM, 128-bit stores (i >= 4).
// Sub-step 1 covers rows R0-2 .. R1+1, sub-step 2 R0-1 .. R1, sub-step 3 R0 .. R1-1; sub-step k
// is valid on span columns [k, span-k), which contain the owned columns [4, span-4).
//
// Staging is one stage deep: the copies of row r+1 are issued right after the first block
// barrier of iteration i (everyone has read row r by then) and land while sub-steps 2 and 3
// run.  A second stage would hide more copy latency but costs 9 plane-rows, and without them
// a fourth block fits on the SM: 12 warps instead of 9 hide the shared-memory and barrier
// latency this kernel is bound by (profiles/r07_k10_four_blocks.md).
//
// The ring is lean: planes 0, 2 and 4 are pulled from the thread's own columns, so they stay
// in registers (plane 4 of row r is used in the same iteration, plane 0 of row r-1 is carried
// one iteration, plane 2 of rows r-2 and r-1 two).  Only the six x-shifted planes go through
// shared memory: 12 plane-rows per level instead of 17.  With plane 0 of level 2 (2 rows)
// that is 9 + 2 x 12 + 2 = 35 plane-rows of 1568 B (53.6 KB): four blocks (12 warps) share an SM.
//
// Ordering: two block barriers per iteration, one after each ring level is written.  Each
// also orders the reads of the previous iteration before the writes of this one (WAR), so no
// "slots free" barrier is needed.
//
// Same per-cell arithmetic as every other kernel (quad_update): the strict build is bit-exact
// against the reference arithmetic, the default build bit-identical to three K1a steps.
#pragma once
#include "lbm_tb2.cuh"

namespace lbm {

#ifndef LBM_TB3_MIN_BLOCKS
#define LBM_TB3_MIN_BLOCKS (LBM_TB2_THREADS <= 96 ? 4 : 2)
#endif

#ifdef LBM_EXPERIMENTS
// clock64() cycles K10 spends waiting for staged rows [0] and in its tiles [1], summed over the
// warps (lane 0 of each); read and cleared by lbm_gpu_exp_tb3_cycles (tools/build_variants.py)
__device__ unsigned long long tb3_exp_cycles[2];
// %globaltimer of K10's blocks: earliest start [0], latest end [1], sum of block durations [2]
// (start = the previous pass's data is available, end = the tile is published); read and
// cleared by lbm_gpu_exp_tb3_blocks
__device__ unsigned long long tb3_exp_blocks[3] = {~0ULL, 0ULL, 0ULL};
#endif

struct Tb3Level {                       // one level of the ring: the x-shifted planes of sub-step-k rows
  float r13[2][2][LBM_TB2_ROWF];        // planes 1,3 of the rows of this and the previous iteration
  float r56[3][2][LBM_TB2_ROWF];        // planes 5,6 of the rows of the last three iterations
  float r78[2][LBM_TB2_ROWF];           // planes 7,8 of this iteration's row
};
struct Tb3Smem {
  float in[1][9][LBM_TB2_ROWF];         // one stage of pulled plane-rows (bulk copy destination; the stage
                                        // index keeps K7's tb2_expect / tb2_issue usable)
  Tb3Level lv[2];                       // sub-step-1 rows, sub-step-2 rows
  float p0[2][LBM_TB2_ROWF];            // plane 0 of the sub-step-2 rows of this and the previous iteration
                                        // (in shared memory, not registers: 12 warps per SM leave 168 each)
  unsigned long long mbar[1];           // "stage filled"
};
constexpr int kTb3PlaneRows = 9 + 2 * 12 + 2;
static_assert(sizeof(Tb3Smem) == kTb3PlaneRows * LBM_TB2_ROWF * sizeof(float) + 8, "ring layout");
// per block: the dynamic layout, block_accumulate's 512 B of static scratch, 1 KB reserved by the SM
static_assert((sizeof(Tb3Smem) + 512 + 1024) * LBM_TB3_MIN_BLOCKS <= 228 * 1024,
              "LBM_TB3_MIN_BLOCKS blocks of shared memory per SM");

__device__ __forceinline__ void tb3_init_smem(Tb3Smem& sm, const int span) {
  const int tid = threadIdx.x;
  for (int i = tid; i < kTb3PlaneRows * 2 * LBM_TB2_PAD; i += blockDim.x) {
    float* row = &sm.in[0][0][0] + (size_t)(i / (2 * LBM_TB2_PAD)) * LBM_TB2_ROWF;
    const int e = i % (2 * LBM_TB2_PAD);
    row[e < LBM_TB2_PAD ? e : span + e] = 0.f;
  }
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&sm.mbar[0])) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
}

// sub-steps 2 and 3 on row y pull from the rows y-1 (slot s56 of level L, plane 2 in p2),
// y (slot s13, plane 0 in p0) and y+1 (r78, plane 4 in p4) of the sub-step before
__device__ __forceinline__ void tb3_gather(const Tb3Level& L, const int c0, const int s13, const int s56,
                                           const float (&p0)[4], const float (&p2)[4], const float (&p4)[4],
                                           float (&in)[4][9]) {
#pragma unroll
  for (int j = 0; j < 4; j++) { in[j][0] = p0[j]; in[j][2] = p2[j]; in[j][4] = p4[j]; }
  tb2_get_west(L.r13[s13][0], c0, in[0][1], in[1][1], in[2][1], in[3][1]);
  tb2_get_east(L.r13[s13][1], c0, in[0][3], in[1][3], in[2][3], in[3][3]);
  tb2_get_west(L.r56[s56][0], c0, in[0][5], in[1][5], in[2][5], in[3][5]);
  tb2_get_east(L.r56[s56][1], c0, in[0][6], in[1][6], in[2][6], in[3][6]);
  tb2_get_east(L.r78[0], c0, in[0][7], in[1][7], in[2][7], in[3][7]);
  tb2_get_west(L.r78[1], c0, in[0][8], in[1][8], in[2][8], in[3][8]);
}
// ... and write a sub-step's row into level L (slots of iteration i); planes 0, 2, 4 stay in registers
__device__ __forceinline__ void tb3_put_level(Tb3Level& L, const int c0, const int i, const float (&o)[4][9]) {
  tb2_put(L.r13[i & 1][0], c0, o, 1);
  tb2_put(L.r13[i & 1][1], c0, o, 3);
  tb2_put(L.r56[i % 3][0], c0, o, 5);
  tb2_put(L.r56[i % 3][1], c0, o, 6);
  tb2_put(L.r78[0], c0, o, 7);
  tb2_put(L.r78[1], c0, o, 8);
}

template <bool STRICT>
__device__ __forceinline__ void tb3_accelerate(const StepArgs<float>& a, float (&o)[4][9], const uint32_t mbits) {
#pragma unroll
  for (int j = 0; j < 4; j++)
    cell_accelerate<float, STRICT>(o[j][1], o[j][3], o[j][5], o[j][6], o[j][7], o[j][8], (mbits >> j) & 1u, a.aw1, a.aw2);
}

// registers a level carries from iteration to iteration
struct Tb3Carry {
  float p0[4];        // plane 0 of the previous iteration's row
  float p2a[4];       // plane 2 of the row two iterations back
  float p2b[4];       // plane 2 of the previous iteration's row
  __device__ __forceinline__ void shift(const float (&o)[4][9]) {
#pragma unroll
    for (int j = 0; j < 4; j++) { p0[j] = o[j][0]; p2a[j] = p2b[j]; p2b[j] = o[j][2]; }
  }
};

// One tile = one strip x one segment, three timesteps.
template <bool STRICT>
__device__ __forceinline__ void tb3_tile(const Tb2Args& ta, Tb3Smem& sm, const int strip, const int seg,
                                         unsigned long long (&q)[3], bool (&bad)[3]) {
  const StepArgs<float>& a = ta.s;
  const int tid = threadIdx.x;
  const int X0 = strip * ta.wout;                              // first owned column
  const int S0 = (X0 >= LBM_TB2_PAD) ? X0 - LBM_TB2_PAD : X0 - LBM_TB2_PAD + a.nx;   // first staged column
  const bool big = seg < ta.n_big;
  const int R0 = big ? seg * ta.seg_rows : ta.big_rows + (seg - ta.n_big) * ta.seg_rows_tail;
  const int R1 = big ? min(R0 + ta.seg_rows, ta.big_rows) : min(R0 + ta.seg_rows_tail, a.rows);
  const int n_it = R1 - R0 + 4;                                // sub-step-1 rows R0-2 .. R1+1

  const int c0 = min(4 * tid, ta.span - 4);
  int xg = S0 + c0;
  while (xg >= a.nx) xg -= a.nx;
  const bool owned = (tid >= 1) && (4 * tid < ta.span) && (c0 - LBM_TB2_PAD < ta.wout) &&
                     (X0 + c0 - LBM_TB2_PAD < a.nx);

  const int my_plane = tb2_plane_of_thread();
  if (tid == 0) tb2_expect(sm, 0, ta.span);
  tb2_issue<true>(a, sm, 0, R0 - 2, S0, ta.span, my_plane);

  const QuadConsts<float, STRICT> qc(a.omega);
  const int mword_idx = xg >> 5, mshift = xg & 31;
  auto wrap = [&](const int row) { return (row < 0) ? row + a.rows : (row >= a.rows) ? row - a.rows : row; };
  auto mask_bits = [&](const int row) -> uint32_t {
    return (a.mask[(long long)wrap(row) * a.mask_pitch + mword_idx] >> mshift) & 0xFu;
  };
  uint32_t m1 = mask_bits(R0 - 2), m2 = 0u, m3 = 0u;   // masks of the rows of sub-steps 1, 2, 3
  Tb3Carry c1, c2;                                      // levels 1 and 2 (level 2 keeps plane 0 in sm.p0)
  uint32_t phase = 0u;                                  // parity the staging barrier completes next
#ifdef LBM_EXPERIMENTS
  const long long t_tile = clock64();
  long long t_wait = 0;
#endif

#pragma unroll 1
  for (int i = 0; i < n_it; i++) {
    const int r = R0 - 2 + i;
    const uint32_t m_next = (i + 1 < n_it) ? mask_bits(r + 1) : 0u;
    float in[4][9], out[4][9];
    bool b;
    // ---------------- sub-step 1 on row r: pulled values are staged in sm.in[0] -----------------
#ifdef LBM_EXPERIMENTS
    const long long t0 = clock64();
    tb2_mbar_wait(&sm.mbar[0], phase);
    t_wait += clock64() - t0;
#else
    tb2_mbar_wait(&sm.mbar[0], phase);
#endif
    phase ^= 1u;
    if (tid == 0 && i + 1 < n_it) tb2_expect(sm, 0, ta.span);       // the refill with row r+1, issued after the barrier below
    {
      const float(*row)[LBM_TB2_ROWF] = sm.in[0];
      tb2_get(row[0], c0, in[0][0], in[1][0], in[2][0], in[3][0]);
      tb2_get(row[2], c0, in[0][2], in[1][2], in[2][2], in[3][2]);
      tb2_get(row[4], c0, in[0][4], in[1][4], in[2][4], in[3][4]);
      tb2_get_west(row[1], c0, in[0][1], in[1][1], in[2][1], in[3][1]);
      tb2_get_west(row[5], c0, in[0][5], in[1][5], in[2][5], in[3][5]);
      tb2_get_west(row[8], c0, in[0][8], in[1][8], in[2][8], in[3][8]);
      tb2_get_east(row[3], c0, in[0][3], in[1][3], in[2][3], in[3][3]);
      tb2_get_east(row[6], c0, in[0][6], in[1][6], in[2][6], in[3][6]);
      tb2_get_east(row[7], c0, in[0][7], in[1][7], in[2][7], in[3][7]);
    }
    unsigned long long qq = quad_update<float, STRICT>(in, m1, qc, out, b);
    if (owned && r >= R0 && r < R1) { q[0] += qq; bad[0] |= b; }
    if (wrap(r) == a.accel_row) tb3_accelerate<STRICT>(a, out, m1);   // before the next step pulls (d2q9-bgk.c:229-260)
    tb3_put_level(sm.lv[0], c0, i, out);
    float p4[4];
#pragma unroll
    for (int j = 0; j < 4; j++) p4[j] = out[j][4];
    __syncthreads();          // level-1 row r is complete; the stage has been read by everyone
    if (i + 1 < n_it) tb2_issue<true>(a, sm, 0, r + 1, S0, ta.span, my_plane);

    if (i >= 2) {
      // ---------------- sub-step 2 on row y = r - 1 from level-1 rows y-1, y, y+1 --------------
      const int y = r - 1;
      tb3_gather(sm.lv[0], c0, (i - 1) & 1, (i - 2) % 3, c1.p0, c1.p2a, p4, in);
      c1.shift(out);
      qq = quad_update<float, STRICT>(in, m2, qc, out, b);
      if (owned && y >= R0 && y < R1) { q[1] += qq; bad[1] |= b; }
      if (wrap(y) == a.accel_row) tb3_accelerate<STRICT>(a, out, m2);
      tb3_put_level(sm.lv[1], c0, i, out);
      tb2_put(sm.p0[i & 1], c0, out, 0);
      float n2[4];
#pragma unroll
      for (int j = 0; j < 4; j++) { n2[j] = out[j][2]; p4[j] = out[j][4]; }
      __syncthreads();        // level-2 row y is complete

      if (i >= 4) {
        // ---------------- sub-step 3 on row z = r - 2 from level-2 rows z-1, z, z+1 -------------
        const int z = r - 2;
        tb3_gather(sm.lv[1], c0, (i - 1) & 1, (i - 2) % 3, c2.p2a, c2.p2a, p4, in);   // plane 0: below
        tb2_get(sm.p0[(i - 1) & 1], c0, in[0][0], in[1][0], in[2][0], in[3][0]);
        qq = quad_update<float, STRICT>(in, m3, qc, out, b);
        if (owned) {
          q[2] += qq;
          bad[2] |= b;
          tb2_store_row<STRICT>(a, z, xg, out, m3);
        }
      }
#pragma unroll
      for (int j = 0; j < 4; j++) { c2.p2a[j] = c2.p2b[j]; c2.p2b[j] = n2[j]; }
    } else {
      c1.shift(out);
    }
    m3 = m2;
    m2 = m1;
    m1 = m_next;
  }
#ifdef LBM_EXPERIMENTS
  if ((tid & 31) == 0) {
    atomicAdd(&tb3_exp_cycles[0], (unsigned long long)t_wait);
    atomicAdd(&tb3_exp_cycles[1], (unsigned long long)(clock64() - t_tile));
  }
#endif
}

// Blocks take the segments middle-out (m, m-1, m+1, m-2, ...; m = tiles_y / 2), so the last
// blocks of a pass are segments 0 and tiles_y-1 and their neighbours: the first blocks of the next
// pass, around m, do not wait for the last ones of this pass.  The order changes no result.
__device__ __forceinline__ int tb3_seg_of_slot(const int slot, const int tiles_y) {
  return (slot & 1) ? tiles_y / 2 - (slot + 1) / 2 : tiles_y / 2 + slot / 2;
}
__device__ __forceinline__ int tb3_slot_of_seg(const int seg, const int tiles_y) {
  return (seg >= tiles_y / 2) ? 2 * (seg - tiles_y / 2) : 2 * (tiles_y / 2 - seg) - 1;
}

__device__ __forceinline__ uint32_t ld_acquire_gpu_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// Overlapped passes: thread 0 waits until the 3 x 3 neighbourhood of tile (strip, seg), periodic
// in x and y, has completed the previous pass: its words count passes completed, so they must
// reach a.pass (signed difference, so wrap-around is harmless; a word starts at 0, which no pass
// after the first can mistake for its predecessor).  The host allows the overlap only where that
// neighbourhood holds every tile that reads a cell this tile writes, and every tile that writes a
// cell this tile reads (Grid::tb3_overlap_fits).  The wait is bounded like boundary_wait: on a time-out, or when
// another block gave up, the block records why, raises the abort word and carries on; the run's
// results are void and lbm_gpu_run reports it.
__device__ __forceinline__ void tb3_wait_tiles(const Tb2Args& ta, const int strip, const int seg) {
  const StepArgs<float>& a = ta.s;
  const uint32_t done = (uint32_t)a.pass;
  const unsigned long long t0 = global_timer_ns();
  unsigned ns = 32;
#pragma unroll 1
  for (int dy = -1; dy <= 1; dy++) {
    if ((dy == -1 && a.tiles_y < 2) || (dy == 1 && a.tiles_y < 3)) continue;    // fewer than three segments
    const int y = (seg + dy + a.tiles_y) % a.tiles_y;
#pragma unroll 1
    for (int dx = -1; dx <= 1; dx++) {
      if ((dx == -1 && a.tiles_x < 2) || (dx == 1 && a.tiles_x < 3)) continue;  // ... or strips
      const uint32_t* f = ta.tile_done + (size_t)tb3_slot_of_seg(y, a.tiles_y) * a.tiles_x + (strip + dx + a.tiles_x) % a.tiles_x;
      while ((int)(ld_acquire_gpu_u32(f) - done) < 0) {
        if (ld_acquire_sys(a.abort_word) != 0ULL) return;
        if (global_timer_ns() - t0 > a.timeout_ns) {
          atomicCAS(a.abort_word + 1, 0ULL, (LBM_SYNC_TILE_TIMEOUT << 56) | (a.pass & 0xffffffffffffffULL));
          st_release_sys(a.abort_word, 1ULL);
          return;
        }
        __nanosleep(ns);
        ns = min(2u * ns, 1024u);
      }
    }
  }
}

// ------------------------------------------------------------------------------------
// K10  lbm_step3_tb: one launch = three timesteps of a slab that holds the whole grid
// ------------------------------------------------------------------------------------
// Consecutive K10 passes overlap (ta.tile_done set): every block triggers the next launch as soon
// as it is resident, and publishes the number of passes its tile has completed after its last
// global write.  A block
// of a pass that follows a K10 pass (ta.wait_tiles) waits for its nine neighbour tiles of that
// pass instead of the whole grid.  Deadlock freedom: the next grid launches only once every block
// of this one has triggered, i.e. is resident or finished, so every tile a waiting block depends
// on already holds an SM or is done; the oldest pass in flight waits for nothing that is not.
// A kernel after K10 that calls cudaGridDependencySynchronize (K7, K1a) still waits for the
// whole grid to complete and flush, as does anything launched without programmatic
// serialization.
// The words of ta.tile_done are indexed by block, not by tile: the epilogue then needs nothing
// the row loop has to keep in registers.
template <bool STRICT>
__global__ void __launch_bounds__(LBM_TB2_THREADS, LBM_TB3_MIN_BLOCKS)
lbm_step3_tb(const __grid_constant__ Tb2Args ta) {
  extern __shared__ __align__(128) unsigned char tb3_smem_raw[];
  Tb3Smem& sm = *reinterpret_cast<Tb3Smem*>(tb3_smem_raw);
  const StepArgs<float>& a = ta.s;
  const int slot = (int)(blockIdx.x / (unsigned)a.tiles_x);
  const int strip = (int)blockIdx.x - slot * a.tiles_x;
  const int seg = tb3_seg_of_slot(slot, a.tiles_y);
  tb3_init_smem(sm, ta.span);
  if (ta.tile_done) cudaTriggerProgrammaticLaunchCompletion();
  if (ta.wait_tiles) {
    if (threadIdx.x == 0) tb3_wait_tiles(ta, strip, seg);
  } else {
    cudaGridDependencySynchronize();         // PDL: the previous pass's writes are visible from here on
  }
  __syncthreads();
  if (ta.wait_tiles) asm volatile("fence.proxy.async.global;" ::: "memory");   // the staging copies are async-proxy reads
#ifdef LBM_EXPERIMENTS
  const unsigned long long t_start = global_timer_ns();
#endif
  unsigned long long q[3] = {0ULL, 0ULL, 0ULL};
  bool bad[3] = {false, false, false};
  tb3_tile<STRICT>(ta, sm, strip, seg, q, bad);
  if (bad[0]) atomicOr(a.av + 1, LBM_NONFINITE_MARK);
  if (bad[1]) atomicOr(ta.av2 + 1, LBM_NONFINITE_MARK);
  if (bad[2]) atomicOr(ta.av3 + 1, LBM_NONFINITE_MARK);
  block_accumulate(q[0], a.av);
  __syncthreads();            // block_accumulate's shared scratch is reused
  block_accumulate(q[1], ta.av2);
  __syncthreads();
  block_accumulate(q[2], ta.av3);
  if (ta.tile_done) {
    // every store of the tile, its ghost-row pushes and its sums are made visible before the
    // tile is published (stores of this pass may be read by bulk copies of the next)
    asm volatile("fence.proxy.async.global;" ::: "memory");
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence();
      asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(ta.tile_done + blockIdx.x),
                   "r"((uint32_t)a.pass + 1u) : "memory");
    }
  }
#ifdef LBM_EXPERIMENTS
  if (threadIdx.x == 0) {
    const unsigned long long t_end = global_timer_ns();
    atomicMin(&tb3_exp_blocks[0], t_start);
    atomicMax(&tb3_exp_blocks[1], t_end);
    atomicAdd(&tb3_exp_blocks[2], t_end - t_start);
  }
#endif
}

}  // namespace lbm
