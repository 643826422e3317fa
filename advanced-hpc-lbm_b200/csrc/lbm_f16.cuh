// lbm_f16.cuh -- shifted binary16 lattice storage (LBM_GPU_STORE_F16), sm_100a.
//
// The lattice holds s_k = binary16(f_k - c_k), c_k the rest-state value of speed k (RestShift in
// lbm_kernels.cuh): half the bytes per distribution.  Every kernel here decodes after the load,
// runs the ordinary fp32 per-cell code (quad_update, cell_accelerate) and encodes before the
// store, so a timestep is the fp32 step between a decode and an encode.  Two values are not
// rounded: the accelerated row ny-2 (the side row stays fp32, and K7-f16 keeps the accelerated
// sub-step-1 row in fp32 shared memory) and the |u| of av_vels (from the fp32 results).
//
// One slab holds the whole grid, so rows beyond its ends are its own rows, read straight from
// the source lattice: no ghost rows, no pushes, no cross-slab ordering.
//   K1a-f16  lbm_step_vec4_f16  one step per pass, K1a's shape: four cells per thread, four
//            binary16 values (8 B) per plane per load, x shifts by warp shuffle.  Any nx.
//   K7-f16   lbm_step2_tb_f16   two steps per pass, K7's strips, segments and bulk-copy staging,
//            with binary16 staged rows and a binary16 sub-step-1 ring (decoded when read).
//            18 B per update.  Its bulk copies move 16-byte pieces, so nx must be a multiple of 8.
#pragma once
#include "lbm_kernels.cuh"
#include "lbm_tb2.cuh"

namespace lbm {

struct F16Args {
  const __half* src;           // lattice buffer read this pass
  __half* dst;                 // lattice buffer written
  const float* side_src;       // accelerated row ny-2, planes {1,3,5,6,7,8} x pitch (fp32, read)
  float* side_dst;             // same, written for the next step
  const uint32_t* mask;
  unsigned long long* av;      // |u| sums of the (first) step of the pass
  unsigned long long* av2;     // K7-f16: of the second step
  long long plane_stride;
  int nx, rows, pitch, mask_pitch, accel_row;
  int tiles_x, tiles_y;
  float omega, aw1, aw2;
  RestShift rest;
  int wout, span, seg_rows, n_big, big_rows, seg_rows_tail;   // K7-f16, as in Tb2Args
};

__device__ __forceinline__ int wrap_row(const int r, const int rows) { return r < 0 ? r + rows : (r >= rows ? r - rows : r); }

// four binary16 values (8 bytes, aligned) decoded / four fp32 values encoded
__device__ __forceinline__ Vec4<float> dec4(const uint2 u, const float c) {
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x));
  const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
  Vec4<float> v;
  v.x = __fadd_rn(a.x, c); v.y = __fadd_rn(a.y, c); v.z = __fadd_rn(b.x, c); v.w = __fadd_rn(b.y, c);
  return v;
}
__device__ __forceinline__ uint2 enc4(const float x, const float y, const float z, const float w, const float c) {
  const __half2 lo = __halves2half2(f16_enc(x, c), f16_enc(y, c));
  const __half2 hi = __halves2half2(f16_enc(z, c), f16_enc(w, c));
  uint2 u;
  u.x = *reinterpret_cast<const uint32_t*>(&lo);
  u.y = *reinterpret_cast<const uint32_t*>(&hi);
  return u;
}
__device__ __forceinline__ float round_f16(const float f, const float c) { return f16_dec(f16_enc(f, c), c); }

// a thread's quad of a finished row: encoded into the destination lattice; row ny-2 also, from the
// values as stored (decoded) and then accelerated, into the fp32 side row
template <bool STRICT>
__device__ __forceinline__ void f16_store_quad(const F16Args& a, const int y, const int x, const float (&out)[4][9],
                                               const uint32_t mbits) {
  __half* d = a.dst + (long long)y * a.pitch + x;
#pragma unroll
  for (int k = 0; k < 9; k++)
    *reinterpret_cast<uint2*>(d + k * a.plane_stride) = enc4(out[0][k], out[1][k], out[2][k], out[3][k], a.rest.of(k));
  if (y == a.accel_row) {
    const int ks[6] = {1, 3, 5, 6, 7, 8};
    float f[4][6];
#pragma unroll
    for (int j = 0; j < 4; j++) {
#pragma unroll
      for (int n = 0; n < 6; n++) f[j][n] = round_f16(out[j][ks[n]], a.rest.of(ks[n]));
      cell_accelerate<float, STRICT>(f[j][0], f[j][1], f[j][2], f[j][3], f[j][4], f[j][5], (mbits >> j) & 1u, a.aw1, a.aw2);
    }
#pragma unroll
    for (int n = 0; n < 6; n++) {
      Vec4<float> v; v.x = f[0][n]; v.y = f[1][n]; v.z = f[2][n]; v.w = f[3][n];
      st4(a.side_dst + (long long)n * a.pitch + x, v);
    }
  }
}

// ------------------------------------------------------------------------------------
// K1a-f16  lbm_step_vec4_f16: K1a (lbm_step_vec4) on a binary16 lattice
// ------------------------------------------------------------------------------------
// where the pull of plane k comes from: a binary16 plane row, or (f != nullptr) the fp32 side row
struct F16Row { const __half* h; const float* f; };

__device__ __forceinline__ Vec4<float> f16_row4(const F16Row& p, const int x, const float c) {
  return p.f ? ld4(p.f + x) : dec4(*reinterpret_cast<const uint2*>(p.h + x), c);
}
__device__ __forceinline__ float f16_row1(const F16Row& p, const int x, const float c) {
  return p.f ? p.f[x] : f16_dec(p.h[x], c);
}

template <bool STRICT>
__global__ void __launch_bounds__(LBM_BLOCK_THREADS, LBM_MIN_BLOCKS)
lbm_step_vec4_f16(const __grid_constant__ F16Args a) {
  int tx, ty;
  tile_of_block(a.tiles_x, a.tiles_y, 1, tx, ty);
  cudaGridDependencySynchronize();           // PDL: the previous pass's writes are visible from here on
  const QuadConsts<float, STRICT> qc(a.omega);
  const int lane = threadIdx.x & 31;
  const int x0 = (tx * (int)blockDim.x + (int)threadIdx.x) * 4;
  const int r = ty * (int)blockDim.y + (int)threadIdx.y;
  const bool active = (x0 < a.nx) && (r < a.rows);
  const int xc = active ? x0 : 0;            // inactive threads take part in the shuffles only
  const int rc = active ? r : 0;
  const long long PS = a.plane_stride;
  const int rs = wrap_row(rc - 1, a.rows), rn = wrap_row(rc + 1, a.rows);
  const bool cA = (rc == a.accel_row), sA = (rs == a.accel_row), nA = (rn == a.accel_row);
  const __half* c = a.src + (long long)rc * a.pitch;
  const __half* s = a.src + (long long)rs * a.pitch;
  const __half* n = a.src + (long long)rn * a.pitch;
  const float* sd = a.side_src;
  const F16Row p0 = {c, nullptr}, p2 = {s + 2 * PS, nullptr}, p4 = {n + 4 * PS, nullptr};
  const F16Row p1 = {c + PS, cA ? sd : nullptr}, p3 = {c + 3 * PS, cA ? sd + a.pitch : nullptr};
  const F16Row p5 = {s + 5 * PS, sA ? sd + 2 * a.pitch : nullptr}, p6 = {s + 6 * PS, sA ? sd + 3 * a.pitch : nullptr};
  const F16Row p7 = {n + 7 * PS, nA ? sd + 4 * a.pitch : nullptr}, p8 = {n + 8 * PS, nA ? sd + 5 * a.pitch : nullptr};
  const float c0 = a.rest.w0, c1 = a.rest.w1, c2 = a.rest.w2;

  const bool need_w = (lane == 0) || (xc == 0);
  const bool need_e = (lane == 31) || (xc + 4 >= a.nx);
  const int xw = (xc == 0) ? a.nx - 1 : xc - 1;
  const int xe = (xc + 4 >= a.nx) ? 0 : xc + 4;
  float w1e = 0, w5e = 0, w8e = 0, e3e = 0, e6e = 0, e7e = 0;
  if (need_w) { w1e = f16_row1(p1, xw, c1); w5e = f16_row1(p5, xw, c2); w8e = f16_row1(p8, xw, c2); }
  if (need_e) { e3e = f16_row1(p3, xe, c1); e6e = f16_row1(p6, xe, c2); e7e = f16_row1(p7, xe, c2); }
  const Vec4<float> v0 = f16_row4(p0, xc, c0), v1 = f16_row4(p1, xc, c1), v2 = f16_row4(p2, xc, c1),
                    v3 = f16_row4(p3, xc, c1), v4 = f16_row4(p4, xc, c1), v5 = f16_row4(p5, xc, c2),
                    v6 = f16_row4(p6, xc, c2), v7 = f16_row4(p7, xc, c2), v8 = f16_row4(p8, xc, c2);
  const uint32_t mword = a.mask[(long long)rc * a.mask_pitch + (xc >> 5)];
  const uint32_t mbits = (mword >> (xc & 31)) & 0xFu;

  float l1 = __shfl_up_sync(0xffffffffu, v1.w, 1), l5 = __shfl_up_sync(0xffffffffu, v5.w, 1),
        l8 = __shfl_up_sync(0xffffffffu, v8.w, 1);
  float r3 = __shfl_down_sync(0xffffffffu, v3.x, 1), r6 = __shfl_down_sync(0xffffffffu, v6.x, 1),
        r7 = __shfl_down_sync(0xffffffffu, v7.x, 1);
  l1 = need_w ? w1e : l1; l5 = need_w ? w5e : l5; l8 = need_w ? w8e : l8;
  r3 = need_e ? e3e : r3; r6 = need_e ? e6e : r6; r7 = need_e ? e7e : r7;

  // a ragged last quad: padding cells are obstacles, the wrap element goes to the last valid cell
  const int nvalid = a.nx - xc;
  const bool n1 = (nvalid == 1), n2 = (nvalid == 2), n3 = (nvalid == 3);
  const uint32_t obits = (nvalid < 4) ? (mbits | ((0xFu << nvalid) & 0xFu)) : mbits;

  float in[4][9], out[4][9];
  in[0][0] = v0.x; in[1][0] = v0.y; in[2][0] = v0.z; in[3][0] = v0.w;
  in[0][1] = l1;   in[1][1] = v1.x; in[2][1] = v1.y; in[3][1] = v1.z;
  in[0][2] = v2.x; in[1][2] = v2.y; in[2][2] = v2.z; in[3][2] = v2.w;
  in[0][3] = n1 ? r3 : v3.y; in[1][3] = n2 ? r3 : v3.z; in[2][3] = n3 ? r3 : v3.w; in[3][3] = r3;
  in[0][4] = v4.x; in[1][4] = v4.y; in[2][4] = v4.z; in[3][4] = v4.w;
  in[0][5] = l5;   in[1][5] = v5.x; in[2][5] = v5.y; in[3][5] = v5.z;
  in[0][6] = n1 ? r6 : v6.y; in[1][6] = n2 ? r6 : v6.z; in[2][6] = n3 ? r6 : v6.w; in[3][6] = r6;
  in[0][7] = n1 ? r7 : v7.y; in[1][7] = n2 ? r7 : v7.z; in[2][7] = n3 ? r7 : v7.w; in[3][7] = r7;
  in[0][8] = l8;   in[1][8] = v8.x; in[2][8] = v8.y; in[3][8] = v8.z;

  bool bad;
  unsigned long long q = quad_update<float, STRICT>(in, obits, qc, out, bad);
  if (active) {
    if (bad) atomicOr(a.av + 1, LBM_NONFINITE_MARK);
    f16_store_quad<STRICT>(a, rc, xc, out, mbits);
  } else {
    q = 0ULL;
  }
  block_accumulate(q, a.av);
}

// ------------------------------------------------------------------------------------
// K7-f16  lbm_step2_tb_f16: K7 (lbm_tb2.cuh) on a binary16 lattice
// ------------------------------------------------------------------------------------
// Staged rows and ring rows are binary16: column j of the span at [LBM_TB2H_PAD + j].  The halo is
// LBM_TB2H_PAD columns on each side (K7: 4) so that every bulk copy starts on a 16-byte boundary in
// both memories.  Plane-rows of the accelerated side row, and the accelerated sub-step-1 row, are
// fp32 rows with column j at [4 + j].
#define LBM_TB2H_PAD 8
#define LBM_TB2H_ROWH (LBM_TB2_SPAN + 2 * LBM_TB2H_PAD)     /* 400 halves = 800 B */
#define LBM_TB2H_ROWF (LBM_TB2_SPAN + 8)                     /* 392 floats */
#define LBM_TB2H_MAX_WOUT (LBM_TB2_SPAN - 2 * LBM_TB2H_PAD) /* owned columns per strip */

struct Tb2hSmem {
  __half in[2][9][LBM_TB2H_ROWH];    // two stages of pulled plane-rows (bulk-copy destination)
  __half r013[2][3][LBM_TB2H_ROWH];  // sub-step-1 rows as stored: planes 0,1,3 (read one iteration later)
  __half r256[3][3][LBM_TB2H_ROWH];  // planes 2,5,6 (two iterations later)
  __half r78[2][LBM_TB2H_ROWH];      // planes 7,8 (the same iteration; plane 4 stays in registers)
  float side[2][2][LBM_TB2H_ROWF];   // per stage: the two plane-rows that come from the side row
  float acc[6][LBM_TB2H_ROWF];       // sub-step-1 row ny-2 after accelerate_flow, planes 1,3,5,6,7,8
  unsigned long long mbar[2];
  unsigned long long mbar_free;
};
static_assert(sizeof(Tb2hSmem) * LBM_TB2_MIN_BLOCKS <= 225 * 1024, "LBM_TB2_MIN_BLOCKS blocks of shared memory per SM");
static_assert((LBM_TB2H_ROWH * 2) % 16 == 0 && (LBM_TB2H_PAD * 2) % 16 == 0 && (LBM_TB2H_ROWF * 4) % 16 == 0,
              "staged rows and their first column must keep 16-byte alignment");

// bytes the copies of sub-step-1 row r bring: nine binary16 plane-rows, of which two are fp32 rows
// of the side row when r, r-1 or r+1 is row ny-2
__device__ __forceinline__ uint32_t tb2h_stage_bytes(const F16Args& a, const int r) {
  const bool side = wrap_row(r, a.rows) == a.accel_row || wrap_row(r - 1, a.rows) == a.accel_row ||
                    wrap_row(r + 1, a.rows) == a.accel_row;
  return (uint32_t)a.span * (side ? 22u : 18u);
}
__device__ __forceinline__ void tb2h_expect(Tb2hSmem& sm, const int stage, const uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&sm.mbar[stage])), "r"(bytes)
               : "memory");
}
// thread k < 9 copies plane k of the rows sub-step 1 on row r pulls from (see tb2_issue)
__device__ __forceinline__ void tb2h_issue(const F16Args& a, Tb2hSmem& sm, const int stage, const int r, const int s0,
                                           const int k) {
  if (k < 0) return;
  const int dy = (k == 2 || k == 5 || k == 6) ? -1 : (k == 4 || k == 7 || k == 8) ? 1 : 0;
  const int row = wrap_row(r + dy, a.rows);
  const bool side = (row == a.accel_row) && k != 0 && k != 2 && k != 4;
  const char* src;
  char* dst;
  uint32_t elem;
  if (side) {
    const int idx = (k == 1) ? 0 : (k == 3) ? 1 : k - 3;       // side row order 1,3,5,6,7,8
    src = (const char*)(a.side_src + (long long)idx * a.pitch);
    dst = (char*)&sm.side[stage][idx & 1][4];
    elem = 4;
  } else {
    src = (const char*)(a.src + (long long)k * a.plane_stride + (long long)row * a.pitch);
    dst = (char*)&sm.in[stage][k][LBM_TB2H_PAD];
    elem = 2;
  }
  int col = s0, left = a.span;
  while (left > 0) {
    const int n = min(left, a.nx - col);
    tb2_bulk_load((float*)dst, (const float*)(src + (size_t)col * elem), (uint32_t)n * elem, &sm.mbar[stage]);
    dst += (size_t)n * elem;
    left -= n;
    col = 0;
  }
}

// the four cells of a quad from a staged row: as stored / shifted one column (binary16, decoded)
__device__ __forceinline__ void h_get(const __half* row, const int c0, const float c, float& v0, float& v1, float& v2,
                                      float& v3) {
  const Vec4<float> v = dec4(*reinterpret_cast<const uint2*>(row + LBM_TB2H_PAD + c0), c);
  v0 = v.x; v1 = v.y; v2 = v.z; v3 = v.w;
}
__device__ __forceinline__ void h_get_west(const __half* row, const int c0, const float c, float& v0, float& v1,
                                           float& v2, float& v3) {
  const Vec4<float> v = dec4(*reinterpret_cast<const uint2*>(row + LBM_TB2H_PAD + c0), c);
  v0 = f16_dec(row[LBM_TB2H_PAD + c0 - 1], c); v1 = v.x; v2 = v.y; v3 = v.z;
}
__device__ __forceinline__ void h_get_east(const __half* row, const int c0, const float c, float& v0, float& v1,
                                           float& v2, float& v3) {
  const Vec4<float> v = dec4(*reinterpret_cast<const uint2*>(row + LBM_TB2H_PAD + c0), c);
  v0 = v.y; v1 = v.z; v2 = v.w; v3 = f16_dec(row[LBM_TB2H_PAD + c0 + 4], c);
}
// a plane-row that is binary16 (fp == nullptr) or an fp32 row, shifted west / east
__device__ __forceinline__ void hf_get_west(const __half* h, const float* fp, const int c0, const float c, float& v0,
                                            float& v1, float& v2, float& v3) {
  if (fp) tb2_get_west(fp, c0, v0, v1, v2, v3);
  else h_get_west(h, c0, c, v0, v1, v2, v3);
}
__device__ __forceinline__ void hf_get_east(const __half* h, const float* fp, const int c0, const float c, float& v0,
                                            float& v1, float& v2, float& v3) {
  if (fp) tb2_get_east(fp, c0, v0, v1, v2, v3);
  else h_get_east(h, c0, c, v0, v1, v2, v3);
}
__device__ __forceinline__ void h_put(__half* row, const int c0, const uint2 v) {
  *reinterpret_cast<uint2*>(row + LBM_TB2H_PAD + c0) = v;
}

template <bool STRICT>
__device__ __forceinline__ void tb2h_tile(const F16Args& a, Tb2hSmem& sm, const int strip, const int seg,
                                          unsigned long long& q1, unsigned long long& q2, bool& bad1, bool& bad2) {
  const int tid = threadIdx.x;
  const int X0 = strip * a.wout;                               // first owned column (a multiple of 8)
  const int S0 = (X0 >= LBM_TB2H_PAD) ? X0 - LBM_TB2H_PAD : X0 - LBM_TB2H_PAD + a.nx;
  const bool big = seg < a.n_big;
  const int R0 = big ? seg * a.seg_rows : a.big_rows + (seg - a.n_big) * a.seg_rows_tail;
  const int R1 = big ? min(R0 + a.seg_rows, a.big_rows) : min(R0 + a.seg_rows_tail, a.rows);
  const int n_it = R1 - R0 + 2;                                // sub-step-1 rows R0-1 .. R1

  const int c0 = min(4 * tid, a.span - 4);
  int xg = S0 + c0;
  while (xg >= a.nx) xg -= a.nx;
  const bool owned = (c0 >= LBM_TB2H_PAD) && (4 * tid < a.span) && (c0 - LBM_TB2H_PAD < a.wout) &&
                     (X0 + c0 - LBM_TB2H_PAD < a.nx);
  const float k0 = a.rest.w0, k1 = a.rest.w1, k2 = a.rest.w2;

  const int my_plane = tb2_plane_of_thread();
  if (tid == 0) { tb2h_expect(sm, 0, tb2h_stage_bytes(a, R0 - 1)); tb2h_expect(sm, 1, tb2h_stage_bytes(a, R0)); }
#pragma unroll 1
  for (int k = 0; k < 2; k++) tb2h_issue(a, sm, k, R0 - 1 + k, S0, my_plane);

  const QuadConsts<float, STRICT> qc(a.omega);
  const int mword_idx = xg >> 5, mshift = xg & 31;
  auto mask_bits = [&](const int row) -> uint32_t {
    return (a.mask[(long long)wrap_row(row, a.rows) * a.mask_pitch + mword_idx] >> mshift) & 0xFu;
  };
  uint32_t mbits = mask_bits(R0 - 1);
  uint32_t mbits_prev = 0u;
  uint32_t phases = 0u;

#pragma unroll 1
  for (int i = 0; i < n_it; i++) {
    const int st = i & 1;
    const int r = R0 - 1 + i;
    const int rw = wrap_row(r, a.rows);
    const uint32_t mbits_next = (i + 1 < n_it) ? mask_bits(r + 1) : 0u;
    float keep4[4];
    {
      // ---------------- sub-step 1 on row r: pulled values are staged in sm.in[st] / sm.side[st] ----
      tb2_mbar_wait(&sm.mbar[st], (phases >> st) & 1u);
      phases ^= 1u << st;
      if (tid == 0 && i + 2 < n_it) tb2h_expect(sm, st, tb2h_stage_bytes(a, r + 2));
      const bool cA = rw == a.accel_row, sA = wrap_row(r - 1, a.rows) == a.accel_row,
                 nA = wrap_row(r + 1, a.rows) == a.accel_row;
      float in[4][9], out[4][9];
      const __half(*row)[LBM_TB2H_ROWH] = sm.in[st];
      const float* sd0 = sm.side[st][0];
      const float* sd1 = sm.side[st][1];
      h_get(row[0], c0, k0, in[0][0], in[1][0], in[2][0], in[3][0]);
      h_get(row[2], c0, k1, in[0][2], in[1][2], in[2][2], in[3][2]);
      h_get(row[4], c0, k1, in[0][4], in[1][4], in[2][4], in[3][4]);
      hf_get_west(row[1], cA ? sd0 : nullptr, c0, k1, in[0][1], in[1][1], in[2][1], in[3][1]);
      hf_get_east(row[3], cA ? sd1 : nullptr, c0, k1, in[0][3], in[1][3], in[2][3], in[3][3]);
      hf_get_west(row[5], sA ? sd0 : nullptr, c0, k2, in[0][5], in[1][5], in[2][5], in[3][5]);
      hf_get_east(row[6], sA ? sd1 : nullptr, c0, k2, in[0][6], in[1][6], in[2][6], in[3][6]);
      hf_get_east(row[7], nA ? sd0 : nullptr, c0, k2, in[0][7], in[1][7], in[2][7], in[3][7]);
      hf_get_west(row[8], nA ? sd1 : nullptr, c0, k2, in[0][8], in[1][8], in[2][8], in[3][8]);
      bool bad;
      const unsigned long long q = quad_update<float, STRICT>(in, mbits, qc, out, bad);
      if (owned && r >= R0 && r < R1) { q1 += q; bad1 |= bad; }
      uint2 enc[9];
#pragma unroll
      for (int k = 0; k < 9; k++) enc[k] = enc4(out[0][k], out[1][k], out[2][k], out[3][k], a.rest.of(k));
      if (cA) {
        // accelerate_flow between the two steps, on the values as stored; kept in fp32.  acc is read
        // only while sub-step 2 works on rows ny-3 .. ny-1, never in the iteration that writes it
        const int ks[6] = {1, 3, 5, 6, 7, 8};
        float f[4][6];
#pragma unroll
        for (int j = 0; j < 4; j++) {
#pragma unroll
          for (int n = 0; n < 6; n++) f[j][n] = round_f16(out[j][ks[n]], a.rest.of(ks[n]));
          cell_accelerate<float, STRICT>(f[j][0], f[j][1], f[j][2], f[j][3], f[j][4], f[j][5], (mbits >> j) & 1u,
                                         a.aw1, a.aw2);
        }
#pragma unroll
        for (int n = 0; n < 6; n++)
          *reinterpret_cast<float4*>(&sm.acc[n][4 + c0]) = make_float4(f[0][n], f[1][n], f[2][n], f[3][n]);
      }
      if (i > 0) {
        tb2_mbar_wait(&sm.mbar_free, (phases >> 2) & 1u);
        phases ^= 4u;
      }
      h_put(sm.r013[i & 1][0], c0, enc[0]);
      h_put(sm.r013[i & 1][1], c0, enc[1]);
      h_put(sm.r013[i & 1][2], c0, enc[3]);
      h_put(sm.r256[i % 3][0], c0, enc[2]);
      h_put(sm.r256[i % 3][1], c0, enc[5]);
      h_put(sm.r256[i % 3][2], c0, enc[6]);
      h_put(sm.r78[0], c0, enc[7]);
      h_put(sm.r78[1], c0, enc[8]);
      const Vec4<float> v4 = dec4(enc[4], k1);                   // row r's plane 4 as stored
      keep4[0] = v4.x; keep4[1] = v4.y; keep4[2] = v4.z; keep4[3] = v4.w;
    }
    __syncthreads();          // ring rows of this iteration are complete; stage `st` has been read by everyone
    if (i + 2 < n_it) tb2h_issue(a, sm, st, r + 2, S0, my_plane);

    if (i >= 2) {
      // ---------------- sub-step 2 on row y = r - 1, pulling sub-step-1 rows y-1, y, y+1 ----
      const int y = r - 1;
      const bool cA = y == a.accel_row, sA = wrap_row(y - 1, a.rows) == a.accel_row, nA = rw == a.accel_row;
      float in[4][9], out[4][9];
      const __half(*c)[LBM_TB2H_ROWH] = sm.r013[(i - 1) & 1];  // row y
      const __half(*s)[LBM_TB2H_ROWH] = sm.r256[(i - 2) % 3];  // row y - 1
      h_get(c[0], c0, k0, in[0][0], in[1][0], in[2][0], in[3][0]);
      hf_get_west(c[1], cA ? sm.acc[0] : nullptr, c0, k1, in[0][1], in[1][1], in[2][1], in[3][1]);
      hf_get_east(c[2], cA ? sm.acc[1] : nullptr, c0, k1, in[0][3], in[1][3], in[2][3], in[3][3]);
      h_get(s[0], c0, k1, in[0][2], in[1][2], in[2][2], in[3][2]);
      hf_get_west(s[1], sA ? sm.acc[2] : nullptr, c0, k2, in[0][5], in[1][5], in[2][5], in[3][5]);
      hf_get_east(s[2], sA ? sm.acc[3] : nullptr, c0, k2, in[0][6], in[1][6], in[2][6], in[3][6]);
#pragma unroll
      for (int j = 0; j < 4; j++) in[j][4] = keep4[j];
      hf_get_east(sm.r78[0], nA ? sm.acc[4] : nullptr, c0, k2, in[0][7], in[1][7], in[2][7], in[3][7]);
      hf_get_west(sm.r78[1], nA ? sm.acc[5] : nullptr, c0, k2, in[0][8], in[1][8], in[2][8], in[3][8]);
      __syncwarp();
      if ((threadIdx.x & 31) == 0)
        asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&sm.mbar_free)) : "memory");
      bool bad;
      const unsigned long long q = quad_update<float, STRICT>(in, mbits_prev, qc, out, bad);
      if (owned) {
        q2 += q;
        bad2 |= bad;
        f16_store_quad<STRICT>(a, y, xg, out, mbits_prev);
      }
    } else {
      __syncwarp();             // one arrival per warp per iteration
      if ((threadIdx.x & 31) == 0)
        asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&sm.mbar_free)) : "memory");
    }
    mbits_prev = mbits;
    mbits = mbits_next;
  }
}

// the pads of every staged and ring row are read by the edge quads of the span (whose results are
// never used): keep them defined; then the barriers
__device__ __forceinline__ void tb2h_init_smem(Tb2hSmem& sm, const int span) {
  const int tid = threadIdx.x;
  for (int i = tid; i < 35 * 2 * LBM_TB2H_PAD; i += blockDim.x) {
    __half* row = &sm.in[0][0][0] + (size_t)(i / (2 * LBM_TB2H_PAD)) * LBM_TB2H_ROWH;
    const int e = i % (2 * LBM_TB2H_PAD);
    row[e < LBM_TB2H_PAD ? e : span + e] = __float2half_rn(0.f);
  }
  for (int i = tid; i < 10 * 8; i += blockDim.x) {
    float* row = &sm.side[0][0][0] + (size_t)(i / 8) * LBM_TB2H_ROWF;
    const int e = i % 8;
    row[e < 4 ? e : span + e] = 0.f;
  }
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&sm.mbar[0])) : "memory");
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&sm.mbar[1])) : "memory");
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(&sm.mbar_free)), "r"((uint32_t)(blockDim.x >> 5)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
}

template <bool STRICT>
__global__ void __launch_bounds__(LBM_TB2_THREADS, LBM_TB2_MIN_BLOCKS)
lbm_step2_tb_f16(const __grid_constant__ F16Args a) {
  extern __shared__ __align__(128) unsigned char tb2h_smem_raw[];
  Tb2hSmem& sm = *reinterpret_cast<Tb2hSmem*>(tb2h_smem_raw);
  int strip, seg;
  tile_of_block(a.tiles_x, a.tiles_y, 1, strip, seg);
  tb2h_init_smem(sm, a.span);
  cudaGridDependencySynchronize();           // PDL: the previous pass's writes are visible from here on
  __syncthreads();
  unsigned long long q1 = 0ULL, q2 = 0ULL;
  bool bad1 = false, bad2 = false;
  tb2h_tile<STRICT>(a, sm, strip, seg, q1, q2, bad1, bad2);
  if (bad1) atomicOr(a.av + 1, LBM_NONFINITE_MARK);
  if (bad2) atomicOr(a.av2 + 1, LBM_NONFINITE_MARK);
  block_accumulate(q1, a.av);
  __syncthreads();            // block_accumulate's shared scratch is reused
  block_accumulate(q2, a.av2);
}

// ------------------------------------------------------------------------------------
// the side row of the current state: row ny-2 decoded, then accelerate_flow (d2q9-bgk.c:229-260)
// ------------------------------------------------------------------------------------
__global__ void lbm_prepare_f16(const __half* __restrict__ cur, float* __restrict__ side, const uint32_t* __restrict__ mask,
                                long long plane_stride, int nx, int pitch, int mask_pitch, int accel_row, RestShift rest,
                                float aw1, float aw2) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= nx) return;
  const long long o = (long long)accel_row * pitch + x;
  float f[9];
#pragma unroll
  for (int k = 0; k < 9; k++) f[k] = f16_dec(cur[k * plane_stride + o], rest.of(k));
  const bool obst = (mask[(long long)accel_row * mask_pitch + (x >> 5)] >> (x & 31)) & 1u;
  cell_accelerate<float, true>(f[1], f[3], f[5], f[6], f[7], f[8], obst, aw1, aw2);
  side[0 * pitch + x] = f[1]; side[1 * pitch + x] = f[3];
  side[2 * pitch + x] = f[5]; side[3 * pitch + x] = f[6];
  side[4 * pitch + x] = f[7]; side[5 * pitch + x] = f[8];
}

}  // namespace lbm
