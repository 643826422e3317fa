// lbm_kernels.cuh -- sm_100a device code of the d2q9-bgk timestep loop.
//
// One fused kernel per timestep does what the reference's timestep_new2 does
// (d2q9-bgk.c:228-1813): accelerate_flow (:229-260), pull-propagate (:990-998),
// rebound (:971-981), BGK collision (:983-1100) and the av_velocity contribution
// (:1103-1130), plus -- new here -- the ghost-row push into the neighbouring slabs.
//
// Data layout in HBM (one "slab" = the rows one GPU holds, DESIGN.md section 3):
//   lattice  2 buffers x 9 planes x rows x pitch   structure-of-arrays;
//   window   ghost rows, 2 parities x 2 directions x 2 depths x 9 planes x pitch.  Direction
//            "from below" holds the rows under the slab's first row (depth 0 = row -1,
//            depth 1 = row -2), "from above" the rows over its last row (periodic in y, so
//            with one slab they are the slab's own opposite edge rows).  Written by the
//            NEIGHBOURS' step kernels (peer stores over NVLink), read by this slab's edge
//            rows.  The one-step kernels use speeds 2,5,6 / 4,7,8 of depth 0 only; the
//            two-step kernel (K7) also needs 0,1,3 of depth 0 and 2,5,6 / 4,7,8 of depth 1.
//            Behind them: the mask words of rows -1 and `rows`, and the sync words.  The
//            window is the only memory other GPUs / processes map;
//   mask     rows x pitch/32 uint32, bit = 1 for an obstacle cell;
//   side     2 x 6 x pitch: row ny-2 of planes 1,3,5,6,7,8 AFTER accelerate_flow.
//            The lattice itself always holds the un-accelerated state; readers that
//            pull from row ny-2 take those six planes from `side` instead.  This is
//            the same arithmetic as accelerating in place before streaming
//            (d2q9-bgk.c:229-260) without a separate kernel or a pre-pass.
#pragma once
#include <cuda.h>            // CUtensorMap (type only; the encoder is fetched at run time)
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

// Compile-time tuning knobs of the step kernels (defaults = the measured best, see
// profiles/r01_kernel_variants.md; tools/build_variants.py builds the alternatives).
#ifndef LBM_BLOCK_THREADS
#define LBM_BLOCK_THREADS 128       // threads per block of K1a/K1b/K5
#endif
#ifndef LBM_MIN_BLOCKS
#define LBM_MIN_BLOCKS 4            // K1a fp32: the packed collision wants ~100 registers; 7 blocks per SM (72
#endif                              // registers) spill: 78.7 GLUPS against 93.9 at 4 blocks (profiles/r02_kernel_variants.md)
#ifndef LBM_LOAD_MODE
#define LBM_LOAD_MODE 0             // 0 plain, 1 ld.global.cs (evict-first), 2 ld.global.nc, 3 nc + L1::no_allocate
#endif
#ifndef LBM_PERSIST_MIN_BLOCKS
#define LBM_PERSIST_MIN_BLOCKS 3    // K5: no spills; 1024^2 104 GLUPS against 75 at 6 blocks per SM (same file)
#endif
// Timing experiments that produce WRONG results exist only in builds made with
// -DLBM_EXPERIMENTS (tools/build_variants.py); the shipped library cannot contain them.
#ifdef LBM_EXPERIMENTS
#ifndef LBM_AV_MODE
#define LBM_AV_MODE 0               // 1 = no av sums
#endif
#ifndef LBM_K5_EXPERIMENT
#define LBM_K5_EXPERIMENT 0         // 1 = no grid barrier, 2 = barrier only
#endif
#else
#if defined(LBM_AV_MODE) || defined(LBM_K5_EXPERIMENT)
#error "LBM_AV_MODE / LBM_K5_EXPERIMENT need -DLBM_EXPERIMENTS: they produce wrong results"
#endif
#define LBM_AV_MODE 0
#define LBM_K5_EXPERIMENT 0
#endif
static_assert(
#ifdef LBM_EXPERIMENTS
    true ||
#endif
    (LBM_AV_MODE == 0 && LBM_K5_EXPERIMENT == 0), "the shipped build has every experiment switch off");
#ifndef LBM_STORE_MODE
#define LBM_STORE_MODE 0            // 0 plain, 1 st.global.cs (streaming), 2 st.global.cg
#endif
#ifndef LBM_BARRIER_MODE
#define LBM_BARRIER_MODE 1          // grid barrier of K5/K9: 1 = red.release + acquire spin; 0 = fence + atomic + spin + fence
                                    // (4-12 % slower per timestep on L2-resident grids, profiles/r02_kernel_variants.md)
#endif
#ifndef LBM_PACKED
#define LBM_PACKED 1                // default fp32 collision: 1 = packed f32x2 lanes (two cells per instruction),
#endif                              // 0 = the same operation sequence one cell at a time (same bits)

namespace lbm {

// ------------------------------------------------------------------------------------
// arithmetic policy.
//   STRICT   mirrors the reference's C expression trees with round-to-nearest single
//            operations (never contracted into FMA) so the result is bit-identical to a
//            gcc -O2 -ffp-contract=off build of d2q9-bgk.c:983-1128.
//   default  the same maths in an algebraically equal, cheaper form, written ONCE over a
//            "lane" type with explicit round-to-nearest add / mul / fma (nothing is left
//            to the compiler's contraction choices): Lane<float2> issues the packed
//            FADD2 / FMUL2 / FFMA2 of sm_100a -- two cells per instruction -- and
//            Lane<float> / Lane<double> are the one-cell forms of the SAME operation
//            sequence, so every kernel variant of one precision produces the same bits.
// ------------------------------------------------------------------------------------
template <typename real, bool STRICT> struct Ops;

template <> struct Ops<float, true> {
  static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
  static __device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
  static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
  static __device__ __forceinline__ float div(float a, float b) { return __fdiv_rn(a, b); }
  static __device__ __forceinline__ float sqrt(float a) { return __fsqrt_rn(a); }
};
template <> struct Ops<double, true> {
  static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
  static __device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
  static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
  static __device__ __forceinline__ double div(double a, double b) { return __ddiv_rn(a, b); }
  static __device__ __forceinline__ double sqrt(double a) { return __dsqrt_rn(a); }
};

__device__ __forceinline__ float rcp_approx(float x) {
  float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r;
}
__device__ __forceinline__ float sqrt_approx(float x) {
  float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r;
}

template <typename V> struct Lane;
template <> struct Lane<float> {
  typedef float S;
  static __device__ __forceinline__ float bc(float s) { return s; }
  static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
  static __device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
  static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
  static __device__ __forceinline__ float fma(float a, float b, float c) { return __fmaf_rn(a, b, c); }
  // -(1/x): hardware reciprocal (1 ulp) of -x plus one Newton step
  static __device__ __forceinline__ float nrcp(float x) {
    const float nr = rcp_approx(-x);
    return __fmaf_rn(nr, __fmaf_rn(x, nr, 1.0f), nr);
  }
};
template <> struct Lane<double> {
  typedef double S;
  static __device__ __forceinline__ double bc(double s) { return s; }
  static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
  static __device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
  static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
  static __device__ __forceinline__ double fma(double a, double b, double c) { return __fma_rn(a, b, c); }
  static __device__ __forceinline__ double nrcp(double x) { return __ddiv_rn(-1.0, x); }
};
#define LBM_F32X2_OP2(name, ptx)                                                                        \
  static __device__ __forceinline__ float2 name(float2 a, float2 b) {                                   \
    float2 d;                                                                                           \
    asm("{.reg .b64 ra, rb, rd; mov.b64 ra, {%2,%3}; mov.b64 rb, {%4,%5}; " ptx ".rn.f32x2 rd, ra, rb; " \
        "mov.b64 {%0,%1}, rd;}" : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));       \
    return d;                                                                                           \
  }
template <> struct Lane<float2> {
  typedef float S;
  static __device__ __forceinline__ float2 bc(float s) { return make_float2(s, s); }
  LBM_F32X2_OP2(add, "add")
  LBM_F32X2_OP2(sub, "sub")
  LBM_F32X2_OP2(mul, "mul")
  static __device__ __forceinline__ float2 fma(float2 a, float2 b, float2 c) {
    float2 d;
    asm("{.reg .b64 ra, rb, rc, rd; mov.b64 ra, {%2,%3}; mov.b64 rb, {%4,%5}; mov.b64 rc, {%6,%7}; "
        "fma.rn.f32x2 rd, ra, rb, rc; mov.b64 {%0,%1}, rd;}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
    return d;
  }
  static __device__ __forceinline__ float2 nrcp(float2 x) {
    const float2 nr = make_float2(rcp_approx(-x.x), rcp_approx(-x.y));
    return fma(nr, fma(x, nr, make_float2(1.0f, 1.0f)), nr);
  }
};
#undef LBM_F32X2_OP2

// loop-invariant operands of the default collision, broadcast to the lane type once per thread
template <typename V>
struct FastConsts {
  V keep, ow0, ow1, ow2, one, m15, three, mthree, f45;
  __device__ __forceinline__ explicit FastConsts(const typename Lane<V>::S omega) {
    typedef typename Lane<V>::S S;
    typedef Lane<V> L;
    keep = L::bc((S)1 - omega);
    ow0 = L::bc(omega * (S)(4.0 / 9.0));
    ow1 = L::bc(omega * (S)(1.0 / 9.0));
    ow2 = L::bc(omega * (S)(1.0 / 36.0));
    one = L::bc((S)1); m15 = L::bc((S)-1.5); three = L::bc((S)3); mthree = L::bc((S)-3); f45 = L::bc((S)4.5);
  }
};

// BGK collision (d2q9-bgk.c:983-1100) of one lane of cells, default arithmetic:
//   c_k = (1 - omega) p_k + omega w_k rho (1 + 3 u_k + 4.5 u_k^2 - 1.5 u^2)
// with one reciprocal instead of two divisions and 1/c_sq = 3, 1/(2 c_sq^2) = 4.5,
// 1/(2 c_sq) = 1.5.  Returns u^2 of the PULLED values.  BGK conserves mass and momentum, so
// this is also u^2 of the stored values (what d2q9-bgk.c:1103-1128 recomputes for the
// average) up to rounding -- the reference's own collision_and_vel (d2q9-bgk.c:2543) takes
// the average from the same place.  60 lane operations per call.
template <typename V>
__device__ __forceinline__ V collide_fast(const V (&p)[9], const FastConsts<V>& k, V (&c)[9]) {
  typedef Lane<V> L;
  const V e = L::add(L::add(p[1], p[5]), p[8]);
  const V w = L::add(L::add(p[3], p[6]), p[7]);
  const V n = L::add(L::add(p[2], p[5]), p[6]);
  const V s = L::add(L::add(p[4], p[7]), p[8]);
  const V rho = L::add(L::add(L::add(p[0], p[2]), L::add(p[4], e)), w);
  const V ninv = L::nrcp(rho);
  const V ux = L::mul(L::sub(w, e), ninv);
  const V uy = L::mul(L::sub(s, n), ninv);
  const V usq = L::fma(uy, uy, L::mul(ux, ux));
  const V base = L::fma(k.m15, usq, k.one);
  const V r1 = L::mul(rho, k.ow1), r2 = L::mul(rho, k.ow2);
  const V b0 = L::mul(L::mul(rho, k.ow0), base);
  const V b1 = L::mul(r1, base), l1 = L::mul(r1, k.three), n1 = L::mul(r1, k.mthree), q1 = L::mul(r1, k.f45);
  const V b2 = L::mul(r2, base), l2 = L::mul(r2, k.three), n2 = L::mul(r2, k.mthree), q2 = L::mul(r2, k.f45);
  const V upv = L::add(ux, uy), umv = L::sub(ux, uy);
  c[0] = L::fma(k.keep, p[0], b0);
  // omega w rho (base + 3 u + 4.5 u^2) = b + u (l + q u); the opposite direction takes l -> -l
#define LBM_DIR(kk, u, lin, quad, b) c[kk] = L::fma(k.keep, p[kk], L::fma(u, L::fma(quad, u, lin), b))
  LBM_DIR(1, ux, l1, q1, b1);  LBM_DIR(3, ux, n1, q1, b1);
  LBM_DIR(2, uy, l1, q1, b1);  LBM_DIR(4, uy, n1, q1, b1);
  LBM_DIR(5, upv, l2, q2, b2); LBM_DIR(7, upv, n2, q2, b2);
  LBM_DIR(8, umv, l2, q2, b2); LBM_DIR(6, umv, n2, q2, b2);
#undef LBM_DIR
  return usq;
}

__device__ __forceinline__ float speed_of(float usq) { return sqrt_approx(usq); }
__device__ __forceinline__ double speed_of(double usq) { return ::sqrt(usq); }

// |u| is accumulated as an exact 128-bit fixed-point sum (unit 2^-52): integer adds
// are associative, so the per-step average does not depend on block scheduling, grid
// shape or on how the rows are split over GPUs.
#define LBM_FIX_SCALE 4503599627370496.0 /* 2^52 */
// A cell whose |u| is NaN or beyond any physical value (the lattice has blown up; the speed
// of sound is 0.577) cannot be represented in the fixed-point sum: the step's high word gets
// this bit and the host reports that step's average as NaN, which is what the reference's
// float sum would give a few steps later at the latest.  Every kernel, in both builds, tests
// each fluid cell's |u| against it on its own (quad_sum_fixed, scalar_tile, K6), and so does
// the av_velocity read-out, so one lattice gives one NaN pattern.  The bound also keeps every
// per-thread partial sum (up to 4 cells x 256 rows) below 2^64; partial sums are split
// into 32-bit halves before they are added across threads.
#define LBM_SPEED_LIMIT 2.0
#define LBM_NONFINITE_MARK (1ULL << 63)
__device__ __forceinline__ unsigned long long to_fixed(float s) {
  return __float2ull_rn(s * 4503599627370496.0f);
}
__device__ __forceinline__ unsigned long long to_fixed(double s) {
  return __double2ull_rn(s * 4503599627370496.0);
}

// bounce-back of the pulled values (d2q9-bgk.c:971-981)
template <typename real>
__device__ __forceinline__ void cell_rebound(const real (&p)[9], real (&o)[9]) {
  o[0] = p[0]; o[1] = p[3]; o[2] = p[4]; o[3] = p[1]; o[4] = p[2];
  o[5] = p[7]; o[6] = p[8]; o[7] = p[5]; o[8] = p[6];
}

// ------------------------------------------------------------------------------------
// one cell: p[0..8] pulled values -> o[0..8] stored values, returns |u| of the stored
// values (0 for an obstacle cell).
// ------------------------------------------------------------------------------------
template <typename real, bool STRICT>
__device__ __forceinline__ real cell_update(const real (&p)[9], const bool obstacle, const real omega,
                                            real (&o)[9]) {
  typedef Ops<real, true> M;
  real c[9];
  real speed;
  if (STRICT) {
    // d2q9-bgk.c:983-1100, expression trees as written there
    const real c_sq = (real)1 / (real)3;
    const real w0 = (real)4 / (real)9;
    const real w1 = (real)1 / (real)9;
    const real w2 = (real)1 / (real)36;
    const real two_csq = (real)2 * c_sq;
    const real two_csq_csq = (real)2 * c_sq * c_sq;
    real rho = M::add((real)0, p[0]);
#pragma unroll
    for (int k = 1; k < 9; k++) rho = M::add(rho, p[k]);
    const real ux = M::div(M::sub(M::add(M::add(p[1], p[5]), p[8]), M::add(M::add(p[3], p[6]), p[7])), rho);
    const real uy = M::div(M::sub(M::add(M::add(p[2], p[5]), p[6]), M::add(M::add(p[4], p[7]), p[8])), rho);
    const real usq = M::add(M::mul(ux, ux), M::mul(uy, uy));
    real u[9];
    u[1] = ux;                 u[2] = uy;
    u[3] = -ux;                u[4] = -uy;
    u[5] = M::add(ux, uy);     u[6] = M::add(-ux, uy);
    u[7] = M::sub(-ux, uy);    u[8] = M::sub(ux, uy);
    const real t_usq = M::div(usq, two_csq);
    real d[9];
    d[0] = M::mul(M::mul(w0, rho), M::sub((real)1, t_usq));
#pragma unroll
    for (int k = 1; k < 9; k++) {
      const real w = (k < 5) ? w1 : w2;
      const real poly = M::sub(M::add(M::add((real)1, M::div(u[k], c_sq)),
                                      M::div(M::mul(u[k], u[k]), two_csq_csq)), t_usq);
      d[k] = M::mul(M::mul(w, rho), poly);
    }
#pragma unroll
    for (int k = 0; k < 9; k++) c[k] = M::add(p[k], M::mul(omega, M::sub(d[k], p[k])));
    // d2q9-bgk.c:1103-1128: velocity recomputed from the values just stored
    real rho2 = M::add((real)0, c[0]);
#pragma unroll
    for (int k = 1; k < 9; k++) rho2 = M::add(rho2, c[k]);
    const real vx = M::div(M::sub(M::add(M::add(c[1], c[5]), c[8]), M::add(M::add(c[3], c[6]), c[7])), rho2);
    const real vy = M::div(M::sub(M::add(M::add(c[2], c[5]), c[6]), M::add(M::add(c[4], c[7]), c[8])), rho2);
    speed = M::sqrt(M::add(M::mul(vx, vx), M::mul(vy, vy)));
  } else {
    const FastConsts<real> k(omega);
    speed = speed_of(collide_fast<real>(p, k, c));
  }
  if (obstacle) {
    cell_rebound<real>(p, o);
    return (real)0;
  }
#pragma unroll
  for (int k = 0; k < 9; k++) o[k] = c[k];
  return speed;
}

// Four neighbouring cells of one thread (the unit of the vectorised kernels): in[j] pulled
// values of cell j, bit j of `obits` set for an obstacle (or padding) cell.  Returns the
// quad's contribution to the step's fixed-point |u| sum; `bad` is set when a speed is NaN
// or beyond LBM_SPEED_LIMIT.  Default fp32 build: the cells go through the packed lanes as
// the pairs (0,1) and (2,3), the rare obstacle cells are patched afterwards, and the four
// speeds are added as floats -- (s0 + s1) + (s2 + s3), a fixed order on a fixed, aligned set
// of cells, so the sum does not depend on the decomposition -- and converted once.
template <typename real, bool STRICT> struct QuadConsts {
  real omega;
  __device__ __forceinline__ explicit QuadConsts(real om) : omega(om) {}
};
template <> struct QuadConsts<float, false> {
#if LBM_PACKED
  FastConsts<float2> k;
#else
  FastConsts<float> k;
#endif
  __device__ __forceinline__ explicit QuadConsts(float om) : k(om) {}
};
template <> struct QuadConsts<double, false> {
  FastConsts<double> k;
  __device__ __forceinline__ explicit QuadConsts(double om) : k(om) {}
};

// Every cell is held to LBM_SPEED_LIMIT on its own, as in the strict build and in av_velocity:
// a bound on the quad's sum would let one cell of up to four times the limit through.  The
// compares are written so that a NaN speed fails them (fmaxf would drop it).  With each speed
// below 2 the quad's sum stays below 8, which is the headroom the fixed-point sum relies on.
template <typename real>
__device__ __forceinline__ unsigned long long quad_sum_fixed(real s0, real s1, real s2, real s3, bool& bad) {
  typedef Ops<real, true> M;
  const real L = (real)LBM_SPEED_LIMIT;
  bad = !(s0 < L && s1 < L && s2 < L && s3 < L);
  return to_fixed(M::add(M::add(s0, s1), M::add(s2, s3)));
}

template <typename real, bool STRICT>
__device__ __forceinline__ unsigned long long quad_update(const real (&in)[4][9], const uint32_t obits,
                                                          const QuadConsts<real, STRICT>& qc, real (&out)[4][9],
                                                          bool& bad) {
  if constexpr (STRICT) {
    unsigned long long q = 0ULL;
    bad = false;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const real s = cell_update<real, true>(in[j], (obits >> j) & 1u, qc.omega, out[j]);
      q += to_fixed(s);
      bad |= !(s < (real)LBM_SPEED_LIMIT);
    }
    return q;
  } else {
    real s[4];
    if constexpr (sizeof(real) == 4 && LBM_PACKED) {
#pragma unroll
      for (int h = 0; h < 2; h++) {
        float2 p[9], c[9];
#pragma unroll
        for (int k = 0; k < 9; k++) p[k] = make_float2(in[2 * h][k], in[2 * h + 1][k]);
        const float2 usq = collide_fast<float2>(p, qc.k, c);
#pragma unroll
        for (int k = 0; k < 9; k++) { out[2 * h][k] = c[k].x; out[2 * h + 1][k] = c[k].y; }
        s[2 * h] = speed_of(usq.x);
        s[2 * h + 1] = speed_of(usq.y);
      }
    } else {
#pragma unroll
      for (int j = 0; j < 4; j++) s[j] = speed_of(collide_fast<real>(in[j], qc.k, out[j]));
    }
    if (obits != 0u) {            // rare: walls, the 1 % random obstacles of the synthetic channel
#pragma unroll
      for (int j = 0; j < 4; j++)
        if ((obits >> j) & 1u) { cell_rebound<real>(in[j], out[j]); s[j] = (real)0; }
    }
    return quad_sum_fixed<real>(s[0], s[1], s[2], s[3], bad);
  }
}

// accelerate_flow on one cell's speeds (d2q9-bgk.c:246-258); a[] = {f1,f3,f5,f6,f7,f8}.
template <typename real, bool STRICT>
__device__ __forceinline__ void cell_accelerate(real& f1, real& f3, real& f5, real& f6, real& f7, real& f8,
                                                const bool obstacle, const real aw1, const real aw2) {
  typedef Ops<real, true> M;   // single adds/subs: nothing to contract, always exact ops
  const bool go = !obstacle && M::sub(f3, aw1) > (real)0 && M::sub(f6, aw2) > (real)0 &&
                  M::sub(f7, aw2) > (real)0;
  if (go) {
    f1 = M::add(f1, aw1); f5 = M::add(f5, aw2); f8 = M::add(f8, aw2);
    f3 = M::sub(f3, aw1); f6 = M::sub(f6, aw2); f7 = M::sub(f7, aw2);
  }
}

// |u| etc. of a stored cell (d2q9-bgk.c:2681-2705 / :2948-2972), reference tree order.
template <typename real>
__device__ __forceinline__ real cell_macroscopic(const real (&f)[9], real& ux, real& uy, real& rho) {
  typedef Ops<real, true> M;
  rho = M::add((real)0, f[0]);
#pragma unroll
  for (int k = 1; k < 9; k++) rho = M::add(rho, f[k]);
  ux = M::div(M::sub(M::add(M::add(f[1], f[5]), f[8]), M::add(M::add(f[3], f[6]), f[7])), rho);
  uy = M::div(M::sub(M::add(M::add(f[2], f[5]), f[6]), M::add(M::add(f[4], f[7]), f[8])), rho);
  return M::sqrt(M::add(M::mul(ux, ux), M::mul(uy, uy)));
}

// ------------------------------------------------------------------------------------
// kernel arguments
// ------------------------------------------------------------------------------------
template <typename real>
struct StepArgs {
  const real* src;             // lattice buffer read this step (plane 0, local row 0)
  real* dst;                   // lattice buffer written this step
  const real* side_src;        // accelerated row ny-2, planes {1,3,5,6,7,8} x pitch (read)
  real* side_dst;              // same, written for the next step
  const uint32_t* mask;        // rows x mask_pitch words
  unsigned long long* av;      // this step's |u| sums: LBM_AV_SLOTS lines of {low halves, high halves, pad}
  // ghost rows, see "window" above: plane k of depth d at (d * 9 + k) * pitch
  const real* ghost_s;         // own window, src parity, "from below" (row -1, row -2)
  const real* ghost_n;         // own window, src parity, "from above" (row rows, row rows+1)
  real* push_up;               // neighbour above's window, dst parity, "from below"
  real* push_dn;               // neighbour below's window, dst parity, "from above"
  // cross-slab ordering (only when MULTI): counters of completed PASSES (kernel launches)
  volatile unsigned long long* flag_from_below;  // local: passes completed by neighbour below
  volatile unsigned long long* flag_from_above;
  unsigned long long* up_flag;                   // neighbour above's flag_from_below
  unsigned long long* dn_flag;                   // neighbour below's flag_from_above
  unsigned long long* boundary_done;             // local counter of finished boundary blocks
  unsigned long long* abort_word;                // local: non-zero = give up (set by a neighbour or a time-out)
  unsigned long long* up_abort;                  // the neighbours' abort words
  unsigned long long* dn_abort;
  unsigned long long pass;                       // index of this pass (0-based, since creation)
  unsigned long long timeout_ns;                 // longest wait for a neighbour
  long long plane_stride;      // rows * pitch
  int nx;
  int rows;                    // local rows
  int pitch;                   // elements per row, multiple of 32
  int mask_pitch;              // words per mask row
  int accel_row;               // local row holding global row ny-2, or LBM_NO_ROW
  int tiles_x, tiles_y;
  int edge_tiles;              // tile rows at each end of the slab that touch ghost rows (1; 2 with deep pushes)
  int deep;                    // also push what the two-step kernel reads: planes 0,1,3 of the edge rows and the second rows
  real omega;
  real aw1, aw2;               // density*accel/9, density*accel/36 (d2q9-bgk.c:230-231)
};

// offset (in elements) of a section of the ghost rows inside the window
__host__ __device__ inline size_t ghost_offset(int pitch, int parity, int dir) {
  return (size_t)((parity * 2 + dir) * 18) * (size_t)pitch;
}
#define LBM_GHOST_PLANE_ROWS 72          /* 2 parities x 2 directions x 2 depths x 9 planes */

#define LBM_NO_ROW (-1000)

template <typename real> struct alignas(4 * sizeof(real)) Vec4 { real x, y, z, w; };

__device__ __forceinline__ Vec4<float> ld4(const float* p) {
#if LBM_LOAD_MODE == 1
  const float4 t = __ldcs(reinterpret_cast<const float4*>(p));
#elif LBM_LOAD_MODE == 2
  const float4 t = __ldg(reinterpret_cast<const float4*>(p));
#elif LBM_LOAD_MODE == 3
  float4 t;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(t.x), "=f"(t.y), "=f"(t.z), "=f"(t.w) : "l"(p));
#else
  const float4 t = *reinterpret_cast<const float4*>(p);
#endif
  Vec4<float> v; v.x = t.x; v.y = t.y; v.z = t.z; v.w = t.w;
  return v;
}
__device__ __forceinline__ Vec4<double> ld4(const double* p) { return *reinterpret_cast<const Vec4<double>*>(p); }
__device__ __forceinline__ void st4(float* p, const Vec4<float>& v) {
#if LBM_STORE_MODE == 1
  __stcs(reinterpret_cast<float4*>(p), make_float4(v.x, v.y, v.z, v.w));
#elif LBM_STORE_MODE == 2
  __stcg(reinterpret_cast<float4*>(p), make_float4(v.x, v.y, v.z, v.w));
#else
  *reinterpret_cast<Vec4<float>*>(p) = v;
#endif
}
__device__ __forceinline__ void st4(double* p, const Vec4<double>& v) { *reinterpret_cast<Vec4<double>*>(p) = v; }

// L2-only loads (ld.global.cg): the persistent kernel re-reads, step after step, memory
// that other SMs wrote in the previous step, so nothing may be served from a stale L1 line.
__device__ __forceinline__ Vec4<float> ld4cg(const float* p) {
  const float4 t = __ldcg(reinterpret_cast<const float4*>(p));
  Vec4<float> v; v.x = t.x; v.y = t.y; v.z = t.z; v.w = t.w;
  return v;
}
__device__ __forceinline__ Vec4<double> ld4cg(const double* p) {
  const double2 a = __ldcg(reinterpret_cast<const double2*>(p));
  const double2 b = __ldcg(reinterpret_cast<const double2*>(p) + 1);
  Vec4<double> v; v.x = a.x; v.y = a.y; v.z = b.x; v.w = b.y;
  return v;
}
template <typename real, bool CG>
__device__ __forceinline__ Vec4<real> load4(const real* p) { return CG ? ld4cg(p) : ld4(p); }
template <typename real, bool CG>
__device__ __forceinline__ real load1(const real* p) { return CG ? __ldcg(p) : *p; }

__device__ __forceinline__ unsigned long long ld_acquire_sys(const volatile unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// Exact sum of the per-thread fixed-point |u| (unit 2^-52).  A per-thread partial sum q is
// below 2^63 (LBM_SPEED_LIMIT).  It is cut into three pieces of 26 + 26 + 11 bits, each piece
// is added over the warp with ONE redux.sync (the 32-lane sums fit 32 bits), and lane 0 folds
// them into a pair {lo, hi} with value = hi * 2^32 + lo.  Pairs are added to the step's
// accumulators with two fire-and-forget atomics (RED) on two 64-bit words: no carry to
// propagate, no return value to wait for, no overflow whatever the block or grid size.
// LBM_AV_SLOTS such pairs per step, each in its own 128-byte line: one L2 line takes only
// about 0.47 G atomics/s (measured).
//   block_accumulate  one pair of atomics per block (shared memory + __syncthreads): the
//                     per-step kernels, where a 16384^2 step has 2.1 M warps -- one pair
//                     per WARP was measured 8 % slower there (L2 atomic traffic);
//   warp_accumulate   one pair per warp, no barrier: the persistent kernel, few warps and
//                     a grid barrier right behind (128^2: 3.0 -> 2.6 us per step).
#define LBM_AV_SLOTS 8
#define LBM_AV_STRIDE 16                 /* words between slots: one 128-byte line each */

struct AvPair { unsigned long long lo, hi; };

__device__ __forceinline__ AvPair warp_reduce_fixed(const unsigned long long q) {
  const unsigned a = __reduce_add_sync(0xffffffffu, (unsigned)(q & 0x3ffffffULL));
  const unsigned b = __reduce_add_sync(0xffffffffu, (unsigned)((q >> 26) & 0x3ffffffULL));
  const unsigned c = __reduce_add_sync(0xffffffffu, (unsigned)(q >> 52));
  // a + b 2^26 + c 2^52 = lo + hi 2^32 with lo < 2^33: the accumulator words take millions of
  // such pairs per step without wrapping
  AvPair r;
  r.lo = (unsigned long long)a + ((unsigned long long)(b & 0x3fu) << 26);
  r.hi = (unsigned long long)(b >> 6) + ((unsigned long long)c << 20);
  return r;
}

__device__ __forceinline__ void av_add(const AvPair v, unsigned long long* av_step, const unsigned slot) {
  unsigned long long* p = av_step + LBM_AV_STRIDE * (slot & (LBM_AV_SLOTS - 1));
  if (v.lo) atomicAdd(p, v.lo);
  if (v.hi) atomicAdd(p + 1, v.hi);
}

__device__ __forceinline__ void warp_accumulate(unsigned long long q, unsigned long long* av_step) {
#if LBM_AV_MODE == 1
  if (q == 0xffffffffffffffffULL) *av_step = q;   // keeps q alive, never true
  return;
#endif
  const AvPair v = warp_reduce_fixed(q);
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  if ((tid & 31) == 0) av_add(v, av_step, blockIdx.x + (tid >> 5));
}

__device__ __forceinline__ void block_accumulate(unsigned long long q, unsigned long long* av_step) {
#if LBM_AV_MODE == 1
  if (q == 0xffffffffffffffffULL) *av_step = q;   // keeps q alive, never true
  return;
#endif
  __shared__ AvPair warp_sums[32];
  const AvPair v = warp_reduce_fixed(q);
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  const int nwarps = (blockDim.x * blockDim.y + 31) >> 5;
  if ((tid & 31) == 0) warp_sums[tid >> 5] = v;
  __syncthreads();
  if (tid == 0) {
    AvPair t = warp_sums[0];
    for (int i = 1; i < nwarps; i++) { t.lo += warp_sums[i].lo; t.hi += warp_sums[i].hi; }
    av_add(t, av_step, blockIdx.x);
  }
}

// After a run: fold the LBM_AV_SLOTS padded slots of every step into one {low, high} pair,
// so that 16 bytes per step cross PCIe instead of 1 KiB.  The non-finite mark (bit 63 of a
// high word) is OR-ed, everything else summed.
__global__ void lbm_compact_av(const unsigned long long* __restrict__ av, unsigned long long* __restrict__ out,
                               int n_steps) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_steps) return;
  const unsigned long long* p = av + (size_t)t * (LBM_AV_STRIDE * LBM_AV_SLOTS);
  unsigned long long lo = 0ULL, hi = 0ULL, mark = 0ULL;
#pragma unroll
  for (int k = 0; k < LBM_AV_SLOTS; k++) {
    lo += p[LBM_AV_STRIDE * k];
    const unsigned long long h = p[LBM_AV_STRIDE * k + 1];
    hi += h & ~LBM_NONFINITE_MARK;
    mark |= h & LBM_NONFINITE_MARK;
  }
  out[2 * t] = lo;
  out[2 * t + 1] = hi | mark;
}

// Block -> tile mapping.  The `edge` tile rows at each end of the slab (those that read
// ghost rows or push into the neighbours) get the lowest block indices so that they are
// dispatched first: their pushes leave early and the neighbours' next pass never waits.
__device__ __forceinline__ void tile_of_block(const int tiles_x, const int tiles_y, const int edge, int& tx, int& ty) {
  const unsigned b = blockIdx.x;
  const int slot = (int)(b / (unsigned)tiles_x);
  tx = (int)(b - (unsigned)slot * (unsigned)tiles_x);
  if (tiles_y < 2 * edge) ty = slot;                       // tiny slab: every tile row is an edge
  else if (slot < edge) ty = slot;
  else if (slot < 2 * edge) ty = tiles_y - 1 - (slot - edge);
  else ty = slot - edge;
}
__device__ __forceinline__ bool is_edge_tile(const int ty, const int tiles_y, const int edge) {
  return (ty < edge) || (ty >= tiles_y - edge);
}
__host__ __device__ inline unsigned long long edge_tile_count(int tiles_x, int tiles_y, int edge) {
  return (unsigned long long)tiles_x * (unsigned long long)(tiles_y < 2 * edge ? tiles_y : 2 * edge);
}

__device__ __forceinline__ unsigned long long global_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

// error codes left in the sync block for the host (kSyncError)
#define LBM_SYNC_TIMEOUT 1ULL
#define LBM_SYNC_ABORTED 2ULL
#define LBM_SYNC_TILE_TIMEOUT 3ULL    /* K10: a neighbour tile of the previous pass never completed */

// Wait until both neighbours have completed `pass` passes.  The wait is bounded: when a
// neighbour does not arrive within timeout_ns (its process died, or it was asked for a
// different number of steps), or when the abort word is set, the block records the reason,
// raises the abort word here AND in both neighbours (so that the whole ring drains instead
// of every slab timing out in turn), and carries on -- the results of this run are void and
// lbm_gpu_run reports the failure (the reference's convention is die(), d2q9-bgk.c:3001).
template <typename real, bool MULTI>
__device__ __forceinline__ void boundary_wait(const StepArgs<real>& a, const bool is_boundary) {
  if (MULTI && is_boundary) {
    if (threadIdx.x == 0 && threadIdx.y == 0) {
      const unsigned long long t0 = global_timer_ns();
      unsigned long long why = 0ULL;
      while (ld_acquire_sys(a.flag_from_below) < a.pass || ld_acquire_sys(a.flag_from_above) < a.pass) {
        if (ld_acquire_sys(a.abort_word) != 0ULL) { why = LBM_SYNC_ABORTED; break; }
        if (global_timer_ns() - t0 > a.timeout_ns) { why = LBM_SYNC_TIMEOUT; break; }
      }
      if (why != 0ULL) {
        atomicCAS(a.abort_word + 1, 0ULL, (why << 56) | (a.pass & 0xffffffffffffffULL));   // first reason wins
        st_release_sys(a.abort_word, 1ULL);
        st_release_sys(a.up_abort, 1ULL);
        st_release_sys(a.dn_abort, 1ULL);
      }
    }
    __syncthreads();
  }
}

template <typename real, bool MULTI>
__device__ __forceinline__ void boundary_signal(const StepArgs<real>& a, const bool is_boundary) {
  if (MULTI && is_boundary) {
    __threadfence_system();            // this thread's ghost-row pushes are visible system-wide
    __syncthreads();
    if (threadIdx.x == 0 && threadIdx.y == 0) {
      // the last edge block of this pass publishes it.  The counter restarts from zero for the
      // next pass, whose kernel may have another number of edge blocks (K7 and K1a alternate);
      // that kernel's blocks count only after this grid has completed (stream order, or
      // cudaGridDependencySynchronize under programmatic launch).
      const unsigned long long nb = edge_tile_count(a.tiles_x, a.tiles_y, a.edge_tiles);
      const unsigned long long old = atomicAdd(a.boundary_done, 1ULL);
      if (old + 1ULL == nb) {
        atomicExch(a.boundary_done, 0ULL);
        __threadfence_system();
        st_release_sys(a.up_flag, a.pass + 1ULL);
        st_release_sys(a.dn_flag, a.pass + 1ULL);
      }
    }
  }
}

// End of a run: one thread waits (bounded, like boundary_wait) until both neighbours have
// completed `pass` passes too.  After it nothing of this run is still in flight towards this
// slab's window, so the host may destroy, upload or re-create without a barrier of its own.
template <typename real>
__global__ void lbm_wait_neighbours(const StepArgs<real> a) {
  boundary_wait<real, true>(a, true);
}

// ------------------------------------------------------------------------------------
// K1a  lbm_step_vec4: four cells per thread, 128-bit loads/stores straight from/to the
// SoA planes (any nx: rows are padded to the pitch, a multiple of 32 elements).  x-shifted planes come from the aligned vector plus one
// element of the neighbouring lane (warp shuffle); the two edge lanes of a warp fetch
// that element with a scalar load that also implements the periodic wrap in x.
// blockDim = (BX, BY), BX a multiple of 32 so that a warp never spans two rows.
// ------------------------------------------------------------------------------------
// The pull of one quad (d2q9-bgk.c:990-998 for four neighbouring cells): cells xc..xc+3 of
// local row rc, nine aligned 128-bit loads plus the two x-shift elements from the
// neighbouring lanes.  Every thread of the warp must call it (shuffles); `mbits` are the
// quad's mask bits, `obits` those plus the padding cells of a ragged width.
template <typename real, bool CG>
__device__ __forceinline__ void vec4_pull(const StepArgs<real>& a, const int rc, const int xc, real (&in)[4][9],
                                          uint32_t& mbits, uint32_t& obits) {
  const int lane = threadIdx.x & 31;
  const long long PS = a.plane_stride;
  const long long oC = (long long)rc * a.pitch;

  // Row sources.  South/north neighbours of the slab's first/last row live in the ghost
  // rows; planes 1,3 of the centre row / 5,6 of the south row / 7,8 of the north row
  // come from the accelerated side row when that row is global row ny-2 (the ghost rows
  // already hold accelerated values).  All of this is warp-uniform, and all but five
  // rows of a slab take the first branch.
  const bool first = (rc == 0), last = (rc == a.rows - 1);
  const bool cA = (rc == a.accel_row), sA = (rc - 1 == a.accel_row), nA = (rc + 1 == a.accel_row);
  const real *p0, *p1, *p2, *p3, *p4, *p5, *p6, *p7, *p8;
  {
    const real* c = a.src + oC;
    const real* sr = c - a.pitch;
    const real* nr = c + a.pitch;
    p0 = c;          p1 = c + PS;      p3 = c + 3 * PS;
    p2 = sr + 2 * PS; p5 = sr + 5 * PS; p6 = sr + 6 * PS;
    p4 = nr + 4 * PS; p7 = nr + 7 * PS; p8 = nr + 8 * PS;
  }
  if (first | last | cA | sA | nA) {
    if (cA) { p1 = a.side_src + 0 * a.pitch; p3 = a.side_src + 1 * a.pitch; }
    if (sA) { p5 = a.side_src + 2 * a.pitch; p6 = a.side_src + 3 * a.pitch; }
    if (nA) { p7 = a.side_src + 4 * a.pitch; p8 = a.side_src + 5 * a.pitch; }
    if (first) { p2 = a.ghost_s + 2 * a.pitch; p5 = a.ghost_s + 5 * a.pitch; p6 = a.ghost_s + 6 * a.pitch; }
    if (last) { p4 = a.ghost_n + 4 * a.pitch; p7 = a.ghost_n + 7 * a.pitch; p8 = a.ghost_n + 8 * a.pitch; }
  }

  // edge elements first (scalar, predicated), then the nine aligned vectors
  const bool need_w = (lane == 0) || (xc == 0);
  const bool need_e = (lane == 31) || (xc + 4 >= a.nx);
  const int xw = (xc == 0) ? a.nx - 1 : xc - 1;
  const int xe = (xc + 4 >= a.nx) ? 0 : xc + 4;
  real w1e = 0, w5e = 0, w8e = 0, e3e = 0, e6e = 0, e7e = 0;
  if (need_w) { w1e = load1<real, CG>(p1 + xw); w5e = load1<real, CG>(p5 + xw); w8e = load1<real, CG>(p8 + xw); }
  if (need_e) { e3e = load1<real, CG>(p3 + xe); e6e = load1<real, CG>(p6 + xe); e7e = load1<real, CG>(p7 + xe); }

  const Vec4<real> v0 = load4<real, CG>(p0 + xc), v1 = load4<real, CG>(p1 + xc), v2 = load4<real, CG>(p2 + xc),
                   v3 = load4<real, CG>(p3 + xc), v4 = load4<real, CG>(p4 + xc), v5 = load4<real, CG>(p5 + xc),
                   v6 = load4<real, CG>(p6 + xc), v7 = load4<real, CG>(p7 + xc), v8 = load4<real, CG>(p8 + xc);
  const uint32_t mword = a.mask[(long long)rc * a.mask_pitch + (xc >> 5)];
  mbits = (mword >> (xc & 31)) & 0xFu;

  // element x0-1 of planes 1,5,8 and x0+4 of planes 3,6,7 from the neighbouring lanes
  real l1 = __shfl_up_sync(0xffffffffu, v1.w, 1), l5 = __shfl_up_sync(0xffffffffu, v5.w, 1),
       l8 = __shfl_up_sync(0xffffffffu, v8.w, 1);
  real r3 = __shfl_down_sync(0xffffffffu, v3.x, 1), r6 = __shfl_down_sync(0xffffffffu, v6.x, 1),
       r7 = __shfl_down_sync(0xffffffffu, v7.x, 1);
  l1 = need_w ? w1e : l1; l5 = need_w ? w5e : l5; l8 = need_w ? w8e : l8;
  r3 = need_e ? e3e : r3; r6 = need_e ? e6e : r6; r7 = need_e ? e7e : r7;

  // Widths that are not a multiple of 4: the row's last thread holds 1-3 valid cells, the
  // rest of its vector is row padding (loaded and stored, never used).  The east neighbour
  // of the last valid cell is column 0 -- the wrap element r3/r6/r7 already holds -- and the
  // padding cells are treated as obstacles so that they add nothing to the average.
  const int nvalid = a.nx - xc;
  const bool n1 = (nvalid == 1), n2 = (nvalid == 2), n3 = (nvalid == 3);
  obits = (nvalid < 4) ? (mbits | ((0xFu << nvalid) & 0xFu)) : mbits;

  in[0][0] = v0.x; in[1][0] = v0.y; in[2][0] = v0.z; in[3][0] = v0.w;
  in[0][1] = l1;   in[1][1] = v1.x; in[2][1] = v1.y; in[3][1] = v1.z;
  in[0][2] = v2.x; in[1][2] = v2.y; in[2][2] = v2.z; in[3][2] = v2.w;
  in[0][3] = n1 ? r3 : v3.y; in[1][3] = n2 ? r3 : v3.z; in[2][3] = n3 ? r3 : v3.w; in[3][3] = r3;
  in[0][4] = v4.x; in[1][4] = v4.y; in[2][4] = v4.z; in[3][4] = v4.w;
  in[0][5] = l5;   in[1][5] = v5.x; in[2][5] = v5.y; in[3][5] = v5.z;
  in[0][6] = n1 ? r6 : v6.y; in[1][6] = n2 ? r6 : v6.z; in[2][6] = n3 ? r6 : v6.w; in[3][6] = r6;
  in[0][7] = n1 ? r7 : v7.y; in[1][7] = n2 ? r7 : v7.z; in[2][7] = n3 ? r7 : v7.w; in[3][7] = r7;
  in[0][8] = l8;   in[1][8] = v8.x; in[2][8] = v8.y; in[3][8] = v8.z;
}

template <typename real, bool STRICT, bool CG>
__device__ __forceinline__ unsigned long long vec4_tile(const StepArgs<real>& a, const QuadConsts<real, STRICT>& qc,
                                                        const int tx, const int ty) {
  const int x0 = (tx * (int)blockDim.x + (int)threadIdx.x) * 4;
  const int r = ty * (int)blockDim.y + (int)threadIdx.y;        // local row
  const bool active = (x0 < a.nx) && (r < a.rows);

  // clamp so that inactive threads still form valid addresses (they take part in the
  // shuffles but never store)
  const int xc = active ? x0 : 0;
  const int rc = active ? r : 0;
  const long long PS = a.plane_stride;
  const long long oC = (long long)rc * a.pitch;
  const bool first = (rc == 0), last = (rc == a.rows - 1), cA = (rc == a.accel_row);

  real in[4][9], out[4][9];
  uint32_t mbits, obits;
  vec4_pull<real, CG>(a, rc, xc, in, mbits, obits);

  bool bad;
  unsigned long long q = quad_update<real, STRICT>(in, obits, qc, out, bad);
  if (!active) return 0ULL;
  if (bad) atomicOr(a.av + 1, LBM_NONFINITE_MARK);            // NaN / blow-up

  real* d = a.dst + oC + xc;
#pragma unroll
  for (int k = 0; k < 9; k++) {
    Vec4<real> v; v.x = out[0][k]; v.y = out[1][k]; v.z = out[2][k]; v.w = out[3][k];
    st4(d + k * PS, v);
  }
  const bool second = a.deep && (rc == 1), before_last = a.deep && (rc == a.rows - 2);
  if (first | last | cA | second | before_last) {          // warp-uniform: a warp never spans two rows
    if (cA) {
      // next step's accelerate_flow on the row just produced (d2q9-bgk.c:229-260)
#pragma unroll
      for (int j = 0; j < 4; j++)
        cell_accelerate<real, STRICT>(out[j][1], out[j][3], out[j][5], out[j][6], out[j][7], out[j][8],
                                      (mbits >> j) & 1u, a.aw1, a.aw2);
      const int ks[6] = {1, 3, 5, 6, 7, 8};
#pragma unroll
      for (int i = 0; i < 6; i++) {
        Vec4<real> v; v.x = out[0][ks[i]]; v.y = out[1][ks[i]]; v.z = out[2][ks[i]]; v.w = out[3][ks[i]];
        st4(a.side_dst + (long long)i * a.pitch + xc, v);
      }
    }
    // ghost rows of the neighbours: the row below pulls speeds 4,7,8 of this slab's first
    // row, the row above 2,5,6 of its last row; the two-step kernel also wants 0,1,3 of those
    // rows (depth 0) and 4,7,8 / 2,5,6 of the second / second-to-last row (depth 1)
#define LBM_PUSH(dst, depth, k)                                                                          \
  { Vec4<real> v; v.x = out[0][k]; v.y = out[1][k]; v.z = out[2][k]; v.w = out[3][k];                      \
    st4((dst) + (long long)((depth) * 9 + (k)) * a.pitch + xc, v); }
    if (first) {
      LBM_PUSH(a.push_dn, 0, 4) LBM_PUSH(a.push_dn, 0, 7) LBM_PUSH(a.push_dn, 0, 8)
      if (a.deep) { LBM_PUSH(a.push_dn, 0, 0) LBM_PUSH(a.push_dn, 0, 1) LBM_PUSH(a.push_dn, 0, 3) }
    }
    if (last) {
      LBM_PUSH(a.push_up, 0, 2) LBM_PUSH(a.push_up, 0, 5) LBM_PUSH(a.push_up, 0, 6)
      if (a.deep) { LBM_PUSH(a.push_up, 0, 0) LBM_PUSH(a.push_up, 0, 1) LBM_PUSH(a.push_up, 0, 3) }
    }
    if (second) { LBM_PUSH(a.push_dn, 1, 4) LBM_PUSH(a.push_dn, 1, 7) LBM_PUSH(a.push_dn, 1, 8) }
    if (before_last) { LBM_PUSH(a.push_up, 1, 2) LBM_PUSH(a.push_up, 1, 5) LBM_PUSH(a.push_up, 1, 6) }
#undef LBM_PUSH
  }
  return q;
}

template <typename real, bool STRICT, bool MULTI>
__global__ void __launch_bounds__(LBM_BLOCK_THREADS, (sizeof(real) == 4 ? LBM_MIN_BLOCKS : 1))
lbm_step_vec4(const __grid_constant__ StepArgs<real> a) {
  int tx, ty;
  tile_of_block(a.tiles_x, a.tiles_y, a.edge_tiles, tx, ty);
  // Programmatic dependent launch: when the host launches the steps with
  // cudaLaunchAttributeProgrammaticStreamSerialization this grid may be scheduled while
  // the previous step drains; everything the previous step wrote is visible after this
  // call.  A no-op for an ordinary launch.
  cudaGridDependencySynchronize();
  const bool is_boundary = is_edge_tile(ty, a.tiles_y, a.edge_tiles);
  boundary_wait<real, MULTI>(a, is_boundary);
  const QuadConsts<real, STRICT> qc(a.omega);
  const unsigned long long q = vec4_tile<real, STRICT, false>(a, qc, tx, ty);
  block_accumulate(q, a.av);
  boundary_signal<real, MULTI>(a, is_boundary);
}

// ------------------------------------------------------------------------------------
// K1c  lbm_step_tma (fp32, opt-in with LBM_GPU_KERNEL_TMA): the same step with the nine
// pulled rows of a 512-cell tile staged in shared memory by the Tensor Memory Accelerator
// (one 3-D tensor map per lattice buffer: x, row, plane).  The copy engine does the y part
// of the propagate shift (box row = r - e_y).  It cannot do the x part: the innermost box
// coordinate must be a multiple of 16 bytes -- x = 1 raises an illegal-instruction fault
// (tools/probe/tma_probe.cu) -- so the x-shifted planes get a 4-element halo box on the
// side they pull from and the threads read that one extra element from shared memory,
// where K1a uses a warp shuffle.  The two ends of a row (periodic wrap in x) and the few
// rows that read the ghost rows or the accelerated side row keep the direct-load path
// (vec4_tile), chosen per block.  Built to measure whether staging buys anything over
// K1a: it does not (profiles/r01_kernel_variants.md), every byte is used once either way.
// ------------------------------------------------------------------------------------
#define LBM_TMA_TILE (LBM_BLOCK_THREADS * 4)
#define LBM_TMA_BOX (LBM_TMA_TILE < 256 ? LBM_TMA_TILE : 256)
static_assert(9 * LBM_TMA_TILE * sizeof(float) + 9 * 32 * sizeof(float) + 16 <= 48 * 1024,
              "K1c stages its tile in static shared memory: LBM_BLOCK_THREADS must be <= 256");

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

template <bool STRICT, bool MULTI>
__global__ void __launch_bounds__(LBM_BLOCK_THREADS, LBM_MIN_BLOCKS)
lbm_step_tma(const __grid_constant__ StepArgs<float> a, const __grid_constant__ CUtensorMap src_map,
             const __grid_constant__ CUtensorMap halo_map) {
  __shared__ alignas(128) float tile[9][LBM_TMA_TILE];
  __shared__ alignas(128) float halo[9][32];          // [k][0..3]: planes 1,5,8 cells xt-4..xt-1; 3,6,7 xt+T..xt+T+3
                                                      // (rows 128 B apart: TMA destinations are 128-byte aligned)
  __shared__ alignas(8) unsigned long long mbar;
  int tx, ty;
  tile_of_block(a.tiles_x, a.tiles_y, a.edge_tiles, tx, ty);
  const bool is_boundary = is_edge_tile(ty, a.tiles_y, a.edge_tiles);
  boundary_wait<float, MULTI>(a, is_boundary);

  const int r = ty;                                   // blockDim = (LBM_BLOCK_THREADS, 1): one row per tile
  const bool special = (r == 0) || (r == a.rows - 1) || (r == a.accel_row) || (r - 1 == a.accel_row) ||
                       (r + 1 == a.accel_row);
  unsigned long long q = 0ULL;
  const QuadConsts<float, STRICT> qc(a.omega);
  if (special) {
    q = vec4_tile<float, STRICT, false>(a, qc, tx, ty);
  } else {
    const int tid = threadIdx.x;
    const int xt = tx * LBM_TMA_TILE;                 // first column of the tile
    if (tid == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&mbar)) : "memory");
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&mbar)),
                   "r"((uint32_t)((9 * LBM_TMA_TILE + 6 * 4) * sizeof(float))) : "memory");
      // e_k of d2q9-bgk.c:7-13: the value pulled into (x, r) for speed k sits at (x - ex, r - ey).
      // A TMA box is at most 256 elements per dimension: LBM_TMA_TILE / 256 boxes per plane,
      // plus a 4-element box left of the tile (ex = +1) or right of it (ex = -1).
#define LBM_TMA_LOAD(k, ex, ey)                                                                                  \
  _Pragma("unroll") for (int b = 0; b < LBM_TMA_TILE / LBM_TMA_BOX; b++)                                        \
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" \
                 ::"r"(smem_u32(&tile[k][b * LBM_TMA_BOX])), "l"(&src_map), "r"(smem_u32(&mbar)),                 \
                 "r"(xt + b * LBM_TMA_BOX), "r"(r - (ey)), "r"(k) : "memory");                                   \
  if ((ex) != 0)                                                                                                 \
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" \
                 ::"r"(smem_u32(&halo[k][0])), "l"(&halo_map), "r"(smem_u32(&mbar)),                              \
                 "r"((ex) > 0 ? xt - 4 : xt + LBM_TMA_TILE), "r"(r - (ey)), "r"(k) : "memory")
      LBM_TMA_LOAD(0, 0, 0);  LBM_TMA_LOAD(1, 1, 0);   LBM_TMA_LOAD(2, 0, 1);
      LBM_TMA_LOAD(3, -1, 0); LBM_TMA_LOAD(4, 0, -1);  LBM_TMA_LOAD(5, 1, 1);
      LBM_TMA_LOAD(6, -1, 1); LBM_TMA_LOAD(7, -1, -1); LBM_TMA_LOAD(8, 1, -1);
#undef LBM_TMA_LOAD
    }
    const int x0 = xt + tid * 4;
    const bool active = x0 < a.nx;
    const int xc = active ? x0 : 0;
    const long long PS = a.plane_stride;
    const long long oC = (long long)r * a.pitch, oS = oC - a.pitch, oN = oC + a.pitch;
    // the wrap elements at the two ends of the row come by ordinary loads (the tensor map
    // zero-fills x < 0 and reads row padding beyond nx)
    const bool need_w = active && (x0 == 0);
    const bool need_e = active && (x0 + 4 >= a.nx);
    float w1e = 0, w5e = 0, w8e = 0, e3e = 0, e6e = 0, e7e = 0;
    if (need_w) {
      w1e = a.src[1 * PS + oC + a.nx - 1]; w5e = a.src[5 * PS + oS + a.nx - 1]; w8e = a.src[8 * PS + oN + a.nx - 1];
    }
    if (need_e) { e3e = a.src[3 * PS + oC]; e6e = a.src[6 * PS + oS]; e7e = a.src[7 * PS + oN]; }
    const uint32_t mword = a.mask[(long long)r * a.mask_pitch + (xc >> 5)];
    uint32_t obits = (mword >> (xc & 31)) & 0xFu;

    {   // wait for the rows (phase 0 of a barrier used once)
      uint32_t done = 0;
      while (!done)
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0; selp.b32 %0, 1, 0, p; }"
                     : "=r"(done) : "r"(smem_u32(&mbar)) : "memory");
    }
    float in[4][9], out[4][9];
#define LBM_ROW(k) (*reinterpret_cast<const float4*>(&tile[k][tid * 4]))
#define LBM_WEST(k) (tid == 0 ? halo[k][3] : tile[k][tid * 4 - 1])
#define LBM_EAST(k) (tid == LBM_BLOCK_THREADS - 1 ? halo[k][0] : tile[k][tid * 4 + 4])
    { const float4 v = LBM_ROW(0); in[0][0] = v.x; in[1][0] = v.y; in[2][0] = v.z; in[3][0] = v.w; }
    { const float4 v = LBM_ROW(2); in[0][2] = v.x; in[1][2] = v.y; in[2][2] = v.z; in[3][2] = v.w; }
    { const float4 v = LBM_ROW(4); in[0][4] = v.x; in[1][4] = v.y; in[2][4] = v.z; in[3][4] = v.w; }
    { const float4 v = LBM_ROW(1); in[0][1] = LBM_WEST(1); in[1][1] = v.x; in[2][1] = v.y; in[3][1] = v.z; }
    { const float4 v = LBM_ROW(5); in[0][5] = LBM_WEST(5); in[1][5] = v.x; in[2][5] = v.y; in[3][5] = v.z; }
    { const float4 v = LBM_ROW(8); in[0][8] = LBM_WEST(8); in[1][8] = v.x; in[2][8] = v.y; in[3][8] = v.z; }
    { const float4 v = LBM_ROW(3); in[0][3] = v.y; in[1][3] = v.z; in[2][3] = v.w; in[3][3] = LBM_EAST(3); }
    { const float4 v = LBM_ROW(6); in[0][6] = v.y; in[1][6] = v.z; in[2][6] = v.w; in[3][6] = LBM_EAST(6); }
    { const float4 v = LBM_ROW(7); in[0][7] = v.y; in[1][7] = v.z; in[2][7] = v.w; in[3][7] = LBM_EAST(7); }
#undef LBM_ROW
#undef LBM_WEST
#undef LBM_EAST
    if (need_w) { in[0][1] = w1e; in[0][5] = w5e; in[0][8] = w8e; }
    if (need_e) {
      const int nvalid = a.nx - x0;
      if (nvalid == 1) { in[0][3] = e3e; in[0][6] = e6e; in[0][7] = e7e; }
      else if (nvalid == 2) { in[1][3] = e3e; in[1][6] = e6e; in[1][7] = e7e; }
      else if (nvalid == 3) { in[2][3] = e3e; in[2][6] = e6e; in[2][7] = e7e; }
      else { in[3][3] = e3e; in[3][6] = e6e; in[3][7] = e7e; }
      if (nvalid < 4) obits |= (0xFu << nvalid) & 0xFu;
    }
    bool bad;
    q = quad_update<float, STRICT>(in, obits, qc, out, bad);
    if (active && bad) atomicOr(a.av + 1, LBM_NONFINITE_MARK);
    if (active) {
      float* d = a.dst + oC + x0;
#pragma unroll
      for (int k = 0; k < 9; k++) {
        Vec4<float> v; v.x = out[0][k]; v.y = out[1][k]; v.z = out[2][k]; v.w = out[3][k];
        st4(d + k * PS, v);
      }
    } else {
      q = 0ULL;
    }
  }
  block_accumulate(q, a.av);
  boundary_signal<float, MULTI>(a, is_boundary);
}

// ------------------------------------------------------------------------------------
// K1b  lbm_step_scalar: one cell per thread, any nx.  Same arithmetic; used for grids
// whose width is not a multiple of 4 and as an independent cross-check of K1a.
// ------------------------------------------------------------------------------------
template <typename real, bool STRICT, bool CG>
__device__ __forceinline__ unsigned long long scalar_tile(const StepArgs<real>& a, const int tx, const int ty) {
#define LD(ptr) load1<real, CG>(ptr)
  const int x = tx * (int)blockDim.x + (int)threadIdx.x;
  const int r = ty * (int)blockDim.y + (int)threadIdx.y;
  const bool active = (x < a.nx) && (r < a.rows);
  real s = (real)0;
  if (active) {
    const long long PS = a.plane_stride;
    const long long oC = (long long)r * a.pitch, oS = oC - a.pitch, oN = oC + a.pitch;
    const bool first = (r == 0), last = (r == a.rows - 1);
    const bool cA = (r == a.accel_row), sA = (r - 1 == a.accel_row), nA = (r + 1 == a.accel_row);
    const int xw = (x == 0) ? a.nx - 1 : x - 1;
    const int xe = (x + 1 == a.nx) ? 0 : x + 1;
    real p[9], o[9];
    p[0] = LD(a.src + oC + x);
    p[1] = cA ? LD(a.side_src + 0 * a.pitch + xw) : LD(a.src + 1 * PS + oC + xw);
    p[3] = cA ? LD(a.side_src + 1 * a.pitch + xe) : LD(a.src + 3 * PS + oC + xe);
    p[2] = first ? LD(a.ghost_s + 2 * a.pitch + x) : LD(a.src + 2 * PS + oS + x);
    p[5] = first ? LD(a.ghost_s + 5 * a.pitch + xw) : (sA ? LD(a.side_src + 2 * a.pitch + xw) : LD(a.src + 5 * PS + oS + xw));
    p[6] = first ? LD(a.ghost_s + 6 * a.pitch + xe) : (sA ? LD(a.side_src + 3 * a.pitch + xe) : LD(a.src + 6 * PS + oS + xe));
    p[4] = last ? LD(a.ghost_n + 4 * a.pitch + x) : LD(a.src + 4 * PS + oN + x);
    p[7] = last ? LD(a.ghost_n + 7 * a.pitch + xe) : (nA ? LD(a.side_src + 4 * a.pitch + xe) : LD(a.src + 7 * PS + oN + xe));
    p[8] = last ? LD(a.ghost_n + 8 * a.pitch + xw) : (nA ? LD(a.side_src + 5 * a.pitch + xw) : LD(a.src + 8 * PS + oN + xw));
    const bool obst = (a.mask[(long long)r * a.mask_pitch + (x >> 5)] >> (x & 31)) & 1u;
    s = cell_update<real, STRICT>(p, obst, a.omega, o);
#pragma unroll
    for (int k = 0; k < 9; k++) a.dst[k * PS + oC + x] = o[k];
    if (cA) {
      cell_accelerate<real, STRICT>(o[1], o[3], o[5], o[6], o[7], o[8], obst, a.aw1, a.aw2);
      a.side_dst[0 * a.pitch + x] = o[1]; a.side_dst[1 * a.pitch + x] = o[3];
      a.side_dst[2 * a.pitch + x] = o[5]; a.side_dst[3 * a.pitch + x] = o[6];
      a.side_dst[4 * a.pitch + x] = o[7]; a.side_dst[5 * a.pitch + x] = o[8];
    }
    if (first) {
      a.push_dn[4 * a.pitch + x] = o[4];
      a.push_dn[7 * a.pitch + x] = o[7];
      a.push_dn[8 * a.pitch + x] = o[8];
    }
    if (last) {
      a.push_up[2 * a.pitch + x] = o[2];
      a.push_up[5 * a.pitch + x] = o[5];
      a.push_up[6 * a.pitch + x] = o[6];
    }
  }
#undef LD
  // |u| sum: the strict build converts every cell exactly; the default build adds the four
  // cells of an aligned quad as floats in the order of the vectorised kernels (quad_update),
  // so that every kernel variant returns the same av_vels bits.
  // Both builds hold every cell to LBM_SPEED_LIMIT on its own (see quad_sum_fixed).
  unsigned long long q;
  const bool bad = !(s < (real)LBM_SPEED_LIMIT);
  if (STRICT) {
    q = to_fixed(s);
  } else {
    typedef Ops<real, true> M;
    real t = M::add(s, __shfl_xor_sync(0xffffffffu, s, 1));
    t = M::add(t, __shfl_xor_sync(0xffffffffu, t, 2));
    const bool lead = (threadIdx.x & 3) == 0;
    q = lead ? to_fixed(t) : 0ULL;
  }
  if (active && bad) atomicOr(a.av + 1, LBM_NONFINITE_MARK);
  return q;
}

template <typename real, bool STRICT, bool MULTI>
__global__ void __launch_bounds__(LBM_BLOCK_THREADS)
lbm_step_scalar(const __grid_constant__ StepArgs<real> a) {
  int tx, ty;
  tile_of_block(a.tiles_x, a.tiles_y, a.edge_tiles, tx, ty);
  const bool is_boundary = is_edge_tile(ty, a.tiles_y, a.edge_tiles);
  boundary_wait<real, MULTI>(a, is_boundary);
  const unsigned long long q = scalar_tile<real, STRICT, false>(a, tx, ty);
  block_accumulate(q, a.av);
  boundary_signal<real, MULTI>(a, is_boundary);
}

// ------------------------------------------------------------------------------------
// K5  lbm_steps_persistent: ALL timesteps of a run in one cooperative launch, for grids
// small enough to live in L2 (the reference's shipped inputs: 0.6-38 MB per buffer).
// There the per-step cost of K1a is launch latency, not bandwidth.  Every block owns a
// fixed set of tiles, loops over the steps, and meets the other blocks at a grid barrier
// (one atomic per block) between steps; buffers swap roles inside the kernel.  Single
// slab only (the ghost rows are the slab's own).  Loads are L2-only (see ld4cg).
// VEC = 4 cells per thread (K1a's tile) or, for the smallest grids, 1 cell per thread
// (K1b's tile): four times as many threads share the step's dependent-latency chain.
// Must be launched with cudaLaunchCooperativeKernel so that all blocks are resident.
// ------------------------------------------------------------------------------------
template <typename real>
struct PersistArgs {
  StepArgs<real> s;            // geometry, constants and the step-0 pointers
  real* lattice[2];
  real* side[2];
  real* window;                // own window: ghost rows at ghost_offset(pitch, parity, direction)
  unsigned long long* av;      // n_steps x LBM_AV_SLOTS x LBM_AV_STRIDE words
  unsigned long long* barrier; // zeroed before the launch
  int first_parity;            // buffer index read by the first step
  int n_steps;
  int n_tiles;
};

__device__ __forceinline__ unsigned long long ld_acquire_gpu(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

// All blocks are resident (cooperative launch), so the wait ends unless a block has faulted;
// the spin is still bounded (about a minute) and ends in a trap, which the host sees as a
// CUDA error on its next call instead of a kernel that never returns.
__device__ __forceinline__ void grid_barrier(unsigned long long* counter, const unsigned long long target) {
  __syncthreads();
  if (threadIdx.x == 0 && threadIdx.y == 0) {
#if LBM_BARRIER_MODE == 1
    // one release-reduction instead of fence + atomic + fence: the release is cumulative over
    // what the block's threads wrote before the __syncthreads, the acquire loads order what follows
    asm volatile("red.release.gpu.global.add.u64 [%0], %1;" ::"l"(counter), "l"(1ULL) : "memory");
#else
    __threadfence();
    atomicAdd(counter, 1ULL);
#endif
    unsigned spins = 0;
    while (ld_acquire_gpu(counter) < target) {
      if (++spins == 0x10000000u) __trap();
    }
#if LBM_BARRIER_MODE != 1
    __threadfence();
#endif
  }
  __syncthreads();
}

template <typename real, bool STRICT, int VEC>
__global__ void __launch_bounds__(LBM_BLOCK_THREADS, (sizeof(real) == 4 ? LBM_PERSIST_MIN_BLOCKS : 1))
lbm_steps_persistent(const __grid_constant__ PersistArgs<real> pa) {
  StepArgs<real> a = pa.s;
  const int pitch = a.pitch;
  const QuadConsts<real, STRICT> qc(a.omega);
  for (int t = 0; t < pa.n_steps; t++) {
    const int src = (pa.first_parity + t) & 1, dst = src ^ 1;
    a.src = pa.lattice[src];
    a.dst = pa.lattice[dst];
    a.side_src = pa.side[src];
    a.side_dst = pa.side[dst];
    a.ghost_s = pa.window + ghost_offset(pitch, src, 0);
    a.ghost_n = pa.window + ghost_offset(pitch, src, 1);
    a.push_up = pa.window + ghost_offset(pitch, dst, 0);
    a.push_dn = pa.window + ghost_offset(pitch, dst, 1);
    a.av = pa.av + (size_t)t * (LBM_AV_STRIDE * LBM_AV_SLOTS);
#if LBM_K5_EXPERIMENT != 2
    unsigned long long q = 0ULL;
    for (int tile = blockIdx.x; tile < pa.n_tiles; tile += gridDim.x) {
      const int ty = tile / a.tiles_x;
      const int tx = tile - ty * a.tiles_x;
      q += (VEC == 4) ? vec4_tile<real, STRICT, true>(a, qc, tx, ty) : scalar_tile<real, STRICT, true>(a, tx, ty);
    }
    warp_accumulate(q, a.av);
#endif
#if LBM_K5_EXPERIMENT != 1
    // (a variant where the last arriver publishes an epoch in a separate word that the
    // others poll was measured SLOWER -- one more L2 round trip: 128^2 3.0 -> 3.6 us/step)
    grid_barrier(pa.barrier, (unsigned long long)gridDim.x * (unsigned long long)(t + 1));
#endif
  }
}

// ------------------------------------------------------------------------------------
// K3  lbm_prepare: run once after the lattice was created or uploaded.  Fills the side
// row (accelerate_flow applied to row ny-2 of the current buffer, d2q9-bgk.c:229-260)
// and pushes the slab's edge rows into the neighbours' ghost rows of the same buffer.
// One thread per column.
// ------------------------------------------------------------------------------------
template <typename real>
struct PrepareArgs {
  const real* cur;            // current lattice buffer
  real* side_cur;             // side row of the same parity
  const uint32_t* mask;
  real* push_up;              // neighbour above's window, current parity, "from below"
  real* push_dn;              // neighbour below's window, current parity, "from above"
  uint32_t* mask_up;          // neighbour above's copy of the mask of ITS row -1 (= this slab's last row)
  uint32_t* mask_dn;          // neighbour below's copy of the mask of ITS row `rows` (= this slab's first row)
  long long plane_stride;
  int nx, rows, pitch, mask_pitch, accel_row;
  int deep;                   // also fill what the two-step kernel reads (see "window")
  real aw1, aw2;
};

template <typename real>
__global__ void lbm_prepare(const PrepareArgs<real> a) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x < a.mask_pitch) {
    a.mask_dn[x] = a.mask[x];
    a.mask_up[x] = a.mask[(long long)(a.rows - 1) * a.mask_pitch + x];
  }
  if (x >= a.nx) return;
  const long long PS = a.plane_stride;
#pragma unroll 1
  for (int which = 0; which < 5; which++) {
    // 0: accelerate row -> side; 1: first row -> down, depth 0; 2: last row -> up, depth 0;
    // 3: second row -> down, depth 1; 4: second-to-last row -> up, depth 1
    const int r = (which == 0) ? a.accel_row : (which == 1) ? 0 : (which == 2) ? a.rows - 1 : (which == 3) ? 1 : a.rows - 2;
    if (r < 0 || r >= a.rows) continue;
    if (which >= 3 && !a.deep) continue;
    const long long o = (long long)r * a.pitch + x;
    real f[9];
#pragma unroll
    for (int k = 0; k < 9; k++) f[k] = a.cur[k * PS + o];
    if (r == a.accel_row) {
      const bool obst = (a.mask[(long long)r * a.mask_pitch + (x >> 5)] >> (x & 31)) & 1u;
      cell_accelerate<real, true>(f[1], f[3], f[5], f[6], f[7], f[8], obst, a.aw1, a.aw2);
    }
    if (which == 0) {
      a.side_cur[0 * a.pitch + x] = f[1]; a.side_cur[1 * a.pitch + x] = f[3];
      a.side_cur[2 * a.pitch + x] = f[5]; a.side_cur[3 * a.pitch + x] = f[6];
      a.side_cur[4 * a.pitch + x] = f[7]; a.side_cur[5 * a.pitch + x] = f[8];
    } else {
      const bool down = (which == 1 || which == 3);
      real* dst = (down ? a.push_dn : a.push_up) + (long long)(which >= 3 ? 9 : 0) * a.pitch + x;
      const int k0 = down ? 4 : 2, k1 = down ? 7 : 5, k2 = down ? 8 : 6;
      dst[(long long)k0 * a.pitch] = f[k0];
      dst[(long long)k1 * a.pitch] = f[k1];
      dst[(long long)k2 * a.pitch] = f[k2];
      if (which < 3 && a.deep) {
        dst[0] = f[0];
        dst[(long long)1 * a.pitch] = f[1];
        dst[(long long)3 * a.pitch] = f[3];
      }
    }
  }
}

// ------------------------------------------------------------------------------------
// K4  setup / output kernels (not on the per-step path)
// ------------------------------------------------------------------------------------
// Stored lattice values.  An fp32 / fp64 lattice holds f itself.  A LBM_GPU_STORE_F16 lattice
// holds the binary16 value of f_k - c_k, with c_k the rest-state value of speed k: encoded with
// one fp32 subtract and a round to nearest even, decoded exactly and with one fp32 add.
struct RestShift {
  float w0, w1, w2;             // density*4/9, density/9, density/36 (as the rest state)
  __host__ __device__ __forceinline__ float of(const int k) const { return k == 0 ? w0 : (k < 5 ? w1 : w2); }
};
__device__ __forceinline__ float f16_dec(const __half s, const float c) { return __fadd_rn(__half2float(s), c); }
__device__ __forceinline__ __half f16_enc(const float f, const float c) { return __float2half_rn(__fsub_rn(f, c)); }
template <typename real>
__device__ __forceinline__ real stored_value(const real* p, int, const RestShift&) { return *p; }
__device__ __forceinline__ float stored_value(const __half* p, const int k, const RestShift& r) { return f16_dec(*p, r.of(k)); }
template <typename real>
__device__ __forceinline__ void store_value(real* p, int, const real v, const RestShift&) { *p = v; }
__device__ __forceinline__ void store_value(__half* p, const int k, const float v, const RestShift& r) { *p = f16_enc(v, r.of(k)); }

// rest state, d2q9-bgk.c:2802-2823
template <typename real>
__global__ void lbm_init_rest(real* buf, long long plane_stride, int pitch, int nx, int rows,
                              real w0, real w1, real w2) {
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = (long long)rows * pitch;
  if (n >= total) return;
#pragma unroll
  for (int k = 0; k < 9; k++) buf[k * plane_stride + n] = (k == 0) ? w0 : (k < 5 ? w1 : w2);
}

// AoS rows (9 reals per cell, dense nx) -> SoA planes; `aos` holds nrows rows that go
// to local rows [r0, r0+nrows)
template <typename real, typename store = real>
__global__ void lbm_aos_to_soa(const real* __restrict__ aos, store* __restrict__ buf, long long plane_stride,
                               int pitch, int nx, int r0, long long ncells, RestShift rest = RestShift()) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ncells * 9) return;
  const long long cell = i / 9;
  const int k = (int)(i - cell * 9);
  const long long row = cell / nx;
  const int x = (int)(cell - row * nx);
  store_value(buf + k * plane_stride + (r0 + row) * pitch + x, k, aos[i], rest);
}

template <typename real, typename store = real>
__global__ void lbm_soa_to_aos(const store* __restrict__ buf, real* __restrict__ aos, long long plane_stride,
                               int pitch, int nx, int r0, long long ncells, RestShift rest = RestShift()) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ncells * 9) return;
  const long long cell = i / 9;
  const int k = (int)(i - cell * 9);
  const long long row = cell / nx;
  const int x = (int)(cell - row * nx);
  aos[i] = stored_value(buf + k * plane_stride + (r0 + row) * pitch + x, k, rest);
}

// lbm_gpu_save_rows / lbm_gpu_load_rows: the stored lattice <-> cell-major records (9 elements per
// cell, speed order), bits moved unchanged.  T is the unsigned type of the stored element (uint32
// fp32, uint64 fp64, uint16 binary16).  A block takes kRecCells consecutive cells of the chunk
// (local rows [r0, r0 + ncells / nx)) and transposes them in shared memory, which holds them in
// record order: the record side is then one contiguous run of 16-byte accesses (the chunk starts
// 16-byte aligned and kRecCells * 9 elements is a multiple of 16 bytes), and the plane side reads
// or writes x-consecutive elements, 16 bytes at a time when VEC (nx a multiple of 16 / sizeof(T),
// so that a vector never crosses a row; pitch is a multiple of 32).  Columns nx..pitch-1 (padding)
// are never touched.
constexpr int kRecCells = 256;
constexpr int kRecThreads = 256;

template <typename T, bool VEC>
__global__ void __launch_bounds__(kRecThreads) lbm_pack_rows(const T* __restrict__ buf, T* __restrict__ rec,
                                                             long long plane_stride, int pitch, int nx, int r0,
                                                             long long ncells) {
  constexpr int V = 16 / sizeof(T);
  __shared__ __align__(16) T sm[kRecCells * 9];
  const long long c0 = (long long)blockIdx.x * kRecCells;
  const int nc = (int)min((long long)kRecCells, ncells - c0);
  const long long row_c0 = c0 / nx;
  const int x_c0 = (int)(c0 - row_c0 * nx);
  if (VEC) {
    for (int j = threadIdx.x; j < 9 * (kRecCells / V); j += kRecThreads) {
      const int k = j / (kRecCells / V), c = (j - k * (kRecCells / V)) * V;
      if (c >= nc) continue;
      const int xc = x_c0 + c, dr = xc / nx;
      const uint4 v = *reinterpret_cast<const uint4*>(buf + k * plane_stride + (r0 + row_c0 + dr) * pitch + (xc - dr * nx));
      const T* e = reinterpret_cast<const T*>(&v);
#pragma unroll
      for (int q = 0; q < V; q++) sm[(c + q) * 9 + k] = e[q];
    }
  } else {
    for (int j = threadIdx.x; j < 9 * kRecCells; j += kRecThreads) {
      const int k = j / kRecCells, c = j - k * kRecCells;
      if (c >= nc) continue;
      const int xc = x_c0 + c, dr = xc / nx;
      sm[c * 9 + k] = buf[k * plane_stride + (r0 + row_c0 + dr) * pitch + (xc - dr * nx)];
    }
  }
  __syncthreads();
  T* out = rec + c0 * 9;
  const int n = nc * 9, nv = n / V;
  for (int j = threadIdx.x; j < nv; j += kRecThreads)
    reinterpret_cast<uint4*>(out)[j] = reinterpret_cast<const uint4*>(sm)[j];
  for (int j = nv * V + threadIdx.x; j < n; j += kRecThreads) out[j] = sm[j];
}

template <typename T, bool VEC>
__global__ void __launch_bounds__(kRecThreads) lbm_unpack_rows(const T* __restrict__ rec, T* __restrict__ buf,
                                                               long long plane_stride, int pitch, int nx, int r0,
                                                               long long ncells) {
  constexpr int V = 16 / sizeof(T);
  __shared__ __align__(16) T sm[kRecCells * 9];
  const long long c0 = (long long)blockIdx.x * kRecCells;
  const int nc = (int)min((long long)kRecCells, ncells - c0);
  const long long row_c0 = c0 / nx;
  const int x_c0 = (int)(c0 - row_c0 * nx);
  const T* in = rec + c0 * 9;
  const int n = nc * 9, nv = n / V;
  for (int j = threadIdx.x; j < nv; j += kRecThreads)
    reinterpret_cast<uint4*>(sm)[j] = reinterpret_cast<const uint4*>(in)[j];
  for (int j = nv * V + threadIdx.x; j < n; j += kRecThreads) sm[j] = in[j];
  __syncthreads();
  if (VEC) {
    for (int j = threadIdx.x; j < 9 * (kRecCells / V); j += kRecThreads) {
      const int k = j / (kRecCells / V), c = (j - k * (kRecCells / V)) * V;
      if (c >= nc) continue;
      const int xc = x_c0 + c, dr = xc / nx;
      uint4 v;
      T* e = reinterpret_cast<T*>(&v);
#pragma unroll
      for (int q = 0; q < V; q++) e[q] = sm[(c + q) * 9 + k];
      *reinterpret_cast<uint4*>(buf + k * plane_stride + (r0 + row_c0 + dr) * pitch + (xc - dr * nx)) = v;
    }
  } else {
    for (int j = threadIdx.x; j < 9 * kRecCells; j += kRecThreads) {
      const int k = j / kRecCells, c = j - k * kRecCells;
      if (c >= nc) continue;
      const int xc = x_c0 + c, dr = xc / nx;
      buf[k * plane_stride + (r0 + row_c0 + dr) * pitch + (xc - dr * nx)] = sm[c * 9 + k];
    }
  }
}

// int-per-cell obstacle rows -> bit mask rows; one warp packs 32 cells with a ballot.
// Also counts the blocked cells.
__global__ void lbm_pack_mask(const int* __restrict__ obst, uint32_t* __restrict__ mask, int mask_pitch,
                              int nx, int r0, int nrows, unsigned long long* blocked_count) {
  const long long gw = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;   // global warp
  const int lane = threadIdx.x & 31;
  const int words_per_row = (nx + 31) >> 5;
  if (gw >= (long long)nrows * words_per_row) return;
  const int row = (int)(gw / words_per_row);
  const int wi = (int)(gw - (long long)row * words_per_row);
  const int x = wi * 32 + lane;
  const bool b = (x < nx) && (obst[(long long)row * nx + x] != 0);
  const uint32_t bits = __ballot_sync(0xffffffffu, b);
  if (lane == 0) {
    mask[(long long)(r0 + row) * mask_pitch + wi] = bits;
    if (bits) atomicAdd(blocked_count, (unsigned long long)__popc(bits));
  }
}

// dense bit-packed host rows ((nx+31)/32 words per row) -> pitched mask rows
__global__ void lbm_copy_mask_bits(const uint32_t* __restrict__ in, uint32_t* __restrict__ mask, int mask_pitch,
                                   int nx, int r0, int nrows, unsigned long long* blocked_count) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int words_per_row = (nx + 31) >> 5;
  if (i >= (long long)nrows * words_per_row) return;
  const int row = (int)(i / words_per_row);
  const int wi = (int)(i - (long long)row * words_per_row);
  uint32_t bits = in[i];
  const int valid = nx - wi * 32;
  if (valid < 32) bits &= (1u << valid) - 1u;
  mask[(long long)(r0 + row) * mask_pitch + wi] = bits;
  if (bits) atomicAdd(blocked_count, (unsigned long long)__popc(bits));
}

// write_values' per-cell fields (d2q9-bgk.c:2937-2976) for local rows [r0, r0+nrows):
// dense nx-wide outputs.  Also usable as av_velocity (d2q9-bgk.c:2665-2714) through
// the |u| accumulator (warp_accumulate) when av != NULL; a fluid cell whose |u| is NaN or
// not below LBM_SPEED_LIMIT adds nothing and sets LBM_NONFINITE_MARK in av[1], as the step
// kernels do.
template <typename real, typename store = real>
__global__ void lbm_fields(const store* __restrict__ buf, const uint32_t* __restrict__ mask,
                           long long plane_stride, int pitch, int mask_pitch, int nx, int r0, int nrows,
                           real density, real* __restrict__ ux_out, real* __restrict__ uy_out,
                           real* __restrict__ u_out, real* __restrict__ p_out,
                           unsigned long long* av, RestShift rest = RestShift()) {
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long q = 0ULL;
  if (n < (long long)nrows * nx) {
    const int row = (int)(n / nx);
    const int x = (int)(n - (long long)row * nx);
    const int r = r0 + row;                      // local row
    const bool obst = (mask[(long long)r * mask_pitch + (x >> 5)] >> (x & 31)) & 1u;
    real f[9];
#pragma unroll
    for (int k = 0; k < 9; k++) f[k] = stored_value(buf + k * plane_stride + (long long)r * pitch + x, k, rest);
    real ux, uy, rho;
    real u = cell_macroscopic<real>(f, ux, uy, rho);
    const real c_sq = (real)1 / (real)3;
    real pr = Ops<real, true>::mul(rho, c_sq);
    if (obst) { ux = 0; uy = 0; u = 0; pr = Ops<real, true>::mul(density, c_sq); }
    if (ux_out) ux_out[n] = ux;
    if (uy_out) uy_out[n] = uy;
    if (u_out) u_out[n] = u;
    if (p_out) p_out[n] = pr;
    if (u < (real)LBM_SPEED_LIMIT) q = to_fixed(u);
    else if (av) atomicOr(av + 1, LBM_NONFINITE_MARK);
  }
  if (av) warp_accumulate(q, av);
}

// Block means of lbm_fields' values (lbm_gpu_coarse_fields, include/lbm_gpu.h).  The grid is cut
// into factor x factor blocks from global cell (0,0).  blockIdx.y is one band, coarse row
// J0 + blockIdx.y, restricted to the rows [s_row0, s_row0 + s_rows) this slab holds; blockIdx.x
// is a run of `nc` coarse columns.  nc * factor is a multiple of 4, so thread t's column quad,
// starting at x = C0 * factor + 4t, is aligned for one 128-bit load per plane (64-bit for
// binary16); the thread walks down the band.  Each cell's (u_x, u_y, |u|, pressure) is
// lbm_fields' value bit for bit and enters its block's sum as round_half_even(v * 2^32) in int64:
// integer sums are exact in any order, so the threads' sums meet per coarse column in shared
// memory with atomics, for any factor.  With factor >= 2 a quad touches at most two coarse
// columns: the first `split` of its columns belong to the first.  A value that is not finite or
// of magnitude kCoarseLimit or more marks its field of the block instead; below that bound a
// 256 x 256 block's sum stays under 2^63.
//   raw == nullptr  every band lies wholly in this slab: the block writes the means, fp32 or
//                   binary16 (pressure shifted by p0, the obstacle pressure), ncx per output row;
//   raw != nullptr  partial sums of a band cut by a slab boundary, kCoarseRawWords per block
//                   (four sums, then the mark bits), for the host to add across slabs.
// factor == 1 (binary16 output only): each cell's values are converted directly, no sums.
constexpr float kCoarseLimit = 32768.0f;             // 2^15
constexpr int kCoarseSpan = 1024;                    // columns per block, at most
constexpr int kCoarseThreads = kCoarseSpan / 4;
constexpr int kCoarseRawWords = 5;

__device__ __forceinline__ void load_quad(const float* p, int, const RestShift&, float (&v)[4]) {
  const float4 q = *reinterpret_cast<const float4*>(p);
  v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
}
__device__ __forceinline__ void load_quad(const __half* p, const int k, const RestShift& r, float (&v)[4]) {
  const uint2 q = *reinterpret_cast<const uint2*>(p);
  const __half2 a = *reinterpret_cast<const __half2*>(&q.x), b = *reinterpret_cast<const __half2*>(&q.y);
  const float c = r.of(k);
  v[0] = f16_dec(__low2half(a), c); v[1] = f16_dec(__high2half(a), c);
  v[2] = f16_dec(__low2half(b), c); v[3] = f16_dec(__high2half(b), c);
}
// an output value; binary16 outputs hold v - shift (0 for the velocities, p0 for the pressure)
__device__ __forceinline__ void put_field(float* o, const float v, float) { *o = v; }
__device__ __forceinline__ void put_field(__half* o, const float v, const float shift) { *o = __float2half_rn(__fsub_rn(v, shift)); }

__device__ __forceinline__ void add_fixed(unsigned long long& acc, unsigned& mark, const unsigned bit, const float v) {
  if (::fabsf(v) < kCoarseLimit) acc += (unsigned long long)__float2ll_rn(__fmul_rn(v, 4294967296.0f));
  else mark |= bit;                                  // NaN lands here too
}

template <typename store, typename out_t>
__global__ void __launch_bounds__(kCoarseThreads)
lbm_coarse_fields(const store* __restrict__ buf, const uint32_t* __restrict__ mask, long long plane_stride,
                  int pitch, int mask_pitch, int nx, int ny, long long s_row0, int s_rows, int factor, int nc,
                  int ncx, long long J0, float density, RestShift rest, out_t* __restrict__ ux_out,
                  out_t* __restrict__ uy_out, out_t* __restrict__ u_out, out_t* __restrict__ p_out,
                  unsigned long long* __restrict__ raw) {
  extern __shared__ unsigned long long coarse_sm[];  // nc x 4 sums, then nc mark words
  typedef Ops<float, true> M;
  const float c_sq = 1.0f / 3.0f;
  const float p0 = M::mul(density, c_sq);
  const long long g0 = (J0 + blockIdx.y) * factor, g1 = ::min(g0 + factor, (long long)ny);   // global rows
  const int r0 = (int)(::max(g0, s_row0) - s_row0);                                           // local rows
  const int r1 = (int)(::min(g1, s_row0 + s_rows) - s_row0);
  const int C0 = blockIdx.x * nc;
  const int ncb = ::min(nc, ncx - C0);
  const int xend = ::min((C0 + ncb) * factor, nx);
  const int x4 = C0 * factor + 4 * (int)threadIdx.x;
  const int nvalid = ::min(4, xend - x4);
  const long long orow = (long long)blockIdx.y * ncx;

  if (factor == 1) {
    if (nvalid <= 0) return;
    float f[9][4];
#pragma unroll
    for (int k = 0; k < 9; k++) load_quad(buf + k * plane_stride + (long long)r0 * pitch + x4, k, rest, f[k]);
    const uint32_t ob = mask[(long long)r0 * mask_pitch + (x4 >> 5)] >> (x4 & 31);
#pragma unroll
    for (int j = 0; j < 4; j++) {
      if (j >= nvalid) break;
      float cell[9];
#pragma unroll
      for (int k = 0; k < 9; k++) cell[k] = f[k][j];
      float ux, uy, rho;
      float u = cell_macroscopic<float>(cell, ux, uy, rho);
      float pr = M::mul(rho, c_sq);
      if ((ob >> j) & 1u) { ux = 0; uy = 0; u = 0; pr = p0; }
      const long long o = orow + x4 + j;
      if (ux_out) put_field(ux_out + o, ux, 0.0f);
      if (uy_out) put_field(uy_out + o, uy, 0.0f);
      if (u_out) put_field(u_out + o, u, 0.0f);
      if (p_out) put_field(p_out + o, pr, p0);
    }
    return;
  }

  unsigned long long* sums = coarse_sm;
  unsigned* marks = reinterpret_cast<unsigned*>(coarse_sm + 4 * nc);
  for (int i = threadIdx.x; i < 4 * nc; i += blockDim.x) sums[i] = 0ULL;
  for (int i = threadIdx.x; i < nc; i += blockDim.x) marks[i] = 0u;
  __syncthreads();
  if (nvalid > 0) {
    const int lo = x4 / factor;                      // coarse column of the quad's first column
    const int split = ::min(4, (lo + 1) * factor - x4);
    unsigned long long a0[4] = {0ULL, 0ULL, 0ULL, 0ULL}, a1[4] = {0ULL, 0ULL, 0ULL, 0ULL};
    unsigned mark = 0u;                              // bit 4 * (second column) + field
    for (int r = r0; r < r1; r++) {
      float f[9][4];
#pragma unroll
      for (int k = 0; k < 9; k++) load_quad(buf + k * plane_stride + (long long)r * pitch + x4, k, rest, f[k]);
      const uint32_t ob = mask[(long long)r * mask_pitch + (x4 >> 5)] >> (x4 & 31);
#pragma unroll
      for (int j = 0; j < 4; j++) {
        if (j >= nvalid) break;
        float cell[9];
#pragma unroll
        for (int k = 0; k < 9; k++) cell[k] = f[k][j];
        float ux, uy, rho;
        float u = cell_macroscopic<float>(cell, ux, uy, rho);
        float pr = M::mul(rho, c_sq);
        if ((ob >> j) & 1u) { ux = 0; uy = 0; u = 0; pr = p0; }
        if (j < split) {
          add_fixed(a0[0], mark, 1u, ux); add_fixed(a0[1], mark, 2u, uy);
          add_fixed(a0[2], mark, 4u, u); add_fixed(a0[3], mark, 8u, pr);
        } else {
          add_fixed(a1[0], mark, 16u, ux); add_fixed(a1[1], mark, 32u, uy);
          add_fixed(a1[2], mark, 64u, u); add_fixed(a1[3], mark, 128u, pr);
        }
      }
    }
    const int c = lo - C0;
#pragma unroll
    for (int i = 0; i < 4; i++)
      if (a0[i]) atomicAdd(sums + 4 * c + i, a0[i]);
    if (mark & 15u) atomicOr(marks + c, mark & 15u);
    if (split < nvalid) {
#pragma unroll
      for (int i = 0; i < 4; i++)
        if (a1[i]) atomicAdd(sums + 4 * (c + 1) + i, a1[i]);
      if (mark >> 4) atomicOr(marks + c + 1, mark >> 4);
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < ncb; c += blockDim.x) {
    const int C = C0 + c;
    const unsigned m = marks[c];
    if (raw) {
      unsigned long long* w = raw + (orow + C) * kCoarseRawWords;
#pragma unroll
      for (int i = 0; i < 4; i++) w[i] = sums[4 * c + i];
      w[4] = m;
      continue;
    }
    const double cells = (double)((g1 - g0) * (long long)::min(factor, nx - C * factor));
    float mean[4];
#pragma unroll
    for (int i = 0; i < 4; i++)
      mean[i] = ((m >> i) & 1u) ? __int_as_float(0x7fffffff)
                                : __double2float_rn(__ddiv_rn(__dmul_rn(__ll2double_rn((long long)sums[4 * c + i]),
                                                                        0x1p-32), cells));
    if (ux_out) put_field(ux_out + orow + C, mean[0], 0.0f);
    if (uy_out) put_field(uy_out + orow + C, mean[1], 0.0f);
    if (u_out) put_field(u_out + orow + C, mean[2], 0.0f);
    if (p_out) put_field(p_out + orow + C, mean[3], p0);
  }
}

// K14 lbm_obstacle_force: the momentum-exchange force on the solid cells of each box
// (lbm_gpu_obstacle_force, include/lbm_gpu.h).  A link is a solid cell x_s and a speed d whose
// neighbour x_s + c_d is fluid; it adds -c_d * (f~_d(x_s) + f~_opp(d)(x_s + c_d)) to every box
// that holds x_s, which is the header's formula regrouped by link.  f~ is the stored lattice,
// and the side row on row ny-2.
//
// Each block serves one box: the host gives every box as many blocks as its mask words in this
// slab need (at most one resident wave), from first block `first` on.  A thread takes one 32-cell
// mask word of the box at a time (grid-stride over the box's words only), keeps the word's solid
// cells that lie in the box's columns, and finds their links with word-wide bit operations on the
// mask words of rows r-1, r, r+1 and their neighbouring words (periodic at nx, not at the pitch).
// A word without links in the box reads no lattice value, so a box costs its own mask words plus
// its boundary cells.  Rows r-1 and r+1:
//   whole   the slab holds the whole grid: they wrap inside the slab (K1a-f16 reads them so);
//   else    rows -1 and `rows` are the depth-0 ghost rows (planes 2,5,6 and 4,7,8, already
//           accelerated, exactly the ones a pull across the edge needs) and their mask words
//           are the ghost mask.
// Each value enters as round_half_even(v * 2^32), the digest's conversion.  A thread keeps signed
// 128-bit sums of its box's components in registers; the warp adds them with shuffles, the block
// in shared memory, and the block's sums go into `out` as two 64-bit words with the carry of the
// low word added to the high one: exact modulo 2^128 in any order.  A value that is not finite or
// of magnitude 2^31 or more marks the box instead.
constexpr int kForceThreads = 256;
constexpr int kForceMaxBoxes = 256;
constexpr int kForceOutWords = 5;                    // per box: fx lo, fx hi, fy lo, fy hi, mark

// one box's share of the launch, in this slab's local coordinates (lbm_gpu.cu fills it)
struct ForceBox {
  int first, blocks;                                 // its blocks: [first, first + blocks)
  int r0, w0, nw;                                    // local rows from r0, mask words [w0, w0 + nw) of each
  int x0, x1;                                        // its columns [x0, x1)
  long long words;                                   // rows x nw
};

template <typename store, typename val>
struct ForceArgs {
  const store* buf;                                  // lattice buffer of the current state
  const val* side;                                   // its side row
  const val* ghost_s;                                // depth-0 ghost rows -1 and `rows` (not whole)
  const val* ghost_n;
  const uint32_t* mask;
  const uint32_t* ghost_mask;                        // mask words of rows -1 and `rows` (not whole)
  const ForceBox* boxes;                             // n_boxes
  unsigned long long* out;                           // n_boxes x kForceOutWords
  long long plane_stride;
  int nx, rows, pitch, mask_pitch, accel_row, n_boxes;
  bool whole;
  RestShift rest;
};

__device__ __forceinline__ void add_i128(unsigned long long* p, const __int128 v) {
  const unsigned long long lo = (unsigned long long)v, hi = (unsigned long long)(v >> 64);
  const unsigned long long old = atomicAdd(p, lo);
  const unsigned long long h = hi + (old + lo < old ? 1ULL : 0ULL);
  if (h) atomicAdd(p + 1, h);
}

template <typename store, typename val>
__device__ __forceinline__ const uint32_t* force_mask_row(const ForceArgs<store, val>& a, int r) {
  if (a.whole) return a.mask + (long long)(r < 0 ? r + a.rows : r >= a.rows ? r - a.rows : r) * a.mask_pitch;
  if (r < 0) return a.ghost_mask;
  if (r >= a.rows) return a.ghost_mask + a.mask_pitch;
  return a.mask + (long long)r * a.mask_pitch;
}

// f~_k at local row r (-1 .. rows), column x
template <typename store, typename val>
__device__ __forceinline__ val force_value(const ForceArgs<store, val>& a, const int k, int r, const int x) {
  if (a.whole) {
    r = r < 0 ? r + a.rows : r >= a.rows ? r - a.rows : r;
  } else {
    if (r < 0) return a.ghost_s[(long long)k * a.pitch + x];
    if (r >= a.rows) return a.ghost_n[(long long)k * a.pitch + x];
  }
  if (r == a.accel_row && k != 0 && k != 2 && k != 4) {
    const int idx = (k == 1) ? 0 : (k == 3) ? 1 : k - 3;       // side row order 1,3,5,6,7,8
    return a.side[(long long)idx * a.pitch + x];
  }
  return stored_value(a.buf + k * a.plane_stride + (long long)r * a.pitch + x, k, a.rest);
}

// round_half_even(v * 2^32) into acc; false when v has no fixed-point value
template <typename val>
__device__ __forceinline__ bool force_fixed(const val v, long long& q) {
  if (!(::fabs((double)v) < 2147483648.0)) return false;
  q = __double2ll_rn((double)v * 4294967296.0);
  return true;
}

__device__ __forceinline__ __int128 warp_sum_i128(__int128 v) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const unsigned long long lo = __shfl_down_sync(0xffffffffu, (unsigned long long)v, off);
    const unsigned long long hi = __shfl_down_sync(0xffffffffu, (unsigned long long)(v >> 64), off);
    v += (__int128)(((unsigned __int128)hi << 64) | lo);
  }
  return v;
}

template <typename store, typename val>
__global__ void __launch_bounds__(kForceThreads) lbm_obstacle_force(const ForceArgs<store, val> a) {
  __shared__ unsigned long long acc[4];
  __shared__ unsigned mark;
  __shared__ int box_of_block;
  if (threadIdx.x == 0) {                            // the box whose blocks hold this one
    int lo = 0, hi = a.n_boxes - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (a.boxes[mid].first <= (int)blockIdx.x) lo = mid; else hi = mid - 1;
    }
    box_of_block = lo;
    mark = 0u;
  }
  if (threadIdx.x < 4) acc[threadIdx.x] = 0ULL;
  __syncthreads();
  const int j = box_of_block;
  const ForceBox bx = a.boxes[j];
  __int128 sx = 0, sy = 0;
  bool bad = false;
  const int wpr = (a.nx + 31) >> 5;
  const int last = (a.nx - 1) & 31;                  // bit of column nx-1 in the row's last word
  const long long stride = (long long)bx.blocks * blockDim.x;
  for (long long i = (long long)(blockIdx.x - bx.first) * blockDim.x + threadIdx.x; i < bx.words; i += stride) {
    const int rr = (int)(i / bx.nw), w = bx.w0 + (int)(i - (long long)rr * bx.nw);
    const int r = bx.r0 + rr;
    const uint32_t* m0 = force_mask_row(a, r);
    // solid cells of the word inside the box's columns
    const int lo = ::max(bx.x0 - 32 * w, 0), hi = ::min(bx.x1 - 32 * w, 32);
    const uint32_t cols = (hi >= 32 ? 0xffffffffu : (1u << hi) - 1u) & ~((1u << lo) - 1u);
    const uint32_t s = m0[w] & cols;
    if (!s) continue;
    // for row dy = -1, 0, 1: the mask at x (c), x + 1 (e) and x - 1 (wv) for the 32 columns of word w
    uint32_t c[3], e[3], wv[3];
#pragma unroll
    for (int dy = 0; dy < 3; dy++) {
      const uint32_t* m = dy == 1 ? m0 : force_mask_row(a, r + dy - 1);
      c[dy] = m[w];
      e[dy] = (c[dy] >> 1) | (w + 1 < wpr ? m[w + 1] << 31 : 0u);
      if (w == wpr - 1) e[dy] |= (m[0] & 1u) << last;
      wv[dy] = (c[dy] << 1) | (w > 0 ? m[w - 1] >> 31 : (m[wpr - 1] >> last) & 1u);
    }
    // solid cells of the word whose neighbour along speed d is fluid (c_d = (dx, dy), d = 1..8)
    uint32_t link[9];
    link[0] = 0u;
    link[1] = s & ~e[1];  link[2] = s & ~c[2];  link[3] = s & ~wv[1]; link[4] = s & ~c[0];
    link[5] = s & ~e[2];  link[6] = s & ~wv[2]; link[7] = s & ~wv[0]; link[8] = s & ~e[0];
    uint32_t any = 0u;
#pragma unroll
    for (int d = 1; d < 9; d++) any |= link[d];
    while (any) {
      const int b = __ffs(any) - 1;
      any &= any - 1;
      const int x = w * 32 + b;
#pragma unroll
      for (int d = 1; d < 9; d++) {
        if (!((link[d] >> b) & 1u)) continue;
        const int dx = (d == 1 || d == 5 || d == 8) ? 1 : (d == 3 || d == 6 || d == 7) ? -1 : 0;
        const int dy = (d == 2 || d == 5 || d == 6) ? 1 : (d == 4 || d == 7 || d == 8) ? -1 : 0;
        const int opp = (d < 5) ? ((d + 1) & 3) + 1 : ((d - 3) & 3) + 5;
        const int xn = x + dx < 0 ? a.nx - 1 : x + dx >= a.nx ? 0 : x + dx;
        long long q0 = 0, q1 = 0;
        bad |= !force_fixed(force_value(a, d, r, x), q0);
        bad |= !force_fixed(force_value(a, opp, r + dy, xn), q1);
        const __int128 q = (__int128)q0 + q1;
        if (dx > 0) sx -= q; else if (dx < 0) sx += q;
        if (dy > 0) sy -= q; else if (dy < 0) sy += q;
      }
    }
  }
  // warp sums, one shared atomic per warp and component, one global per block
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) mark = 1u;
  sx = warp_sum_i128(sx);
  sy = warp_sum_i128(sy);
  if ((threadIdx.x & 31) == 0) {
    if (sx) add_i128(&acc[0], sx);
    if (sy) add_i128(&acc[2], sy);
  }
  __syncthreads();
  unsigned long long* o = a.out + (long long)j * kForceOutWords;
  if (threadIdx.x < 2) {
    const __int128 v = (__int128)(((unsigned __int128)acc[2 * threadIdx.x + 1] << 64) | acc[2 * threadIdx.x]);
    if (v) add_i128(o + 2 * threadIdx.x, v);
  }
  if (threadIdx.x == 0 && mark) atomicOr(o + 4, 1ULL);
}

// Digest of the lattice rows [r0, r0+nrows): two wrapping 64-bit integer sums, so they
// are exact, order-independent and additive over slabs / ranks.
//   mass      sum over cells and speeds of round(f * 2^32): total_density of the reference
//             (d2q9-bgk.c:2900-2916) in fixed point -- stays constant step after step;
//   checksum  sum of bit_pattern(f_k(cell)) * odd_weight(global cell index, k): equal for
//             two lattices iff (up to 2^-64) every speed of every cell has the same bits,
//             whatever the decomposition.  Full-size stand-in for a lattice comparison.
// A value that is NaN, infinite or of magnitude 2^31 or more has no fixed-point mass: it adds
// nothing to the mass and sets out[2], and the host reports total_density as NaN.
__device__ __forceinline__ unsigned long long bits_of(float f) { return (unsigned long long)__float_as_uint(f); }
__device__ __forceinline__ unsigned long long bits_of(double f) { return (unsigned long long)__double_as_longlong(f); }

template <typename real, typename store = real>
__global__ void lbm_digest(const store* __restrict__ buf, long long plane_stride, int pitch, int nx, int r0,
                           int nrows, long long global_row0,
                           unsigned long long* out /* [mass, checksum, non-finite mark] */,
                           RestShift rest = RestShift()) {
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long mass = 0ULL, sum = 0ULL;
  bool bad = false;
  if (n < (long long)nrows * nx) {
    const int row = (int)(n / nx);
    const int x = (int)(n - (long long)row * nx);
    const unsigned long long g = (unsigned long long)(global_row0 + row) * (unsigned long long)nx + (unsigned long long)x;
#pragma unroll
    for (int k = 0; k < 9; k++) {
      const real f = stored_value(buf + k * plane_stride + (long long)(r0 + row) * pitch + x, k, rest);
      if (::fabs((double)f) < 2147483648.0) mass += (unsigned long long)__double2ll_rn((double)f * 4294967296.0);
      else bad = true;
      const unsigned long long w = (g * 0x9E3779B97F4A7C15ULL + (unsigned long long)(k + 1) * 0xC2B2AE3D27D4EB4FULL) | 1ULL;
      sum += bits_of(f) * w;
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    mass += __shfl_down_sync(0xffffffffu, mass, off);
    sum += __shfl_down_sync(0xffffffffu, sum, off);
  }
  if ((threadIdx.x & 31) == 0) {
    if (mass) atomicAdd(out + 0, mass);
    if (sum) atomicAdd(out + 1, sum);
  }
  if (bad) atomicOr(out + 2, 1ULL);
}

}  // namespace lbm
