// cta_f32.cuh — the rectangle heads×tails of a single-monomer trial in FP32 ("ΔU … in fp32 with a stated tolerance").
//
// Opt-in (pmc_set_pair_precision, default FP64).  Only the rectangle — idx·(n−1−idx) pairs whose dipoles do not change
// and whose separation changes by the rigid translation D of the tail — is evaluated in single precision; the row
// {idx}×rest (n−1 pairs, both μ_idx and the separation change), the chain state, the running energy, the acceptance test
// and all accumulators stay FP64.  What makes FP32 accurate enough here:
//   * positions are mirrored RELATIVE TO x_idx, rebuilt from the FP64 master copy for every trial, as a PAIR of floats
//     (hi = fl(d), lo = fl(d − hi)): the representation error of an offset is ~4e-15·|d| instead of 6e-8·|d|, and
//     r_ij = (hi_i − hi_j) + (lo_i − lo_j) carries the rounding error of ONE float subtraction, relative to |r_ij| itself —
//     also for two monomers that nearly touch far away from the rotated one (the large terms);
//   * μ_L·r' = μ_L·r − μ_L·D and μ_B·r' = μ_B·r − μ_B·D keep their FP64 structure, every factor carries a relative
//     error of a few 1e-7, and a pair contributes (new − old) with an absolute error of a few 1e-7 of its own magnitude;
//   * the partial sums leave FP32 after kFlush = 32 terms (FP64 accumulators per thread, FP64 reduction);
//   * what remains is r' = r − D, a float difference of floats: its error relative to |r'| is amplified by
//     (|r| + |D|) / |r'| when a trial brings two monomers much closer than they were — then the new term is huge.
// Stated tolerance (include/polymc.h, tests/test_gpu_fp32.py): error ≤ 2e-6·(1 + amplification) of the magnitude of
// each pair term (the sum of the magnitudes of its two parts, μ·μ/r³ and 3(μ·r̂)(μ·r̂)/r³).
// Measured on C2 (4096 chains × 500 trials): 14.0 M updates/s against 7.8 M in FP64; rectangle alone 1.89×
// (tools/rect_bench_f32.cu).  Without the lo parts it would be 16.0 M (rectangle 2.25×) — and wrong by 6e-8·|offset|/|r| per
// term, i.e. useless for long stretched chains; chunk length and accumulation scheme (profiles/r02c_tune_kflush.txt)
// change the speed by < 4 %.
// MUFU.RSQ (rsqrt.approx.f32, 2 ulp) needs no Newton step at this tolerance: 39 FP32 + 2 MUFU per pair against 43 FP64.
// Included by cta_kernels.cuh between its building blocks (CtaView, Team, pair_g, block_sum) and its kernels.
#pragma once

#ifndef PMC_CTA_BUILDING_BLOCKS
#error "include cta_kernels.cuh, which includes this file after its building blocks"
#endif

namespace pmc {

// Mirrors of the staged chain in shared memory, 40 B per monomer: two float4 arrays of their own and a float2 array
// that lives in the FP64 E array of the staged chain (8 B per monomer, unused by this path) — 32 B per monomer of extra
// shared memory, which is what lets four CTAs of the C2 shape share an SM (52 KB each).
struct F32View {
  float4* pa;   // hi parts of {x − x_idx, y − y_idx, z − z_idx}, w: e = μ·D_eff — rebuilt every trial
  float4* pb;   // {μx, μy, μz} — follows the FP64 dipoles (written at load and on accept); w: lo part of the x offset
  float2* pc;   // lo parts of the y and z offsets — rebuilt every trial
};

__host__ __device__ inline size_t f32_smem_bytes(int n) { return (size_t)n * 2 * sizeof(float4); }

__device__ __forceinline__ F32View carve_f32(unsigned char* base, int n, double* E) {
  F32View F;
  F.pa = reinterpret_cast<float4*>(base);
  F.pb = F.pa + n;
  F.pc = reinterpret_cast<float2*>(E);
  return F;
}

__device__ __forceinline__ float rsqrt_f32(float x) {
  float y;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

struct LaneItemF {
  float x, y, z;     // offset from x_idx, hi part
  float lx, ly, lz;  // … lo part
  float ax, ay, az;  // μ
  float tx, ty, tz;  // −3μ
  float c;           // −3μ·D
};

__device__ __forceinline__ LaneItemF load_lane_item_f32(const F32View& F, int L, float Dx, float Dy, float Dz) {
  const float4 a = F.pa[L], u = F.pb[L];
  const float2 l = F.pc[L];
  LaneItemF it;
  it.x = a.x; it.y = a.y; it.z = a.z;
  it.lx = u.w; it.ly = l.x; it.lz = l.y;
  it.ax = u.x; it.ay = u.y; it.az = u.z;
  it.tx = -3.0f * u.x; it.ty = -3.0f * u.y; it.tz = -3.0f * u.z;
  it.c = fmaf(it.tz, Dz, fmaf(it.ty, Dy, it.tx * Dx));
  return it;
}

// new − old of one pair, the same 43-operation form as rect_pair (cta_kernels.cuh) with MUFU.RSQ for 1/|r|.
__device__ __forceinline__ float rect_pair_f32(const LaneItemF& it, const float4 a, const float4 u, const float2 l,
                                               float Dx, float Dy, float Dz, float acc) {
  const float rx = (it.x - a.x) + (it.lx - u.w), ry = (it.y - a.y) + (it.ly - l.x), rz = (it.z - a.z) + (it.lz - l.y);
  const float mm = fmaf(it.az, u.z, fmaf(it.ay, u.y, it.ax * u.x));
  const float r2 = fmaf(rz, rz, fmaf(ry, ry, rx * rx));
  const float a3 = fmaf(it.tz, rz, fmaf(it.ty, ry, it.tx * rx));
  const float bb = fmaf(u.z, rz, fmaf(u.y, ry, u.x * rx));
  const float qx = rx - Dx, qy = ry - Dy, qz = rz - Dz;
  const float q2 = fmaf(qz, qz, fmaf(qy, qy, qx * qx));
  const float a3n = a3 - it.c;
  const float bn = bb - a.w;
  const float y = rsqrt_f32(r2), yn = rsqrt_f32(q2);
  const float y2 = y * y, yn2 = yn * yn;
  const float t = fmaf(a3 * bb, y2, mm);
  const float tn = fmaf(a3n * bn, yn2, mm);
  acc = fmaf(tn, yn2 * yn, acc);
  return fmaf(-t, y2 * y, acc);
}

// FP32 partial sums are folded into FP64 after this many terms: once a large term is in a float accumulator every later
// addition rounds at 6e-8 of the PARTIAL SUM, so the error grows with the number of terms that follow it
// Two lane items in the two halves of packed f32x2 operands (Blackwell add/mul/fma.f32x2: one issue slot for two FP32
// operations); the broadcast item is replicated into both halves.  Same operations in the same order as rect_pair_f32,
// bit-identical results.  MEASURED NEGATIVE, off by default (-DPMC_F32_PACKED=1 to build it): the loop is bound by the
// FP32 pipe, not by issue slots — FFMA2 occupies the pipe twice as long as FFMA — so the rectangle alone gains 2.5 %
// (607 vs 592 G pairs/s, tools/rect_bench_f32.cu) and the full kernel spills 68 B at its 128 registers.
#ifndef PMC_F32_PACKED
#define PMC_F32_PACKED 0
#endif
struct LanePairF {
  float2 x, y, z, lx, ly, lz, ax, ay, az, tx, ty, tz, c;
};

__device__ __forceinline__ LanePairF pack_lane_items(const LaneItemF& p, const LaneItemF& q) {
  LanePairF r;
  r.x = make_float2(p.x, q.x); r.y = make_float2(p.y, q.y); r.z = make_float2(p.z, q.z);
  r.lx = make_float2(p.lx, q.lx); r.ly = make_float2(p.ly, q.ly); r.lz = make_float2(p.lz, q.lz);
  r.ax = make_float2(p.ax, q.ax); r.ay = make_float2(p.ay, q.ay); r.az = make_float2(p.az, q.az);
  r.tx = make_float2(p.tx, q.tx); r.ty = make_float2(p.ty, q.ty); r.tz = make_float2(p.tz, q.tz);
  r.c = make_float2(p.c, q.c);
  return r;
}

__device__ __forceinline__ float2 dup2(float v) { return make_float2(v, v); }
__device__ __forceinline__ float2 neg2(float2 v) { return make_float2(-v.x, -v.y); }
__device__ __forceinline__ float2 sub2(float2 a, float2 b) { return __fadd2_rn(a, neg2(b)); }

__device__ __forceinline__ float2 rect_pair_f32x2(const LanePairF& it, const float4 a, const float4 u, const float2 l,
                                                  float2 Dx, float2 Dy, float2 Dz, float2 acc) {
  // −(broadcast) once per item and half: a − b = a + (−b) keeps every step a packed add
  const float2 nax = dup2(-a.x), nay = dup2(-a.y), naz = dup2(-a.z);
  const float2 nlx = dup2(-u.w), nly = dup2(-l.x), nlz = dup2(-l.y);
  const float2 ux = dup2(u.x), uy = dup2(u.y), uz = dup2(u.z);
  const float2 rx = __fadd2_rn(__fadd2_rn(it.x, nax), __fadd2_rn(it.lx, nlx));
  const float2 ry = __fadd2_rn(__fadd2_rn(it.y, nay), __fadd2_rn(it.ly, nly));
  const float2 rz = __fadd2_rn(__fadd2_rn(it.z, naz), __fadd2_rn(it.lz, nlz));
  const float2 mm = __ffma2_rn(it.az, uz, __ffma2_rn(it.ay, uy, __fmul2_rn(it.ax, ux)));
  const float2 r2 = __ffma2_rn(rz, rz, __ffma2_rn(ry, ry, __fmul2_rn(rx, rx)));
  const float2 a3 = __ffma2_rn(it.tz, rz, __ffma2_rn(it.ty, ry, __fmul2_rn(it.tx, rx)));
  const float2 bb = __ffma2_rn(uz, rz, __ffma2_rn(uy, ry, __fmul2_rn(ux, rx)));
  const float2 qx = sub2(rx, Dx), qy = sub2(ry, Dy), qz = sub2(rz, Dz);
  const float2 q2 = __ffma2_rn(qz, qz, __ffma2_rn(qy, qy, __fmul2_rn(qx, qx)));
  const float2 a3n = sub2(a3, it.c);
  const float2 bn = __fadd2_rn(bb, dup2(-a.w));
  const float2 y = make_float2(rsqrt_f32(r2.x), rsqrt_f32(r2.y));
  const float2 yn = make_float2(rsqrt_f32(q2.x), rsqrt_f32(q2.y));
  const float2 y2 = __fmul2_rn(y, y), yn2 = __fmul2_rn(yn, yn);
  const float2 t = __ffma2_rn(__fmul2_rn(a3, bb), y2, mm);
  const float2 tn = __ffma2_rn(__fmul2_rn(a3n, bn), yn2, mm);
  acc = __ffma2_rn(tn, __fmul2_rn(yn2, yn), acc);
  return __ffma2_rn(neg2(t), __fmul2_rn(y2, y), acc);
}

constexpr int kFlush = 32;

// One pass over bundles of NL groups of 32 lane items (groups g0, g0+NL, …: `nb` bundles) against the B broadcast
// items; the (bundle, broadcast item) space is split evenly over the team's warps.  Returns this thread's share.
template <class TEAM, int NL>
__device__ __forceinline__ double rect_pass_f32(const F32View& F, int baseA, int A, int g0, int nb, int baseB, int B,
                                                float Dx, float Dy, float Dz) {
  constexpr int W = TEAM::kWarps;
  const int lane = TEAM::lane(), warp = TEAM::warp();
  const float4* __restrict__ pa = F.pa + baseB;
  const float4* __restrict__ pb = F.pb + baseB;
  const float2* __restrict__ pc = F.pc + baseB;
  const float2 D2x = make_float2(Dx, Dx), D2y = make_float2(Dy, Dy), D2z = make_float2(Dz, Dz);
  const int U = nb * B;
  int u = (int)(((long long)U * warp) / W);
  const int u1 = (int)(((long long)U * (warp + 1)) / W);
  double acc = 0.0;
  if (u >= u1) return acc;
  int bundle = u / B;
  int k = u - bundle * B;
  while (u < u1) {
    LaneItemF it[NL];
    bool valid[NL];
#pragma unroll
    for (int j = 0; j < NL; ++j) {
      const int l = (g0 + bundle * NL + j) * 32 + lane;
      valid[j] = l < A;
      it[j] = load_lane_item_f32(F, baseA + min(l, A - 1), Dx, Dy, Dz);
    }
    LanePairF pk[NL >= 2 ? NL / 2 : 1];
    if (NL >= 2 && PMC_F32_PACKED) {
#pragma unroll
      for (int j = 0; j < NL / 2; ++j) pk[j] = pack_lane_items(it[2 * j], it[2 * j + 1]);
    }
    const int kend = min(B, k + (u1 - u));
    u += kend - k;
    while (k < kend) {
      const int kc = min(kend, k + kFlush);
      if (NL >= 2 && PMC_F32_PACKED) {
        // two lane items per packed operand: add/mul/fma.f32x2 (sm_100) halve the FP32 issue slots; MUFU per half
        float2 a2[NL >= 2 ? NL / 2 : 1];
#pragma unroll
        for (int j = 0; j < NL / 2; ++j) a2[j] = make_float2(0.0f, 0.0f);
#pragma unroll(NL >= 4 ? 1 : 2)
        for (; k < kc; ++k) {
          const float4 va = pa[k], vu = pb[k];
          const float2 vl = pc[k];
#pragma unroll
          for (int j = 0; j < NL / 2; ++j) a2[j] = rect_pair_f32x2(pk[j], va, vu, vl, D2x, D2y, D2z, a2[j]);
        }
#pragma unroll
        for (int j = 0; j < NL / 2; ++j)   // chunk sums leave FP32 here
          acc += (valid[2 * j] ? (double)a2[j].x : 0.0) + (valid[2 * j + 1] ? (double)a2[j].y : 0.0);
      } else {
        float a[NL];
#pragma unroll
        for (int j = 0; j < NL; ++j) a[j] = 0.0f;
#pragma unroll(NL >= 4 ? 1 : 2)
        for (; k < kc; ++k) {
          const float4 va = pa[k], vu = pb[k];
          const float2 vl = pc[k];
#pragma unroll
          for (int j = 0; j < NL; ++j) a[j] = rect_pair_f32(it[j], va, vu, vl, Dx, Dy, Dz, a[j]);
        }
#pragma unroll
        for (int j = 0; j < NL; ++j) acc += valid[j] ? (double)a[j] : 0.0;   // chunk sums leave FP32 here
      }
    }
    k = 0;
    ++bundle;
  }
  return acc;
}

// Σ over the rectangle of (new − old), this thread's share; F.pa / F.pb hold the current trial's mirrors.
template <class TEAM>
__device__ __forceinline__ double rect_sum_f32(const F32View& F, int baseA, int A, int baseB, int B, float Dx, float Dy,
                                               float Dz) {
  const int G = (A + 31) >> 5;   // groups of 32 lane items
  const int n4 = G >> 2;
  double acc = 0.0;
  if (n4) acc += rect_pass_f32<TEAM, 4>(F, baseA, A, 0, n4, baseB, B, Dx, Dy, Dz);
  int g = n4 * 4;
  if (G - g >= 2) {
    acc += rect_pass_f32<TEAM, 2>(F, baseA, A, g, 1, baseB, B, Dx, Dy, Dz);
    g += 2;
  }
  if (G - g >= 1) acc += rect_pass_f32<TEAM, 1>(F, baseA, A, g, 1, baseB, B, Dx, Dy, Dz);
  return acc;
}

// Mirrors of one trial: offsets from x_idx and e = μ·D_eff for every monomer (the lane side ignores e).
template <class TEAM>
__device__ __forceinline__ void build_mirrors_f32(const CtaView& S, const F32View& F, int n, int idx, float ex, float ey,
                                                  float ez) {
  const double xi = S.sx[idx], yi = S.sy[idx], zi = S.sz[idx];
  for (int k = TEAM::ltid(); k < n; k += TEAM::kLocalThreads) {
    float4 u = F.pb[k];
    const double dx = S.sx[k] - xi, dy = S.sy[k] - yi, dz = S.sz[k] - zi;
    float4 a;
    a.x = (float)dx; a.y = (float)dy; a.z = (float)dz;
    a.w = fmaf(u.z, ez, fmaf(u.y, ey, u.x * ex));
    u.w = (float)(dx - (double)a.x);
    F.pa[k] = a;
    F.pb[k] = u;
    F.pc[k] = make_float2((float)(dy - (double)a.y), (float)(dz - (double)a.z));
  }
}

template <class TEAM>
__device__ __forceinline__ void fill_mu_f32(const CtaView& S, const F32View& F, int n) {
  for (int k = TEAM::ltid(); k < n; k += TEAM::kLocalThreads)
    F.pb[k] = make_float4((float)S.mx[k], (float)S.my[k], (float)S.mz[k], 0.0f);
}

// delta_pairs_partial (cta_kernels.cuh) with the rectangle in FP32; the row {idx}×rest stays FP64.  Contains one team
// barrier (mirrors visible).
template <class TEAM>
__device__ __forceinline__ double delta_pairs_partial_f32(const CtaView& S, const F32View& F, int n, double b, int idx,
                                                          double npx, double npy, double npz, double dnx, double dny,
                                                          double dnz) {
  constexpr int T = TEAM::kThreads;
  const int tid = TEAM::tid();
  const double Dx = b * dnx, Dy = b * dny, Dz = b * dnz;
  const double hx = 0.5 * Dx, hy = 0.5 * Dy, hz = 0.5 * Dz;
  const int H = idx, Tl = n - 1 - idx;
  const bool rect = H > 0 && Tl > 0;
  bool lanes_are_heads = true;
  if (rect) {   // lane side = the one that wastes fewer lanes (bundles of up to 4 groups of 32)
    const long long costH = (long long)((H + 31) >> 5) * Tl;
    const long long costT = (long long)((Tl + 31) >> 5) * H;
    lanes_are_heads = costH <= costT;
  }
  const double sgn = lanes_are_heads ? 1.0 : -1.0;
  const float ex = (float)(sgn * Dx), ey = (float)(sgn * Dy), ez = (float)(sgn * Dz);
  const int baseA = lanes_are_heads ? 0 : idx + 1, A = lanes_are_heads ? H : Tl;
  const int baseB = lanes_are_heads ? idx + 1 : 0, B = lanes_are_heads ? Tl : H;
  if (rect) build_mirrors_f32<TEAM>(S, F, n, idx, ex, ey, ez);
  double acc = 0.0;
  {
    const double xi = S.sx[idx], yi = S.sy[idx], zi = S.sz[idx];
    const double ox = S.mx[idx], oy = S.my[idx], oz = S.mz[idx];
    for (int j = tid; j < n; j += T) {
      if (j == idx) continue;
      const double rx = xi - S.sx[j], ry = yi - S.sy[j], rz = zi - S.sz[j];
      const double s = (j < idx) ? 1.0 : -1.0;
      const double ux = S.mx[j], uy = S.my[j], uz = S.mz[j];
      acc += pair_g(npx, npy, npz, ux, uy, uz, fma(s, hx, rx), fma(s, hy, ry), fma(s, hz, rz)) -
             pair_g(ox, oy, oz, ux, uy, uz, rx, ry, rz);
    }
  }
  TEAM::sync();  // mirrors visible
  if (rect) acc += rect_sum_f32<TEAM>(F, baseA, A, baseB, B, ex, ey, ez);
  return acc;
}

template <int T>
__device__ __forceinline__ double cta_delta_pairs_f32(const CtaView& S, const F32View& F, int n, double b, int idx,
                                                      double npx, double npy, double npz, double dnx, double dny,
                                                      double dnz) {
  const double acc = delta_pairs_partial_f32<Team<T / 32>>(S, F, n, b, idx, npx, npy, npz, dnx, dny, dnz);
  return block_sum<T>(acc, S.part, /*trailing_sync=*/false);
}

}  // namespace pmc
