// RoI warping, mask resize and mask pooling.
//
// Replaces the three MNC Caffe layers' Forward_gpu:
//   ROIWarping   caffe-mnc/src/caffe/layers/roi_warping_layer.cu:67-107 (+ bilinear :18-64)
//   MaskResize   caffe-mnc/src/caffe/layers/mask_resize_layer.cu:57-73  (+ bilinear :13-54)
//   MaskPooling  caffe-mnc/src/caffe/layers/mask_pooling_layer.cu:13-26
// in two forms:
//   *_nchw  : the layer contract itself (fp32 NCHW blobs in and out) -- what the ROIWarpingLayer /
//             MaskResizeLayer / MaskPoolingLayer host mirrors call and what the HBM microbench
//             (BASELINE.json config 4) times.  One CTA per (RoI, channel slab): the RoI's window of
//             the feature map is staged in shared memory once, interpolation tables are built once
//             per RoI, and every output element is written exactly once with coalesced 16 B stores
//             (the reference writes 3x the bytes: top + argmax_h + argmax_w).
//   *_split : the fused forms the batched engine uses on split-bf16 NHWC activations: warp (+ the
//             2x2 max pool of test.prototxt:494-505) straight to the 14x14 grid and the 7x7 box
//             pool in one pass, never materialising the (R,512,28,28) tensor; mask pooling fused
//             with its 2x2 pool.
// The bilinear arithmetic uses explicit round-to-nearest mul/add in the reference's operation order
// (weights first, then a left-to-right sum), so fp32 results equal the C oracle's bit for bit.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>

#include "mnc_b200.h"
#include "tri.cuh"
#include "launch_util.h"

namespace mnc {

struct AxisTap {
  int lo, hi;   // indices (relative to the staged window for the nchw kernel)
  float l, h;   // l = frac, h = 1 - frac
  int ok;       // 0: sample out of range -> output 0
};

// roi_warping_layer.cu:18-47 for one axis.
__device__ __forceinline__ AxisTap axis_tap(float x, int dim) {
  AxisTap t;
  t.ok = !(x < -0.5 || x > dim - 0.5);
  if (x <= 0) x = 0;
  int lo = static_cast<int>(x), hi;
  if (lo >= dim - 1) {
    hi = lo = dim - 1;
    x = static_cast<float>(lo);
  } else {
    hi = lo + 1;
  }
  t.lo = lo;
  t.hi = hi;
  t.l = __fsub_rn(x, static_cast<float>(lo));
  t.h = __fsub_rn(1.f, t.l);
  return t;
}

__device__ __forceinline__ float bilerp(const AxisTap& th, const AxisTap& tw, float v1, float v2,
                                        float v3, float v4) {
  const float w1 = __fmul_rn(th.h, tw.h), w2 = __fmul_rn(th.h, tw.l);
  const float w3 = __fmul_rn(th.l, tw.h), w4 = __fmul_rn(th.l, tw.l);
  float val = __fmul_rn(w1, v1);
  val = __fadd_rn(val, __fmul_rn(w2, v2));
  val = __fadd_rn(val, __fmul_rn(w3, v3));
  val = __fadd_rn(val, __fmul_rn(w4, v4));
  return val;
}

struct RoiGeom {
  int level;
  float start_h, start_w, bin_h, bin_w;
};

// roi_warping_layer.cu:78-90
__device__ __forceinline__ RoiGeom roi_geom(const float* roi, float spatial_scale, int ph_n,
                                            int pw_n) {
  RoiGeom g;
  g.level = static_cast<int>(roi[0]);
  const float sw = roundf(__fmul_rn(roi[1], spatial_scale));
  const float sh = roundf(__fmul_rn(roi[2], spatial_scale));
  const float ew = roundf(__fmul_rn(roi[3], spatial_scale));
  const float eh = roundf(__fmul_rn(roi[4], spatial_scale));
  const float rw = fmaxf(__fsub_rn(ew, sw), 0.f);
  const float rh = fmaxf(__fsub_rn(eh, sh), 0.f);
  g.start_h = sh;
  g.start_w = sw;
  g.bin_h = __fdiv_rn(rh, static_cast<float>(ph_n));
  g.bin_w = __fdiv_rn(rw, static_cast<float>(pw_n));
  return g;
}

// ------------------------------------------------------------------------ ROIWarping, NCHW fp32
constexpr int kWarpSlab = 16;    // channels per CTA
constexpr int kMaxPooled = 32;   // pooled_h, pooled_w <= 32

// One CTA per (RoI, 16-channel slab).  The per-RoI interpolation tables (row taps, column taps)
// are built once in shared memory; each thread then fixes EPT consecutive outputs of the P x P
// plane and keeps, in registers, their four gather offsets and four bilinear weights (weights
// formed first, as roi_warping_layer.cu:56 does).  The channel loop is then 4 read-only gathers
// (a RoI's window of one channel is <= 9.6 KB, L1-resident after first touch) + 7 un-fused fp32
// ops per output and one vector streaming store per EPT outputs: ~13 instructions per output
// instead of ~50 when offsets and weights are recomputed per element (profiles/README.md).
// Output bytes are written exactly once, coalesced (the reference also writes argmax_h/argmax_w).
template <int PH, int PW, int EPT>
__global__ void __launch_bounds__(256)
roi_warp_nchw_kernel(const float* __restrict__ feat, int C, int H, int W,
                     const float* __restrict__ rois, float spatial_scale,
                     float* __restrict__ out) {
  constexpr int PP = PH * PW;
  static_assert(PP % EPT == 0, "plane must split into whole vectors");
  constexpr int TPC = PP / EPT;         // threads per channel plane
  constexpr int CLN = 256 / TPC > 0 ? 256 / TPC : 1;  // channel lanes per CTA
  __shared__ AxisTap tap_h[PH], tap_w[PW];
  const int r = blockIdx.x;
  const int c0 = blockIdx.y * kWarpSlab;
  const int tid = threadIdx.x;
  const RoiGeom g = roi_geom(rois + static_cast<long long>(r) * 5, spatial_scale, PH, PW);
  if (tid < PH) tap_h[tid] = axis_tap(__fadd_rn(g.start_h, __fmul_rn(static_cast<float>(tid), g.bin_h)), H);
  if (tid >= 32 && tid < 32 + PW)
    tap_w[tid - 32] = axis_tap(__fadd_rn(g.start_w, __fmul_rn(static_cast<float>(tid - 32), g.bin_w)), W);
  __syncthreads();
  const int q = tid % TPC, cl = tid / TPC;
  if (cl >= CLN) return;
  int off[EPT][4];
  float wgt[EPT][4];
  bool ok[EPT];
#pragma unroll
  for (int e = 0; e < EPT; ++e) {
    const int i = q * EPT + e;
    const int ph = i / PW, pw = i - ph * PW;
    const AxisTap th = tap_h[ph], tw = tap_w[pw];
    ok[e] = th.ok && tw.ok;
    off[e][0] = ok[e] ? th.lo * W + tw.lo : 0;
    off[e][1] = ok[e] ? th.lo * W + tw.hi : 0;
    off[e][2] = ok[e] ? th.hi * W + tw.lo : 0;
    off[e][3] = ok[e] ? th.hi * W + tw.hi : 0;
    wgt[e][0] = __fmul_rn(th.h, tw.h);
    wgt[e][1] = __fmul_rn(th.h, tw.l);
    wgt[e][2] = __fmul_rn(th.l, tw.h);
    wgt[e][3] = __fmul_rn(th.l, tw.l);
  }
  const int nch = min(kWarpSlab, C - c0);
  const int HW = H * W;
  const float* fbase = feat + (static_cast<long long>(g.level) * C + c0) * HW;
  float* obase = out + (static_cast<long long>(r) * C + c0) * PP + q * EPT;
  const bool aligned = (reinterpret_cast<uintptr_t>(obase) & (EPT * 4 - 1)) == 0 && (PP % EPT == 0);
#pragma unroll 2
  for (int c = cl; c < nch; c += CLN) {
    const float* plane = fbase + static_cast<long long>(c) * HW;
    float v[EPT];
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      const float v1 = __ldg(plane + off[e][0]), v2 = __ldg(plane + off[e][1]);
      const float v3 = __ldg(plane + off[e][2]), v4 = __ldg(plane + off[e][3]);
      float val = __fmul_rn(wgt[e][0], v1);
      val = __fadd_rn(val, __fmul_rn(wgt[e][1], v2));
      val = __fadd_rn(val, __fmul_rn(wgt[e][2], v3));
      val = __fadd_rn(val, __fmul_rn(wgt[e][3], v4));
      v[e] = ok[e] ? val : 0.f;
    }
    float* o = obase + c * PP;
    if (EPT == 4 && aligned) {
      __stcs(reinterpret_cast<float4*>(o), make_float4(v[0], v[EPT > 1 ? 1 : 0], v[EPT > 2 ? 2 : 0], v[EPT > 3 ? 3 : 0]));
    } else if (EPT == 2 && aligned) {
      __stcs(reinterpret_cast<float2*>(o), make_float2(v[0], v[EPT > 1 ? 1 : 0]));
    } else {
#pragma unroll
      for (int e = 0; e < EPT; ++e) __stcs(o + e, v[e]);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// ROIWarping 28x28 with the RoI's feature window STAGED IN SHARED MEMORY (the design
// BASELINE.json's north_star names): one CTA per (RoI, 16-channel group).  The taps of a RoI only
// touch the window rows [r0, r1] x columns [c0, c1] of the map (<= 38 x 63 floats per channel);
// the CTA copies that window with 4-byte cp.async (all copies in flight together) for as many
// channels as fit a 48 KB budget (all 16 for a typical proposal, 4 for a full-map RoI), stored
// CHANNEL-PAIR INTERLEAVED: one 8-byte LDS returns a tap of two channels.  Every thread owns 4
// consecutive outputs of the 28 x 28 plane with their window offsets and bilinear weights in
// registers (weights formed first, products summed left to right: the operation order of
// roi_warping_layer.cu:56) and walks the channel pairs with PACKED fp32x2 arithmetic
// (__fmul2_rn / __fadd2_rn: two IEEE operations per instruction, no FMA contraction -- still
// bit-exact with the reference built with -fmad=false): 4 LDS.64 + 7 packed ops per TWO outputs
// instead of 4 LDG + 7 ops per output, one 16-byte streaming store per 4 outputs.  3.2 x fewer
// instructions per output than the gather kernel; the window is read once from L2 instead of
// ~7 times through L1.
constexpr int kStageGroup = 16;            // channels per CTA
constexpr int kStageFloats = 12 * 1024;    // 48 KB window budget

// Packed fp32x2 arithmetic WITHOUT fusion.  sm_100 has FMUL2 and FFMA2 but no packed add, and
// ptxas folds every mul.rn.f32x2 -> add.rn.f32x2 (or fma by a literal 1.0) chain into one FFMA2 --
// a single rounding, which would break bit-exactness with the reference's separately rounded
// products and sums (measured: -fmad=false does not stop it).  So the products are FMUL2 and each
// sum is fma(p, one, acc) with `one` = 1.0f handed in as a KERNEL ARGUMENT: p * 1.0 is exact, the
// fma rounds once = an IEEE add, and the compiler cannot see the value, so nothing is folded.
__device__ __forceinline__ float2 mul2_rn(float2 a, float2 b) {
  float2 r;
  asm("{\n\t.reg .b64 ra, rb, rc;\n\t"
      "mov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
      "mul.rn.f32x2 rc, ra, rb;\n\t"
      "mov.b64 {%0, %1}, rc;\n\t}"
      : "=f"(r.x), "=f"(r.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return r;
}
__device__ __forceinline__ float2 add2_rn(float2 a, float2 b, float one) {
  float2 r;
  asm("{\n\t.reg .b64 ra, rb, rc, ro;\n\t"
      "mov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 ro, {%6, %6};\n\t"
      "fma.rn.f32x2 rc, rb, ro, ra;\n\t"
      "mov.b64 {%0, %1}, rc;\n\t}"
      : "=f"(r.x), "=f"(r.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(one));
  return r;
}

// One staged pass of NP channel pairs: window layout [pixel][S] float2 with S = NP + 1 (the odd
// pitch spreads neighbouring pixels over the banks); a tap's pairs sit at compile-time offsets of
// its address, so the pair loop has no address arithmetic.
template <int NP>
__device__ __forceinline__ void warp28_pass(const float2* __restrict__ win2, const int (&off)[4][4],
                                            const float2 (&wgt)[4][4], const bool (&ok)[4],
                                            float* __restrict__ o, int n_c, float one) {
  constexpr int S = NP + 1, PP = 28 * 28;
  const float2* t[4][4];
#pragma unroll
  for (int e = 0; e < 4; ++e)
#pragma unroll
    for (int k = 0; k < 4; ++k) t[e][k] = win2 + off[e][k] * S;
#pragma unroll
  for (int p = 0; p < NP; ++p) {
    if (2 * p >= n_c) break;
    float2 v[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float2 val = mul2_rn(wgt[e][0], t[e][0][p]);
      val = add2_rn(val, mul2_rn(wgt[e][1], t[e][1][p]), one);
      val = add2_rn(val, mul2_rn(wgt[e][2], t[e][2][p]), one);
      val = add2_rn(val, mul2_rn(wgt[e][3], t[e][3][p]), one);
      v[e] = ok[e] ? val : make_float2(0.f, 0.f);
    }
    __stcs(reinterpret_cast<float4*>(o + 2 * p * PP), make_float4(v[0].x, v[1].x, v[2].x, v[3].x));
    if (2 * p + 1 < n_c)   // odd channel tail: the second half of the last pair holds stale data
      __stcs(reinterpret_cast<float4*>(o + (2 * p + 1) * PP), make_float4(v[0].y, v[1].y, v[2].y, v[3].y));
  }
}

__global__ void __launch_bounds__(256)
roi_warp28_stage_kernel(const float* __restrict__ feat, int C, int H, int W,
                        const float* __restrict__ rois, float spatial_scale, float* __restrict__ out,
                        float one) {
  constexpr int P = 28, PP = P * P, EPT = 4, TPC = PP / EPT;   // 196 threads compute
  extern __shared__ float2 win2[];                             // [pixel][pairs + 1] (2 channels)
  __shared__ AxisTap tap_h[P], tap_w[P];
  __shared__ int bounds[4];
  const int r = blockIdx.x;
  const int cg0 = blockIdx.y * kStageGroup;
  const int tid = threadIdx.x;
  const RoiGeom g = roi_geom(rois + static_cast<long long>(r) * 5, spatial_scale, P, P);
  if (tid < P) tap_h[tid] = axis_tap(__fadd_rn(g.start_h, __fmul_rn(static_cast<float>(tid), g.bin_h)), H);
  if (tid >= 32 && tid < 32 + P)
    tap_w[tid - 32] = axis_tap(__fadd_rn(g.start_w, __fmul_rn(static_cast<float>(tid - 32), g.bin_w)), W);
  __syncthreads();
  if (tid < 32) {   // window bounds: warp-wide min / max over the valid taps
    int r0 = H, r1 = -1, c0 = W, c1 = -1;
    if (tid < P) {
      if (tap_h[tid].ok) { r0 = tap_h[tid].lo; r1 = tap_h[tid].hi; }
      if (tap_w[tid].ok) { c0 = tap_w[tid].lo; c1 = tap_w[tid].hi; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      r0 = min(r0, __shfl_xor_sync(0xffffffffu, r0, o));
      r1 = max(r1, __shfl_xor_sync(0xffffffffu, r1, o));
      c0 = min(c0, __shfl_xor_sync(0xffffffffu, c0, o));
      c1 = max(c1, __shfl_xor_sync(0xffffffffu, c1, o));
    }
    if (tid == 0) { bounds[0] = r0; bounds[1] = r1; bounds[2] = c0; bounds[3] = c1; }
  }
  __syncthreads();
  const int r0 = bounds[0], r1 = bounds[1], c0 = bounds[2], c1 = bounds[3];
  const int nch = min(kStageGroup, C - cg0);
  const int q = tid;                       // output quad (threads >= TPC only help staging)
  float* obase = out + (static_cast<long long>(r) * C + cg0) * PP + q * EPT;
  if (r1 < r0 || c1 < c0) {                // no sample inside the map: the RoI's output is zero
    if (q < TPC)
      for (int c = 0; c < nch; ++c)
        __stcs(reinterpret_cast<float4*>(obase + c * PP), make_float4(0.f, 0.f, 0.f, 0.f));
    return;
  }
  const int wh = r1 - r0 + 1, ww = c1 - c0 + 1;
  const int per_ch = wh * ww;
  // pairs per pass: the largest of 8 / 4 / 2 / 1 whose padded window fits the budget
  // (a full 38 x 63 map: 2394 px x 2 float2 x 8 B = 38 KB -> 1 pair)
  const int budget_px = (kStageFloats / 2) / per_ch;    // float2 slots per pixel
  const int np = budget_px >= 9 ? 8 : (budget_px >= 5 ? 4 : (budget_px >= 3 ? 2 : 1));
  const int S = np + 1;
  int off[EPT][4];
  float2 wgt[EPT][4];
  bool ok[EPT];
  if (q < TPC) {
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      const int i = q * EPT + e;
      const int ph = i / P, pw = i - ph * P;
      const AxisTap th = tap_h[ph];
      const AxisTap tw = tap_w[pw];
      ok[e] = th.ok && tw.ok;
      const int lo_h = ok[e] ? th.lo - r0 : 0, hi_h = ok[e] ? th.hi - r0 : 0;
      const int lo_w = ok[e] ? tw.lo - c0 : 0, hi_w = ok[e] ? tw.hi - c0 : 0;
      off[e][0] = lo_h * ww + lo_w;
      off[e][1] = lo_h * ww + hi_w;
      off[e][2] = hi_h * ww + lo_w;
      off[e][3] = hi_h * ww + hi_w;
      const float w1 = __fmul_rn(th.h, tw.h), w2 = __fmul_rn(th.h, tw.l);
      const float w3 = __fmul_rn(th.l, tw.h), w4 = __fmul_rn(th.l, tw.l);
      wgt[e][0] = make_float2(w1, w1);
      wgt[e][1] = make_float2(w2, w2);
      wgt[e][2] = make_float2(w3, w3);
      wgt[e][3] = make_float2(w4, w4);
    }
  }
  const int HW = H * W;
  const float* fbase = feat + (static_cast<long long>(g.level) * C + cg0) * HW + r0 * W + c0;
  float* winf = reinterpret_cast<float*>(win2);
  for (int cb = 0; cb < nch; cb += 2 * np) {
    const int n_c = min(2 * np, nch - cb);
    {  // stage: thread = (column, row lane); channel ch -> half (ch & 1) of pair (ch >> 1)
      const int x = tid & 63, rl = tid >> 6;
      if (x < ww) {
        int ch = 0, y = rl;
        while (y >= wh) { y -= wh; ++ch; }
        while (ch < n_c) {
          const float* src = fbase + static_cast<long long>(cb + ch) * HW + y * W + x;
          const uint32_t dst = static_cast<uint32_t>(
              __cvta_generic_to_shared(winf + (((y * ww + x) * S + (ch >> 1)) << 1) + (ch & 1)));
          asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
          y += 4;
          while (y >= wh) { y -= wh; ++ch; }
        }
      }
      asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();
    if (q < TPC) {
      float* o = obase + cb * PP;
      if (np == 8) warp28_pass<8>(win2, off, wgt, ok, o, n_c, one);
      else if (np == 4) warp28_pass<4>(win2, off, wgt, ok, o, n_c, one);
      else if (np == 2) warp28_pass<2>(win2, off, wgt, ok, o, n_c, one);
      else warp28_pass<1>(win2, off, wgt, ok, o, n_c, one);
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// ROIWarping by ROW WALK: a warp owns one output plane (RoI, channel); lane = output column pw, and
// the warp walks the P sample rows top to bottom.  The four taps of (ph, pw) are (row lo / hi) x
// (column lo / hi); consecutive sample rows advance by bin_h < 1.4 feature rows, so the two feature
// rows a lane needs are kept in registers and re-read only when the row taps move on -- ~2 loads
// per new feature row instead of 4 per output: 1.5 loads per output for a typical proposal, and
// each load is one coalesced row segment (lanes = neighbouring columns).  Control flow depends only
// on the RoI: the warp never diverges.  The value formula is unchanged (weights first, products
// summed left to right, no FMA): bit-exact with the reference built with -fmad=false.
// Stores: one 4 x P byte row segment per sample row, consecutive rows contiguous (whole plane
// written once, streaming).  P = 14 packs two planes into one warp (lanes 0-13 and 16-29).
template <int P, int CH = ((P > 16) ? 8 : 4)>   // CH: planes walked together by one lane (ILP; the row
                                                // bookkeeping and the 4 weights are shared; measured)
__global__ void __launch_bounds__(256)
roi_warp_rowwalk_kernel(const float* __restrict__ feat, int C, int H, int W,
                        const float* __restrict__ rois, float spatial_scale, int ch_per_cta,
                        float* __restrict__ out) {
  constexpr int PP = P * P;
  constexpr int PPW = (P <= 16) ? 2 : 1;          // plane groups per warp
  __shared__ int4 tap_hq[P];                      // {lo (or -1: out of range), hi, bits(h), bits(l)}
  const int r = blockIdx.x;
  const int cbase = blockIdx.y * ch_per_cta;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const RoiGeom g = roi_geom(rois + static_cast<long long>(r) * 5, spatial_scale, P, P);
  if (tid < P) {
    const AxisTap t = axis_tap(__fadd_rn(g.start_h, __fmul_rn(static_cast<float>(tid), g.bin_h)), H);
    tap_hq[tid] = make_int4(t.ok ? t.lo : -1, t.hi, __float_as_int(t.h), __float_as_int(t.l));
  }
  const int sub = (PPW == 2) ? (lane >> 4) : 0;     // which plane group of the warp
  const int pw = (PPW == 2) ? (lane & 15) : lane;
  const bool live = pw < P;
  const AxisTap tw = axis_tap(__fadd_rn(g.start_w, __fmul_rn(static_cast<float>(live ? pw : 0), g.bin_w)), W);
  __syncthreads();
  const int HW = H * W;
  const int nch = min(ch_per_cta, C - cbase);
  const int nwarps = blockDim.x >> 5;
  for (int c = (warp * PPW + sub) * CH; c < nch; c += nwarps * PPW * CH) {
    const float* plane = feat + (static_cast<long long>(g.level) * C + cbase + c) * HW;
    float* o = out + (static_cast<long long>(r) * C + cbase + c) * PP + pw;
    int koff[CH];                                   // plane offsets (a channel tail re-reads plane 0)
#pragma unroll
    for (int k = 0; k < CH; ++k) koff[k] = (c + k < nch ? k : 0) * HW;
    int cur_lo = -1, cur_hi = -1;
    float a_lo[CH], a_hi[CH], b_lo[CH], b_hi[CH];   // rows cur_lo / cur_hi at columns lo / hi
#pragma unroll
    for (int k = 0; k < CH; ++k) a_lo[k] = a_hi[k] = b_lo[k] = b_hi[k] = 0.f;
#pragma unroll 2
    for (int ph = 0; ph < P; ++ph) {
      const int4 tq = tap_hq[ph];
      float val[CH];
#pragma unroll
      for (int k = 0; k < CH; ++k) val[k] = 0.f;
      if (tq.x >= 0) {
        if (tq.x != cur_lo) {
          if (tq.x == cur_hi) {
#pragma unroll
            for (int k = 0; k < CH; ++k) { a_lo[k] = b_lo[k]; a_hi[k] = b_hi[k]; }
          } else {
#pragma unroll
            for (int k = 0; k < CH; ++k) {
              a_lo[k] = __ldg(plane + koff[k] + tq.x * W + tw.lo);
              a_hi[k] = __ldg(plane + koff[k] + tq.x * W + tw.hi);
            }
          }
          cur_lo = tq.x;
          cur_hi = -1;
        }
        if (tq.y != cur_hi) {
          if (tq.y == tq.x) {
#pragma unroll
            for (int k = 0; k < CH; ++k) { b_lo[k] = a_lo[k]; b_hi[k] = a_hi[k]; }
          } else {
#pragma unroll
            for (int k = 0; k < CH; ++k) {
              b_lo[k] = __ldg(plane + koff[k] + tq.y * W + tw.lo);
              b_hi[k] = __ldg(plane + koff[k] + tq.y * W + tw.hi);
            }
          }
          cur_hi = tq.y;
        }
        const float th_h = __int_as_float(tq.z), th_l = __int_as_float(tq.w);
        const float w1 = __fmul_rn(th_h, tw.h), w2 = __fmul_rn(th_h, tw.l);
        const float w3 = __fmul_rn(th_l, tw.h), w4 = __fmul_rn(th_l, tw.l);
#pragma unroll
        for (int k = 0; k < CH; ++k) {
          float v = __fmul_rn(w1, a_lo[k]);
          v = __fadd_rn(v, __fmul_rn(w2, a_hi[k]));
          v = __fadd_rn(v, __fmul_rn(w3, b_lo[k]));
          v = __fadd_rn(v, __fmul_rn(w4, b_hi[k]));
          val[k] = tw.ok ? v : 0.f;
        }
      }
      if (live) {
#pragma unroll
        for (int k = 0; k < CH; ++k)
          if (c + k < nch) __stcs(o + k * PP + ph * P, val[k]);
      }
    }
  }
}

// generic pooled size (runtime), same scheme, scalar stores
__global__ void __launch_bounds__(256)
roi_warp_nchw_generic_kernel(const float* __restrict__ feat, int C, int H, int W,
                             const float* __restrict__ rois, int ph_n, int pw_n,
                             float spatial_scale, float* __restrict__ out) {
  __shared__ AxisTap tap_h[kMaxPooled], tap_w[kMaxPooled];
  const int r = blockIdx.x;
  const int c0 = blockIdx.y * kWarpSlab;
  const int tid = threadIdx.x;
  const RoiGeom g = roi_geom(rois + static_cast<long long>(r) * 5, spatial_scale, ph_n, pw_n);
  if (tid < ph_n) tap_h[tid] = axis_tap(__fadd_rn(g.start_h, __fmul_rn(static_cast<float>(tid), g.bin_h)), H);
  if (tid >= 32 && tid < 32 + pw_n)
    tap_w[tid - 32] = axis_tap(__fadd_rn(g.start_w, __fmul_rn(static_cast<float>(tid - 32), g.bin_w)), W);
  __syncthreads();
  const int pp = ph_n * pw_n;
  const int nch = min(kWarpSlab, C - c0);
  const float* fbase = feat + (static_cast<long long>(g.level) * C + c0) * H * W;
  float* obase = out + (static_cast<long long>(r) * C + c0) * pp;
  for (int i = tid; i < nch * pp; i += 256) {
    const int c = i / pp, rem = i % pp;
    const int ph = rem / pw_n, pw = rem % pw_n;
    const AxisTap th = tap_h[ph], tw = tap_w[pw];
    float val = 0.f;
    if (th.ok && tw.ok) {
      const float* pl = fbase + static_cast<long long>(c) * H * W;
      val = bilerp(th, tw, __ldg(pl + th.lo * W + tw.lo), __ldg(pl + th.lo * W + tw.hi),
                   __ldg(pl + th.hi * W + tw.lo), __ldg(pl + th.hi * W + tw.hi));
    }
    obase[i] = val;
  }
}

// -------------------------------------------------------------- MaskResize / MaskPooling, NCHW
__global__ void mask_resize_nchw_kernel(const float* __restrict__ in, int planes, int ih_n,
                                        int iw_n, int oh_n, int ow_n, float* __restrict__ out) {
  const long long total = static_cast<long long>(planes) * oh_n * ow_n;
  const float ratio_h = __fdiv_rn(static_cast<float>(ih_n), static_cast<float>(oh_n));
  const float ratio_w = __fdiv_rn(static_cast<float>(iw_n), static_cast<float>(ow_n));
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int w = static_cast<int>(i % ow_n);
    const int h = static_cast<int>((i / ow_n) % oh_n);
    const long long p = i / (static_cast<long long>(ow_n) * oh_n);
    const AxisTap th = axis_tap(__fmul_rn(static_cast<float>(h), ratio_h), ih_n);
    const AxisTap tw = axis_tap(__fmul_rn(static_cast<float>(w), ratio_w), iw_n);
    float val = 0.f;
    if (th.ok && tw.ok) {
      const float* b = in + p * ih_n * iw_n;
      val = bilerp(th, tw, b[th.lo * iw_n + tw.lo], b[th.lo * iw_n + tw.hi],
                   b[th.hi * iw_n + tw.lo], b[th.hi * iw_n + tw.hi]);
    }
    out[i] = val;
  }
}

// top[n,c,h,w] = feat[n,c,h,w] * mask[n,0,h,w]; 16-byte streaming loads/stores when hw % 4 == 0.
__global__ void mask_pool_nchw_kernel(const float* __restrict__ feat,
                                      const float* __restrict__ mask, int N, int C, int hw,
                                      float* __restrict__ out) {
  const long long total4 = static_cast<long long>(N) * C * hw / 4;
  const int hw4 = hw / 4;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int q = static_cast<int>(i % hw4);
    const long long n = i / (static_cast<long long>(hw4) * C);
    const float4 f = __ldcs(reinterpret_cast<const float4*>(feat) + i);
    const float4 m = __ldg(reinterpret_cast<const float4*>(mask) + n * hw4 + q);
    __stcs(reinterpret_cast<float4*>(out) + i,
           make_float4(__fmul_rn(f.x, m.x), __fmul_rn(f.y, m.y), __fmul_rn(f.z, m.z),
                       __fmul_rn(f.w, m.w)));
  }
}
__global__ void mask_pool_nchw_scalar_kernel(const float* __restrict__ feat,
                                             const float* __restrict__ mask, int N, int C, int hw,
                                             float* __restrict__ out) {
  const long long total = static_cast<long long>(N) * C * hw;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int q = static_cast<int>(i % hw);
    const long long n = i / (static_cast<long long>(hw) * C);
    out[i] = __fmul_rn(feat[i], mask[n * hw + q]);
  }
}

// ------------------------------------------------------------ fused forms on split-bf16 NHWC
__device__ __forceinline__ float2 ld_split2(const __nv_bfloat16* hi, const __nv_bfloat16* lo,
                                            long long off) {
  const uint32_t h = __ldg(reinterpret_cast<const uint32_t*>(hi + off));
  const uint32_t l = __ldg(reinterpret_cast<const uint32_t*>(lo + off));
  float2 r;
  r.x = __uint_as_float(h << 16) + __uint_as_float(l << 16);
  r.y = __uint_as_float(h & 0xffff0000u) + __uint_as_float(l & 0xffff0000u);
  return r;
}
__device__ __forceinline__ void st_split2(__nv_bfloat16* hi, __nv_bfloat16* lo, long long off,
                                          float a, float b) {
  const __nv_bfloat16 ha = __float2bfloat16_rn(a), hb = __float2bfloat16_rn(b);
  const __nv_bfloat16 la = __float2bfloat16_rn(a - __bfloat162float(ha));
  const __nv_bfloat16 lb = __float2bfloat16_rn(b - __bfloat162float(hb));
  *reinterpret_cast<uint32_t*>(hi + off) =
      static_cast<uint32_t>(__bfloat16_as_ushort(ha)) | (static_cast<uint32_t>(__bfloat16_as_ushort(hb)) << 16);
  *reinterpret_cast<uint32_t*>(lo + off) =
      static_cast<uint32_t>(__bfloat16_as_ushort(la)) | (static_cast<uint32_t>(__bfloat16_as_ushort(lb)) << 16);
}

// One CTA per (RoI, pair of 14x14 output rows).  SUB = 2: warp to 28x28 and take the 2x2 max
// (stage 1, test.prototxt:479-505); SUB = 1: warp straight to 14x14 (stage 2, :809-820).
// Also emits the 7x7 box-branch pool (test.prototxt:571-582).
// The interpolation taps depend only on (RoI, sample row/col): they are computed once per CTA
// into shared memory (2*SUB row taps, 14*SUB column taps).  Threads then run over
// (cell column, 4-channel group): 8-byte loads from each bf16 plane, coalesced along channels.
struct __align__(8) bf4 { uint32_t a, b; };
__device__ __forceinline__ float4 ld_split4(const __nv_bfloat16* hi, const __nv_bfloat16* lo,
                                            long long off) {
  const uint2 h = __ldg(reinterpret_cast<const uint2*>(hi + off));
  const uint2 l = __ldg(reinterpret_cast<const uint2*>(lo + off));
  float4 r;
  r.x = __uint_as_float(h.x << 16) + __uint_as_float(l.x << 16);
  r.y = __uint_as_float(h.x & 0xffff0000u) + __uint_as_float(l.x & 0xffff0000u);
  r.z = __uint_as_float(h.y << 16) + __uint_as_float(l.y << 16);
  r.w = __uint_as_float(h.y & 0xffff0000u) + __uint_as_float(l.y & 0xffff0000u);
  return r;
}
__device__ __forceinline__ uint32_t pack_bf2(__nv_bfloat16 a, __nv_bfloat16 b) {
  return static_cast<uint32_t>(__bfloat16_as_ushort(a)) | (static_cast<uint32_t>(__bfloat16_as_ushort(b)) << 16);
}
__device__ __forceinline__ void st_split4(__nv_bfloat16* hi, __nv_bfloat16* lo, long long off,
                                          const float4 v) {
  const __nv_bfloat16 h0 = __float2bfloat16_rn(v.x), h1 = __float2bfloat16_rn(v.y);
  const __nv_bfloat16 h2 = __float2bfloat16_rn(v.z), h3 = __float2bfloat16_rn(v.w);
  const __nv_bfloat16 l0 = __float2bfloat16_rn(v.x - __bfloat162float(h0));
  const __nv_bfloat16 l1 = __float2bfloat16_rn(v.y - __bfloat162float(h1));
  const __nv_bfloat16 l2 = __float2bfloat16_rn(v.z - __bfloat162float(h2));
  const __nv_bfloat16 l3 = __float2bfloat16_rn(v.w - __bfloat162float(h3));
  // streaming stores: the RoI feature tensors (~1.2 GB per stage) are consumed once by the next
  // GEMM and must not evict conv5_3 (39 MB, re-read by every RoI) from L2
  __stcs(reinterpret_cast<uint2*>(hi + off), make_uint2(pack_bf2(h0, h1), pack_bf2(h2, h3)));
  __stcs(reinterpret_cast<uint2*>(lo + off), make_uint2(pack_bf2(l0, l1), pack_bf2(l2, l3)));
}
// fused-path bilinear: same weights-first formula, evaluated with FMAs (the fused outputs are
// re-quantised to split-bf16 and compared at tolerance; the bit-exact form lives in bilerp()).
__device__ __forceinline__ float4 bilerp4(const float w1, const float w2, const float w3,
                                          const float w4, const float4 v1, const float4 v2,
                                          const float4 v3, const float4 v4) {
  float4 r;
  r.x = fmaf(w4, v4.x, fmaf(w3, v3.x, fmaf(w2, v2.x, w1 * v1.x)));
  r.y = fmaf(w4, v4.y, fmaf(w3, v3.y, fmaf(w2, v2.y, w1 * v1.y)));
  r.z = fmaf(w4, v4.z, fmaf(w3, v3.z, fmaf(w2, v2.z, w1 * v1.z)));
  r.w = fmaf(w4, v4.w, fmaf(w3, v3.w, fmaf(w2, v2.w, w1 * v1.w)));
  return r;
}
__device__ __forceinline__ float4 max4(const float4 a, const float4 b) {
  return make_float4(fmaxf(a.x, b.x), fmaxf(a.y, b.y), fmaxf(a.z, b.z), fmaxf(a.w, b.w));
}

// Work item = (pooled column jp, channel quad).  Everything that depends only on the sample
// position -- the four gather offsets and the four bilinear weights (weights formed first,
// roi_warping_layer.cu:56) -- is computed once per CTA into a shared-memory table (2*SUB sample
// rows x 14*SUB sample columns, 32 B per sample) and read back with two broadcast 128-bit loads.
// The feature map is read as fp32 NHWC (the engine keeps an fp32 copy of conv5_3 = hi + lo, 39 MB
// per batch of 8, so the gathers need no bf16 unpacking): one 16-byte load per tap and quad.
struct __align__(16) SampleTab {
  int off[4];    // element offsets of the 4 taps within the image (channel 0)
  float w[4];    // bilinear weights; all four are 0 for an out-of-range sample
};

// output planes of the fused RoI kernels: split-bf16 (hi, lo) or tri-plane (h, l, c; scale 2^exp)
struct RoiOut {
  void* p14[3];
  void* p7[3];
  float scale;
};
template <bool TRI>
__device__ __forceinline__ void st_feat4(void* const (&pl)[3], long long off, const float4 v, float scale) {
  if (TRI)
    st_tri4(static_cast<__half*>(pl[0]), static_cast<uint8_t*>(pl[1]), static_cast<uint8_t*>(pl[2]), off, v, scale);
  else
    st_split4(static_cast<__nv_bfloat16*>(pl[0]), static_cast<__nv_bfloat16*>(pl[1]), off, v);
}

template <int SUB, bool TRI>
__global__ void __launch_bounds__(256, 4)
roi_warp_split_kernel(const float* __restrict__ feat, int C, int H, int W,
                      const float* __restrict__ rois, float spatial_scale, const RoiOut o,
                      const int* __restrict__ img_hw, int level) {
  constexpr int P = 14 * SUB;
  constexpr int NS = 2 * SUB * P;  // samples handled by this CTA
  __shared__ SampleTab tab[NS];
  const int r = blockIdx.x;
  const int t = blockIdx.y;  // rows 2t, 2t+1 of the 14x14 grid
  const RoiGeom g = roi_geom(rois + static_cast<long long>(r) * 5, spatial_scale, P, P);
  // mixed-size batch: samples are bounded and clamped by the extent of the RoI's image (the row
  // stride stays the blob's W); the extent is clamped to [1, map] so that no sample can land
  // outside the map even for an invalid (zero) size
  int He = H, We = W;
  if (img_hw != nullptr) {
    const int m = (1 << level) - 1;
    He = max(1, min(H, (__ldg(img_hw + 2 * g.level) + m) >> level));
    We = max(1, min(W, (__ldg(img_hw + 2 * g.level + 1) + m) >> level));
  }
  for (int i = threadIdx.x; i < NS; i += blockDim.x) {
    const int sr = i / P, pw = i - sr * P;
    const int ph = 2 * t * SUB + sr;
    const AxisTap th = axis_tap(__fadd_rn(g.start_h, __fmul_rn(static_cast<float>(ph), g.bin_h)), He);
    const AxisTap tw = axis_tap(__fadd_rn(g.start_w, __fmul_rn(static_cast<float>(pw), g.bin_w)), We);
    const bool ok = th.ok && tw.ok;
    SampleTab e;
    e.off[0] = ok ? (th.lo * W + tw.lo) * C : 0;
    e.off[1] = ok ? (th.lo * W + tw.hi) * C : 0;
    e.off[2] = ok ? (th.hi * W + tw.lo) * C : 0;
    e.off[3] = ok ? (th.hi * W + tw.hi) * C : 0;
    e.w[0] = ok ? __fmul_rn(th.h, tw.h) : 0.f;
    e.w[1] = ok ? __fmul_rn(th.h, tw.l) : 0.f;
    e.w[2] = ok ? __fmul_rn(th.l, tw.h) : 0.f;
    e.w[3] = ok ? __fmul_rn(th.l, tw.l) : 0.f;
    tab[i] = e;
  }
  __syncthreads();
  const float* fimg = feat + static_cast<long long>(g.level) * H * W * C;
  const int c4n = C / 4;
  const float kNeg = -3.402823466e+38f;
  for (int item = threadIdx.x; item < 7 * c4n; item += blockDim.x) {
    const int jp = item / c4n;
    const int c = (item - jp * c4n) * 4;
    const float* fc = fimg + c;
    float4 best7 = make_float4(kNeg, kNeg, kNeg, kNeg);
#pragma unroll
    for (int dy = 0; dy < 2; ++dy) {
#pragma unroll
      for (int dx = 0; dx < 2; ++dx) {
        const int j = 2 * jp + dx;
        float4 cell = make_float4(kNeg, kNeg, kNeg, kNeg);
#pragma unroll
        for (int sy = 0; sy < SUB; ++sy) {
#pragma unroll
          for (int sx = 0; sx < SUB; ++sx) {
            const SampleTab& e = tab[(dy * SUB + sy) * P + j * SUB + sx];
            const int4 of = *reinterpret_cast<const int4*>(e.off);
            const float4 wg = *reinterpret_cast<const float4*>(e.w);
            const float4 v1 = __ldg(reinterpret_cast<const float4*>(fc + of.x));
            const float4 v2 = __ldg(reinterpret_cast<const float4*>(fc + of.y));
            const float4 v3 = __ldg(reinterpret_cast<const float4*>(fc + of.z));
            const float4 v4 = __ldg(reinterpret_cast<const float4*>(fc + of.w));
            cell = max4(cell, bilerp4(wg.x, wg.y, wg.z, wg.w, v1, v2, v3, v4));
          }
        }
        st_feat4<TRI>(o.p14, ((static_cast<long long>(r) * 14 + (2 * t + dy)) * 14 + j) * C + c, cell, o.scale);
        best7 = max4(best7, cell);
      }
    }
    st_feat4<TRI>(o.p7, ((static_cast<long long>(r) * 7 + t) * 7 + jp) * C + c, best7, o.scale);
  }
}


// ROW-WALK form of the fused kernel (alternative, mnc_roi_warp_set_rows(1)): thread = (pooled column j, channel quad); it walks the
// 14*SUB sample rows top to bottom keeping, for each of its SUB sample columns, the two live feature
// rows at that column's two taps in registers, and re-reads only when the row taps move on
// (bin_h < 1.4 feature rows per sample row): ~4*SUB loads per NEW FEATURE ROW instead of 4*SUB*SUB
// per pooled cell -- 2.5x fewer 16-byte loads through L1 for a typical proposal (the gather form
// is L1-bandwidth bound: l1tex 94 %, r02 ncu).  Same 4-tap formula as the gather form (weights
// first, FMA chain).  The 2x2 pooling to 7x7 pairs neighbouring columns by one warp shuffle.
// grid (R, C/64), 224 threads = 7 warps x (2 columns x 16 channel quads).
template <int SUB, bool TRI, int NQ>
__global__ void __launch_bounds__(224)
roi_warp_rows_kernel(const float* __restrict__ feat, int C, int H, int W,
                     const float* __restrict__ rois, float spatial_scale, const RoiOut o) {
  constexpr int P = 14 * SUB;
  __shared__ int4 rowq[P];   // {lo (or -1: out of range), hi, bits(h), bits(l)}
  const int r = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const RoiGeom g = roi_geom(rois + static_cast<long long>(r) * 5, spatial_scale, P, P);
  if (tid < P) {
    const AxisTap t = axis_tap(__fadd_rn(g.start_h, __fmul_rn(static_cast<float>(tid), g.bin_h)), H);
    rowq[tid] = make_int4(t.ok ? t.lo : -1, t.hi, __float_as_int(t.h), __float_as_int(t.l));
  }
  const int j = 2 * warp + (lane >> 4);              // pooled column 0..13
  // NQ channel quads per thread, 64 channels apart (independent load chains: ILP)
  const int c_raw = blockIdx.y * (64 * NQ) + (lane & 15) * 4;
  bool chan_ok[NQ];
  int c[NQ];
#pragma unroll
  for (int q = 0; q < NQ; ++q) {
    chan_ok[q] = c_raw + 64 * q < C;                 // (no early exit: the warp shuffles below)
    c[q] = chan_ok[q] ? c_raw + 64 * q : 0;
  }
  AxisTap tw[SUB];
#pragma unroll
  for (int sx = 0; sx < SUB; ++sx)
    tw[sx] = axis_tap(__fadd_rn(g.start_w, __fmul_rn(static_cast<float>(j * SUB + sx), g.bin_w)), W);
  __syncthreads();
  const float* fimg = feat + static_cast<long long>(g.level) * H * W * C;
  const float kNeg = -3.402823466e+38f;
  int cur_lo = -1, cur_hi = -1;
  float4 a_lo[NQ][SUB], a_hi[NQ][SUB], b_lo[NQ][SUB], b_hi[NQ][SUB];
  float4 acc14[NQ], acc7[NQ];
#pragma unroll
  for (int q = 0; q < NQ; ++q) {
#pragma unroll
    for (int sx = 0; sx < SUB; ++sx)
      a_lo[q][sx] = a_hi[q][sx] = b_lo[q][sx] = b_hi[q][sx] = make_float4(0.f, 0.f, 0.f, 0.f);
    acc14[q] = acc7[q] = make_float4(kNeg, kNeg, kNeg, kNeg);
  }
#pragma unroll 2
  for (int ph = 0; ph < P; ++ph) {
    const int4 tq = rowq[ph];
    float4 rowmax[NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) rowmax[q] = make_float4(0.f, 0.f, 0.f, 0.f);   // out of range: 0 (and it pools)
    if (tq.x >= 0) {
      if (tq.x != cur_lo) {
        if (tq.x == cur_hi) {
#pragma unroll
          for (int q = 0; q < NQ; ++q)
#pragma unroll
            for (int sx = 0; sx < SUB; ++sx) { a_lo[q][sx] = b_lo[q][sx]; a_hi[q][sx] = b_hi[q][sx]; }
        } else {
          const float* row = fimg + static_cast<long long>(tq.x) * W * C;
#pragma unroll
          for (int q = 0; q < NQ; ++q)
#pragma unroll
            for (int sx = 0; sx < SUB; ++sx) {
              a_lo[q][sx] = __ldg(reinterpret_cast<const float4*>(row + tw[sx].lo * C + c[q]));
              a_hi[q][sx] = __ldg(reinterpret_cast<const float4*>(row + tw[sx].hi * C + c[q]));
            }
        }
        cur_lo = tq.x;
        cur_hi = -1;
      }
      if (tq.y != cur_hi) {
        if (tq.y == tq.x) {
#pragma unroll
          for (int q = 0; q < NQ; ++q)
#pragma unroll
            for (int sx = 0; sx < SUB; ++sx) { b_lo[q][sx] = a_lo[q][sx]; b_hi[q][sx] = a_hi[q][sx]; }
        } else {
          const float* row = fimg + static_cast<long long>(tq.y) * W * C;
#pragma unroll
          for (int q = 0; q < NQ; ++q)
#pragma unroll
            for (int sx = 0; sx < SUB; ++sx) {
              b_lo[q][sx] = __ldg(reinterpret_cast<const float4*>(row + tw[sx].lo * C + c[q]));
              b_hi[q][sx] = __ldg(reinterpret_cast<const float4*>(row + tw[sx].hi * C + c[q]));
            }
        }
        cur_hi = tq.y;
      }
      const float th_h = __int_as_float(tq.z), th_l = __int_as_float(tq.w);
#pragma unroll
      for (int q = 0; q < NQ; ++q) rowmax[q] = make_float4(kNeg, kNeg, kNeg, kNeg);
#pragma unroll
      for (int sx = 0; sx < SUB; ++sx) {
        const float w1 = __fmul_rn(th_h, tw[sx].h), w2 = __fmul_rn(th_h, tw[sx].l);
        const float w3 = __fmul_rn(th_l, tw[sx].h), w4 = __fmul_rn(th_l, tw[sx].l);
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (tw[sx].ok) v = bilerp4(w1, w2, w3, w4, a_lo[q][sx], a_hi[q][sx], b_lo[q][sx], b_hi[q][sx]);
          rowmax[q] = max4(rowmax[q], v);
        }
      }
    }
#pragma unroll
    for (int q = 0; q < NQ; ++q) acc14[q] = max4(acc14[q], rowmax[q]);
    if (ph % SUB == SUB - 1) {
      const int i = ph / SUB;                        // row of the 14x14 grid
#pragma unroll
      for (int q = 0; q < NQ; ++q) {
        if (chan_ok[q])
          st_feat4<TRI>(o.p14, ((static_cast<long long>(r) * 14 + i) * 14 + j) * C + c[q], acc14[q], o.scale);
        acc7[q] = max4(acc7[q], acc14[q]);
        acc14[q] = make_float4(kNeg, kNeg, kNeg, kNeg);
      }
      if (i & 1) {
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
          float4 oth;
          oth.x = __shfl_xor_sync(0xffffffffu, acc7[q].x, 16);
          oth.y = __shfl_xor_sync(0xffffffffu, acc7[q].y, 16);
          oth.z = __shfl_xor_sync(0xffffffffu, acc7[q].z, 16);
          oth.w = __shfl_xor_sync(0xffffffffu, acc7[q].w, 16);
          if ((lane >> 4) == 0 && chan_ok[q])
            st_feat4<TRI>(o.p7, ((static_cast<long long>(r) * 7 + (i >> 1)) * 7 + (j >> 1)) * C + c[q],
                          max4(acc7[q], oth), o.scale);
          acc7[q] = make_float4(kNeg, kNeg, kNeg, kNeg);
        }
      }
    }
  }
}

template <bool TRI>
static void launch_roi_rows(int nq, int sub, const float* feat, int C, int H, int W, const float* rois,
                            int R, float spatial_scale, const RoiOut& o, cudaStream_t s) {
  dim3 grid(R, (C + 64 * nq - 1) / (64 * nq));
#define MNC_ROWS(SUB_, NQ_) roi_warp_rows_kernel<SUB_, TRI, NQ_><<<grid, 224, 0, s>>>(feat, C, H, W, rois, spatial_scale, o)
  if (sub == 2) {
    if (nq == 2) MNC_ROWS(2, 2); else MNC_ROWS(2, 1);
  } else {
    if (nq == 2) MNC_ROWS(1, 2); else MNC_ROWS(1, 1);
  }
#undef MNC_ROWS
}

// Same outputs, fewer loads.  The sample grid of a RoI is regular, so bilinear sampling separates:
// for a sample row s (row taps y_lo, y_hi fixed) the column function
//     C_s(x) = hy * F[y_lo][x] + ly * F[y_hi][x]
// is all that sample row ever needs, and sample (s, pw) = hx * C_s(x_lo) + lx * C_s(x_hi).
// A thread owns one channel quad and one pooled-7 row (2*SUB sample rows) and WALKS the sample
// columns left to right, keeping C_s(x_lo), C_s(x_hi) of every sample row in registers; when the
// taps move one feature column to the right the pair shifts and one new column is fetched (two
// 16-byte loads per sample row).  A RoI that is Wr feature columns wide costs ~2*(Wr+1) loads per
// sample row instead of 4 per sample (4 * 14 * SUB): 3-4x fewer L1 transactions for typical
// proposals, and never more.  Control flow depends only on the RoI, so warps never diverge.
// (Rounding differs from the weights-first form by an ulp; the fused path is tolerance-checked,
// the bit-exact layer kernel is roi_warp_nchw_kernel.)
__device__ __forceinline__ float4 col_lerp(const float* __restrict__ plo, const float* __restrict__ phi,
                                           int xoff, float hy, float ly) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(plo + xoff));
  const float4 b = __ldg(reinterpret_cast<const float4*>(phi + xoff));
  return make_float4(fmaf(ly, b.x, hy * a.x), fmaf(ly, b.y, hy * a.y), fmaf(ly, b.z, hy * a.z),
                     fmaf(ly, b.w, hy * a.w));
}

template <int SUB>
__global__ void __launch_bounds__(256)
roi_warp_walk_kernel(const float* __restrict__ feat, int C, int H, int W,
                     const float* __restrict__ rois, float spatial_scale,
                     __nv_bfloat16* __restrict__ o14_hi, __nv_bfloat16* __restrict__ o14_lo,
                     __nv_bfloat16* __restrict__ o7_hi, __nv_bfloat16* __restrict__ o7_lo) {
  constexpr int P = 14 * SUB;
  constexpr int NR = 2 * SUB;  // sample rows feeding one row of the 7x7 grid
  __shared__ AxisTap colt[P];
  __shared__ AxisTap rowt[2 * NR];
  const int r = blockIdx.x;
  const RoiGeom g = roi_geom(rois + static_cast<long long>(r) * 5, spatial_scale, P, P);
  if (threadIdx.x < P) {
    colt[threadIdx.x] =
        axis_tap(__fadd_rn(g.start_w, __fmul_rn(static_cast<float>(threadIdx.x), g.bin_w)), W);
  } else if (threadIdx.x < P + 2 * NR) {
    const int i = threadIdx.x - P;
    const int ph = blockIdx.y * 2 * NR + i;   // rows of pooled-7 rows 2*blockIdx.y, 2*blockIdx.y+1
    rowt[i] = axis_tap(__fadd_rn(g.start_h, __fmul_rn(static_cast<float>(ph), g.bin_h)), H);
  }
  __syncthreads();
  const int half = threadIdx.x >> 7;
  const int t = 2 * blockIdx.y + half;
  if (t >= 7) return;
  const float* fimg = feat + static_cast<long long>(g.level) * H * W * C;
  const float kNeg = -3.402823466e+38f;
  for (int c = (threadIdx.x & 127) * 4; c < C; c += 512) {
    const float* plo[NR];
    const float* phi[NR];
    float hy[NR], ly[NR];
    bool rok[NR];
#pragma unroll
    for (int s = 0; s < NR; ++s) {
      const AxisTap th = rowt[half * NR + s];
      plo[s] = fimg + static_cast<long long>(th.lo) * W * C + c;
      phi[s] = fimg + static_cast<long long>(th.hi) * W * C + c;
      hy[s] = th.h;
      ly[s] = th.l;
      rok[s] = th.ok != 0;
    }
    float4 Clo[NR], Chi[NR];
#pragma unroll
    for (int s = 0; s < NR; ++s) Clo[s] = Chi[s] = make_float4(0.f, 0.f, 0.f, 0.f);
    int cx_lo = -1, cx_hi = -1;
    float4 best7 = make_float4(kNeg, kNeg, kNeg, kNeg);
    for (int j = 0; j < 14; ++j) {
      float4 cell[2];
      cell[0] = cell[1] = make_float4(kNeg, kNeg, kNeg, kNeg);
#pragma unroll
      for (int sx = 0; sx < SUB; ++sx) {
        const AxisTap tw = colt[j * SUB + sx];
        if (tw.ok && (tw.lo != cx_lo || tw.hi != cx_hi)) {
          const bool shift = tw.lo == cx_hi;
          const bool keep_lo = tw.lo == cx_lo;
#pragma unroll
          for (int s = 0; s < NR; ++s) {
            if (!rok[s]) continue;
            if (shift) Clo[s] = Chi[s];
            else if (!keep_lo) Clo[s] = col_lerp(plo[s], phi[s], tw.lo * C, hy[s], ly[s]);
            if (tw.hi == tw.lo) Chi[s] = Clo[s];
            else Chi[s] = col_lerp(plo[s], phi[s], tw.hi * C, hy[s], ly[s]);
          }
          cx_lo = tw.lo;
          cx_hi = tw.hi;
        }
#pragma unroll
        for (int s = 0; s < NR; ++s) {
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);   // out-of-range sample: 0 (and it pools)
          if (tw.ok && rok[s])
            v = make_float4(fmaf(tw.l, Chi[s].x, tw.h * Clo[s].x), fmaf(tw.l, Chi[s].y, tw.h * Clo[s].y),
                            fmaf(tw.l, Chi[s].z, tw.h * Clo[s].z), fmaf(tw.l, Chi[s].w, tw.h * Clo[s].w));
          cell[s / SUB] = max4(cell[s / SUB], v);
        }
      }
      st_split4(o14_hi, o14_lo, ((static_cast<long long>(r) * 14 + 2 * t) * 14 + j) * C + c, cell[0]);
      st_split4(o14_hi, o14_lo, ((static_cast<long long>(r) * 14 + 2 * t + 1) * 14 + j) * C + c, cell[1]);
      best7 = max4(best7, max4(cell[0], cell[1]));
      if (j & 1) {
        st_split4(o7_hi, o7_lo, ((static_cast<long long>(r) * 7 + t) * 7 + (j >> 1)) * C + c, best7);
        best7 = make_float4(kNeg, kNeg, kNeg, kNeg);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Sibling test graphs (SURVEY.md section 8f row 4).
//   ROIPooling  caffe-mnc/src/caffe/layers/roi_pooling_layer.cu:17-77 (Fast R-CNN max over integer
//               bins; CFM test net, models/VGG16/cfm/test.prototxt:399-465)
//   ROIWarping at 7x7 straight into fc6 (Faster R-CNN test net,
//               models/VGG16/faster_rcnn_end2end/test.prototxt:479-490)
struct PoolBin {
  int h0, h1, w0, w1;
};

// roi_pooling_layer.cu:29-57 for pooled cell (ph, pw)
__device__ __forceinline__ PoolBin roi_pool_bin(const float* roi, float spatial_scale, int H, int W,
                                                int PH, int PW, int ph, int pw) {
  const int sw = static_cast<int>(roundf(__fmul_rn(roi[1], spatial_scale)));
  const int sh = static_cast<int>(roundf(__fmul_rn(roi[2], spatial_scale)));
  const int ew = static_cast<int>(roundf(__fmul_rn(roi[3], spatial_scale)));
  const int eh = static_cast<int>(roundf(__fmul_rn(roi[4], spatial_scale)));
  const int rw = max(ew - sw + 1, 1), rh = max(eh - sh + 1, 1);
  const float bh = __fdiv_rn(static_cast<float>(rh), static_cast<float>(PH));
  const float bw = __fdiv_rn(static_cast<float>(rw), static_cast<float>(PW));
  PoolBin b;
  b.h0 = static_cast<int>(floorf(__fmul_rn(static_cast<float>(ph), bh)));
  b.w0 = static_cast<int>(floorf(__fmul_rn(static_cast<float>(pw), bw)));
  b.h1 = static_cast<int>(ceilf(__fmul_rn(static_cast<float>(ph + 1), bh)));
  b.w1 = static_cast<int>(ceilf(__fmul_rn(static_cast<float>(pw + 1), bw)));
  b.h0 = min(max(b.h0 + sh, 0), H);
  b.h1 = min(max(b.h1 + sh, 0), H);
  b.w0 = min(max(b.w0 + sw, 0), W);
  b.w1 = min(max(b.w1 + sw, 0), W);
  return b;
}

// Layer contract: fp32 NCHW in and out (+ optional argmax, which the reference always writes).
// grid (R, ceil(C/16)); the RoI's PH*PW bins are computed once per CTA into shared memory.
__global__ void __launch_bounds__(256)
roi_pool_nchw_kernel(const float* __restrict__ feat, int C, int H, int W,
                     const float* __restrict__ rois, float spatial_scale, int PH, int PW,
                     float* __restrict__ out, int* __restrict__ argmax) {
  extern __shared__ PoolBin bins[];
  const int r = blockIdx.x;
  const int c0 = blockIdx.y * kWarpSlab;
  const float* roi = rois + static_cast<long long>(r) * 5;
  const int PP = PH * PW;
  for (int i = threadIdx.x; i < PP; i += blockDim.x)
    bins[i] = roi_pool_bin(roi, spatial_scale, H, W, PH, PW, i / PW, i % PW);
  __syncthreads();
  const int level = static_cast<int>(roi[0]);
  const int nc = min(kWarpSlab, C - c0);
  for (int i = threadIdx.x; i < nc * PP; i += blockDim.x) {
    const int c = c0 + i / PP, cell = i % PP;
    const PoolBin b = bins[cell];
    const float* plane = feat + (static_cast<long long>(level) * C + c) * H * W;
    const bool empty = (b.h1 <= b.h0) || (b.w1 <= b.w0);
    float best = empty ? 0.f : -3.402823466e+38f;
    int arg = -1;
    for (int h = b.h0; h < b.h1; ++h)
      for (int w = b.w0; w < b.w1; ++w) {
        const float v = __ldg(plane + h * W + w);
        if (v > best) {
          best = v;
          arg = h * W + w;
        }
      }
    const long long o = (static_cast<long long>(r) * C + c) * PP + cell;
    out[o] = best;
    if (argmax) argmax[o] = arg;
  }
}

// Engine form: fp32 NHWC feature copy in, split-bf16 rows [r][ph][pw][c] out (the K order the FC
// weights are permuted to).  grid (R, P); each thread owns (pw, channel quad) items of row ph.
__global__ void __launch_bounds__(256)
roi_pool_split_kernel(const float* __restrict__ feat, int C, int H, int W,
                      const float* __restrict__ rois, float spatial_scale, int P,
                      __nv_bfloat16* __restrict__ o_hi, __nv_bfloat16* __restrict__ o_lo) {
  __shared__ PoolBin bins[kMaxPooled];
  const int r = blockIdx.x, ph = blockIdx.y;
  const float* roi = rois + static_cast<long long>(r) * 5;
  if (threadIdx.x < P) bins[threadIdx.x] = roi_pool_bin(roi, spatial_scale, H, W, P, P, ph, threadIdx.x);
  __syncthreads();
  const float* fimg = feat + static_cast<long long>(static_cast<int>(roi[0])) * H * W * C;
  const int c4n = C / 4;
  for (int item = threadIdx.x; item < P * c4n; item += blockDim.x) {
    const int pw = item / c4n, c = (item - pw * c4n) * 4;
    const PoolBin b = bins[pw];
    const bool empty = (b.h1 <= b.h0) || (b.w1 <= b.w0);
    const float init = empty ? 0.f : -3.402823466e+38f;
    float4 best = make_float4(init, init, init, init);
    for (int h = b.h0; h < b.h1; ++h)
      for (int w = b.w0; w < b.w1; ++w)
        best = max4(best, __ldg(reinterpret_cast<const float4*>(fimg + (static_cast<long long>(h) * W + w) * C + c)));
    st_split4(o_hi, o_lo, ((static_cast<long long>(r) * P + ph) * P + pw) * C + c, best);
  }
}

// ROIWarping at P x P straight to split-bf16 rows [r][ph][pw][c] (no pooling after it).
__global__ void __launch_bounds__(256)
roi_sample_split_kernel(const float* __restrict__ feat, int C, int H, int W,
                        const float* __restrict__ rois, float spatial_scale, int P,
                        __nv_bfloat16* __restrict__ o_hi, __nv_bfloat16* __restrict__ o_lo) {
  __shared__ SampleTab tab[kMaxPooled];
  const int r = blockIdx.x, ph = blockIdx.y;
  const RoiGeom g = roi_geom(rois + static_cast<long long>(r) * 5, spatial_scale, P, P);
  if (threadIdx.x < P) {
    const int pw = threadIdx.x;
    const AxisTap th = axis_tap(__fadd_rn(g.start_h, __fmul_rn(static_cast<float>(ph), g.bin_h)), H);
    const AxisTap tw = axis_tap(__fadd_rn(g.start_w, __fmul_rn(static_cast<float>(pw), g.bin_w)), W);
    const bool ok = th.ok && tw.ok;
    SampleTab e;
    e.off[0] = ok ? (th.lo * W + tw.lo) * C : 0;
    e.off[1] = ok ? (th.lo * W + tw.hi) * C : 0;
    e.off[2] = ok ? (th.hi * W + tw.lo) * C : 0;
    e.off[3] = ok ? (th.hi * W + tw.hi) * C : 0;
    e.w[0] = ok ? __fmul_rn(th.h, tw.h) : 0.f;
    e.w[1] = ok ? __fmul_rn(th.h, tw.l) : 0.f;
    e.w[2] = ok ? __fmul_rn(th.l, tw.h) : 0.f;
    e.w[3] = ok ? __fmul_rn(th.l, tw.l) : 0.f;
    tab[pw] = e;
  }
  __syncthreads();
  const float* fimg = feat + static_cast<long long>(g.level) * H * W * C;
  const int c4n = C / 4;
  for (int item = threadIdx.x; item < P * c4n; item += blockDim.x) {
    const int pw = item / c4n, c = (item - pw * c4n) * 4;
    const SampleTab& e = tab[pw];
    const int4 of = *reinterpret_cast<const int4*>(e.off);
    const float4 wg = *reinterpret_cast<const float4*>(e.w);
    const float* fc = fimg + c;
    const float4 v = bilerp4(wg.x, wg.y, wg.z, wg.w, __ldg(reinterpret_cast<const float4*>(fc + of.x)),
                             __ldg(reinterpret_cast<const float4*>(fc + of.y)),
                             __ldg(reinterpret_cast<const float4*>(fc + of.z)),
                             __ldg(reinterpret_cast<const float4*>(fc + of.w)));
    st_split4(o_hi, o_lo, ((static_cast<long long>(r) * P + ph) * P + pw) * C + c, v);
  }
}


// sigmoid (sigmoid_layer.cu:10-14) -> mask_proposal (R,1,M,M) -> MaskResize to (R,1,14,14).
// One CTA per RoI; logits row stride given.
__global__ void __launch_bounds__(256)
sigmoid_resize_kernel(const float* __restrict__ logits, int stride, int M, int O,
                      float* __restrict__ mask_proposal, float* __restrict__ mask_resized) {
  extern __shared__ float sm[];  // M*M
  const int r = blockIdx.x;
  const float* x = logits + static_cast<long long>(r) * stride;
  for (int i = threadIdx.x; i < M * M; i += blockDim.x) {
    const float s = __fdiv_rn(1.f, __fadd_rn(1.f, expf(-x[i])));
    sm[i] = s;
    mask_proposal[static_cast<long long>(r) * M * M + i] = s;
  }
  __syncthreads();
  const float ratio = __fdiv_rn(static_cast<float>(M), static_cast<float>(O));
  for (int i = threadIdx.x; i < O * O; i += blockDim.x) {
    const int h = i / O, w = i % O;
    const AxisTap th = axis_tap(__fmul_rn(static_cast<float>(h), ratio), M);
    const AxisTap tw = axis_tap(__fmul_rn(static_cast<float>(w), ratio), M);
    float val = 0.f;
    if (th.ok && tw.ok)
      val = bilerp(th, tw, sm[th.lo * M + tw.lo], sm[th.lo * M + tw.hi], sm[th.hi * M + tw.lo],
                   sm[th.hi * M + tw.hi]);
    mask_resized[static_cast<long long>(r) * O * O + i] = val;
  }
}

// MaskPooling + 2x2 max pool on split NHWC: out7[r][t][j][c] = max_{dy,dx} feat14*mask14.
__global__ void __launch_bounds__(256)
mask_pool_split_kernel(const __nv_bfloat16* __restrict__ f_hi, const __nv_bfloat16* __restrict__ f_lo,
                       const float* __restrict__ mask14, int C, __nv_bfloat16* __restrict__ o_hi,
                       __nv_bfloat16* __restrict__ o_lo) {
  const int r = blockIdx.x, t = blockIdx.y;
  __shared__ float m[2][14];
  if (threadIdx.x < 28)
    m[threadIdx.x / 14][threadIdx.x % 14] =
        mask14[static_cast<long long>(r) * 196 + (2 * t + threadIdx.x / 14) * 14 + threadIdx.x % 14];
  __syncthreads();
  for (int c = threadIdx.x * 2; c < C; c += blockDim.x * 2) {
    for (int jp = 0; jp < 7; ++jp) {
      float2 best = make_float2(-3.402823466e+38f, -3.402823466e+38f);
#pragma unroll
      for (int dy = 0; dy < 2; ++dy)
#pragma unroll
        for (int dx = 0; dx < 2; ++dx) {
          const int i = 2 * t + dy, j = 2 * jp + dx;
          const float2 f = ld_split2(f_hi, f_lo, ((static_cast<long long>(r) * 14 + i) * 14 + j) * C + c);
          const float mk = m[dy][j];
          best.x = fmaxf(best.x, __fmul_rn(f.x, mk));
          best.y = fmaxf(best.y, __fmul_rn(f.y, mk));
        }
      st_split2(o_hi, o_lo, ((static_cast<long long>(r) * 7 + t) * 7 + jp) * C + c, best.x, best.y);
    }
  }
}

static inline int check_launch() { return cudaGetLastError() == cudaSuccess ? MNC_OK : MNC_ERR_CUDA; }
static inline int grid_for(long long n, int block, int cap) {
  long long g = (n + block - 1) / block;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return static_cast<int>(g);
}

}  // namespace mnc

using namespace mnc;

static int g_roi_stage = 2;   // 2: row walk (default, fastest measured); 1: staged window; 0: gather
extern "C" int mnc_roi_warp_set_stage(int on) {
  const int prev = g_roi_stage;
  g_roi_stage = on;   // 0: gather kernel, 1: shared-memory staged window (28x28), 2: row walk
  return prev;
}

static int g_roi_walk_threads = 128, g_roi_walk_cpc = 32, g_roi_walk_ch14 = 4;
// A/B knob: planes per lane of the 14x14 row walk (4 or 8)
extern "C" int mnc_roi_warp_set_walk_planes14(int planes) {
  if (planes != 4 && planes != 8) return MNC_ERR_ARG;
  g_roi_walk_ch14 = planes;
  return MNC_OK;
}
// A/B knob of the row-walk ROIWarping kernel: threads per CTA (multiple of 32, <= 256) and
// channels per CTA.
extern "C" int mnc_roi_warp_set_walk_shape(int threads, int channels_per_cta) {
  if (threads < 32 || threads > 256 || threads % 32 || channels_per_cta < 4) return MNC_ERR_ARG;
  g_roi_walk_threads = threads;
  g_roi_walk_cpc = channels_per_cta;
  return MNC_OK;
}

extern "C" int mnc_roi_warp_nchw(const float* feat, int C, int H, int W, const float* rois, int R,
                                 int pooled_h, int pooled_w, float spatial_scale, float* out,
                                 void* stream) {
  if (R <= 0) return MNC_OK;
  if (pooled_h > kMaxPooled || pooled_w > kMaxPooled || pooled_h <= 0 || pooled_w <= 0)
    return MNC_ERR_ARG;
  dim3 grid(R, (C + kWarpSlab - 1) / kWarpSlab);
  auto s = static_cast<cudaStream_t>(stream);
  // the two sizes of the MNC graph: shared-memory staged windows (needs 16-byte aligned planes and
  // a window that fits the budget: H * W <= 2457 floats covers every map up to 39 x 63)
  const bool stage = g_roi_stage && (reinterpret_cast<uintptr_t>(out) % 16 == 0) &&
                     static_cast<long long>(H) * W * 5 <= kStageFloats;
  if (g_roi_stage == 2 && pooled_h == pooled_w && (pooled_h == 28 || pooled_h == 14)) {
    // one pass of the CTA's warps covers threads/32 * (planes per warp) channels: 32 channels per
    // CTA = 4 warps (28x28: 8 planes per lane; 14x14: 2 plane groups x 4), so 128 threads keep
    // every warp of the CTA busy (with 256, half of them only waited at the barrier and held
    // their scheduler slots until the CTA retired)
    const int cpc = g_roi_walk_cpc, threads = g_roi_walk_threads;
    dim3 wgrid(R, (C + cpc - 1) / cpc);
    if (pooled_h == 28)
      roi_warp_rowwalk_kernel<28><<<wgrid, threads, 0, s>>>(feat, C, H, W, rois, spatial_scale, cpc, out);
    else if (g_roi_walk_ch14 == 8)
      roi_warp_rowwalk_kernel<14, 8><<<wgrid, threads, 0, s>>>(feat, C, H, W, rois, spatial_scale, cpc, out);
    else
      roi_warp_rowwalk_kernel<14><<<wgrid, threads, 0, s>>>(feat, C, H, W, rois, spatial_scale, cpc, out);
    return check_launch();
  }
  // (14x14: 784 taps per channel against a ~440-float window -- staging does not pay, measured)
  if (stage && g_roi_stage == 1 && pooled_h == 28 && pooled_w == 28) {
    dim3 sgrid(R, (C + kStageGroup - 1) / kStageGroup);
    static SmemGrant grant28;
    const int smem = kStageFloats * 4;
    if (!ensure_dynamic_smem(roi_warp28_stage_kernel, smem, grant28)) return MNC_ERR_CUDA;
    roi_warp28_stage_kernel<<<sgrid, 256, smem, s>>>(feat, C, H, W, rois, spatial_scale, out, 1.0f);
    return check_launch();
  }
  if (pooled_h == 28 && pooled_w == 28)
    roi_warp_nchw_kernel<28, 28, 4><<<grid, 256, 0, s>>>(feat, C, H, W, rois, spatial_scale, out);
  else if (pooled_h == 14 && pooled_w == 14)
    roi_warp_nchw_kernel<14, 14, 2><<<grid, 256, 0, s>>>(feat, C, H, W, rois, spatial_scale, out);
  else if (pooled_h == 7 && pooled_w == 7)
    roi_warp_nchw_kernel<7, 7, 1><<<grid, 256, 0, s>>>(feat, C, H, W, rois, spatial_scale, out);
  else
    roi_warp_nchw_generic_kernel<<<grid, 256, 0, s>>>(feat, C, H, W, rois, pooled_h, pooled_w,
                                                      spatial_scale, out);
  return check_launch();
}

extern "C" int mnc_mask_resize_nchw(const float* in, int N, int C, int in_h, int in_w, int out_h,
                                    int out_w, float* out, void* stream) {
  const long long total = static_cast<long long>(N) * C * out_h * out_w;
  if (total <= 0) return MNC_OK;
  mask_resize_nchw_kernel<<<grid_for(total, 256, 148 * 8), 256, 0,
                            static_cast<cudaStream_t>(stream)>>>(in, N * C, in_h, in_w, out_h,
                                                                 out_w, out);
  return check_launch();
}

extern "C" int mnc_mask_pool_nchw(const float* feat, const float* mask, int N, int C, int H, int W,
                                  float* out, void* stream) {
  const long long total = static_cast<long long>(N) * C * H * W;
  if (total <= 0) return MNC_OK;
  const int hw = H * W;
  const bool vec = (hw % 4 == 0) && ((reinterpret_cast<uintptr_t>(feat) & 15) == 0) &&
                   ((reinterpret_cast<uintptr_t>(mask) & 15) == 0) &&
                   ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
  if (vec)
    mask_pool_nchw_kernel<<<grid_for(total / 4, 256, 148 * 16), 256, 0,
                            static_cast<cudaStream_t>(stream)>>>(feat, mask, N, C, hw, out);
  else
    mask_pool_nchw_scalar_kernel<<<grid_for(total, 256, 148 * 16), 256, 0,
                                   static_cast<cudaStream_t>(stream)>>>(feat, mask, N, C, hw, out);
  return check_launch();
}

static int g_roi_rows = 0;   // fused engine form: 0 = per-cell gathers (default), 1 = row walk (bit-identical,
                             // 2.5x fewer loads, not faster: 0.625-0.641 vs 0.639 ms at 28x28, 0.38-0.41 vs 0.305 at 14x14:
                             // the kernel is bound by its 1.2 GB of output and the 4x sample arithmetic, not by taps)
extern "C" int mnc_roi_warp_set_rows(int on) {
  const int prev = g_roi_rows;
  g_roi_rows = (on == 1 || on == 2) ? on : 0;   // channel quads per thread
  return prev;
}
static int g_roi_walk = 0;  // measured slower on real proposals (profiles/README.md): latency-bound
extern "C" int mnc_roi_warp_set_walk(int on) {
  const int prev = g_roi_walk;
  g_roi_walk = on ? 1 : 0;
  return prev;
}

// img_hw (optional, device int32 [batch][2]) + level: per-image extents of a mixed-size batch;
// the A/B kernel forms (set_walk / set_rows) do not take them.
extern "C" int mnc_roi_warp_split2(const float* feat_nhwc, int C, int H, int W, const float* rois,
                                   int R, int sub, float spatial_scale, void* o14_hi, void* o14_lo,
                                   void* o7_hi, void* o7_lo, const int* img_hw, int level,
                                   void* stream) {
  if (R <= 0) return MNC_OK;
  if (C % 4 != 0 || (sub != 1 && sub != 2) || (reinterpret_cast<uintptr_t>(feat_nhwc) & 15))
    return MNC_ERR_ARG;
  if (img_hw != nullptr && (level < 0 || level > 16 || g_roi_walk || g_roi_rows)) return MNC_ERR_ARG;
  auto s = static_cast<cudaStream_t>(stream);
  if (g_roi_walk) {
    dim3 wgrid(R, 4);
    if (sub == 2)
      roi_warp_walk_kernel<2><<<wgrid, 256, 0, s>>>(
          feat_nhwc, C, H, W, rois, spatial_scale, static_cast<__nv_bfloat16*>(o14_hi),
          static_cast<__nv_bfloat16*>(o14_lo), static_cast<__nv_bfloat16*>(o7_hi),
          static_cast<__nv_bfloat16*>(o7_lo));
    else
      roi_warp_walk_kernel<1><<<wgrid, 256, 0, s>>>(
          feat_nhwc, C, H, W, rois, spatial_scale, static_cast<__nv_bfloat16*>(o14_hi),
          static_cast<__nv_bfloat16*>(o14_lo), static_cast<__nv_bfloat16*>(o7_hi),
          static_cast<__nv_bfloat16*>(o7_lo));
    return check_launch();
  }
  RoiOut o;
  o.p14[0] = o14_hi; o.p14[1] = o14_lo; o.p14[2] = nullptr;
  o.p7[0] = o7_hi; o.p7[1] = o7_lo; o.p7[2] = nullptr;
  o.scale = 1.0f;
  if (g_roi_rows && C % 4 == 0) {
    launch_roi_rows<false>(g_roi_rows, sub, feat_nhwc, C, H, W, rois, R, spatial_scale, o, s);
    return check_launch();
  }
  dim3 grid(R, 7);
  if (sub == 2)
    roi_warp_split_kernel<2, false><<<grid, 256, 0, s>>>(feat_nhwc, C, H, W, rois, spatial_scale, o,
        img_hw, level);
  else
    roi_warp_split_kernel<1, false><<<grid, 256, 0, s>>>(feat_nhwc, C, H, W, rois, spatial_scale, o,
        img_hw, level);
  return check_launch();
}

extern "C" int mnc_roi_warp_split(const float* feat_nhwc, int C, int H, int W, const float* rois,
                                  int R, int sub, float spatial_scale, void* o14_hi, void* o14_lo,
                                  void* o7_hi, void* o7_lo, void* stream) {
  return mnc_roi_warp_split2(feat_nhwc, C, H, W, rois, R, sub, spatial_scale, o14_hi, o14_lo, o7_hi,
                             o7_lo, nullptr, 0, stream);
}

// Same, writing tri-plane outputs (fp16 value, e4m3 residual, e4m3 copy) scaled by `scale` = 2^exp.
extern "C" int mnc_roi_warp_tri2(const float* feat_nhwc, int C, int H, int W, const float* rois,
                                 int R, int sub, float spatial_scale, float scale, void* o14_h,
                                 void* o14_l, void* o14_c, void* o7_h, void* o7_l, void* o7_c,
                                 const int* img_hw, int level, void* stream) {
  if (R <= 0) return MNC_OK;
  if (C % 4 != 0 || (sub != 1 && sub != 2) || (reinterpret_cast<uintptr_t>(feat_nhwc) & 15))
    return MNC_ERR_ARG;
  if (img_hw != nullptr && (level < 0 || level > 16 || g_roi_rows)) return MNC_ERR_ARG;
  auto s = static_cast<cudaStream_t>(stream);
  RoiOut o;
  o.p14[0] = o14_h; o.p14[1] = o14_l; o.p14[2] = o14_c;
  o.p7[0] = o7_h; o.p7[1] = o7_l; o.p7[2] = o7_c;
  o.scale = scale;
  if (g_roi_rows) {
    launch_roi_rows<true>(g_roi_rows, sub, feat_nhwc, C, H, W, rois, R, spatial_scale, o, s);
    return check_launch();
  }
  dim3 grid(R, 7);
  if (sub == 2)
    roi_warp_split_kernel<2, true><<<grid, 256, 0, s>>>(feat_nhwc, C, H, W, rois, spatial_scale, o,
        img_hw, level);
  else
    roi_warp_split_kernel<1, true><<<grid, 256, 0, s>>>(feat_nhwc, C, H, W, rois, spatial_scale, o,
        img_hw, level);
  return check_launch();
}

extern "C" int mnc_roi_warp_tri(const float* feat_nhwc, int C, int H, int W, const float* rois,
                                int R, int sub, float spatial_scale, float scale, void* o14_h,
                                void* o14_l, void* o14_c, void* o7_h, void* o7_l, void* o7_c,
                                void* stream) {
  return mnc_roi_warp_tri2(feat_nhwc, C, H, W, rois, R, sub, spatial_scale, scale, o14_h, o14_l,
                           o14_c, o7_h, o7_l, o7_c, nullptr, 0, stream);
}

extern "C" int mnc_roi_pool_nchw(const float* feat, int C, int H, int W, const float* rois, int R,
                                 int pooled_h, int pooled_w, float spatial_scale, float* out,
                                 int* argmax, void* stream) {
  if (R <= 0) return MNC_OK;
  if (C <= 0 || pooled_h <= 0 || pooled_w <= 0) return MNC_ERR_ARG;
  const int smem = pooled_h * pooled_w * static_cast<int>(sizeof(PoolBin));
  if (smem > 48 * 1024) return MNC_ERR_ARG;
  dim3 grid(R, (C + kWarpSlab - 1) / kWarpSlab);
  roi_pool_nchw_kernel<<<grid, 256, smem, static_cast<cudaStream_t>(stream)>>>(
      feat, C, H, W, rois, spatial_scale, pooled_h, pooled_w, out, argmax);
  return check_launch();
}

extern "C" int mnc_roi_pool_split(const float* feat_nhwc, int C, int H, int W, const float* rois,
                                  int R, int pooled, float spatial_scale, void* o_hi, void* o_lo,
                                  void* stream) {
  if (R <= 0) return MNC_OK;
  if (C % 4 != 0 || pooled <= 0 || pooled > kMaxPooled ||
      (reinterpret_cast<uintptr_t>(feat_nhwc) & 15))
    return MNC_ERR_ARG;
  roi_pool_split_kernel<<<dim3(R, pooled), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      feat_nhwc, C, H, W, rois, spatial_scale, pooled, static_cast<__nv_bfloat16*>(o_hi),
      static_cast<__nv_bfloat16*>(o_lo));
  return check_launch();
}

extern "C" int mnc_roi_sample_split(const float* feat_nhwc, int C, int H, int W, const float* rois,
                                    int R, int pooled, float spatial_scale, void* o_hi, void* o_lo,
                                    void* stream) {
  if (R <= 0) return MNC_OK;
  if (C % 4 != 0 || pooled <= 0 || pooled > kMaxPooled ||
      (reinterpret_cast<uintptr_t>(feat_nhwc) & 15))
    return MNC_ERR_ARG;
  roi_sample_split_kernel<<<dim3(R, pooled), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      feat_nhwc, C, H, W, rois, spatial_scale, pooled, static_cast<__nv_bfloat16*>(o_hi),
      static_cast<__nv_bfloat16*>(o_lo));
  return check_launch();
}

extern "C" int mnc_sigmoid_mask_resize(const float* logits, int stride, int R, int mask_size,
                                       int out_size, float* mask_proposal, float* mask_resized,
                                       void* stream) {
  if (R <= 0) return MNC_OK;
  sigmoid_resize_kernel<<<R, 256, mask_size * mask_size * sizeof(float),
                          static_cast<cudaStream_t>(stream)>>>(logits, stride, mask_size, out_size,
                                                               mask_proposal, mask_resized);
  return check_launch();
}

extern "C" int mnc_mask_pool_split(const void* f_hi, const void* f_lo, const float* mask14, int R,
                                   int C, void* o_hi, void* o_lo, void* stream) {
  if (R <= 0) return MNC_OK;
  if (C % 2 != 0) return MNC_ERR_ARG;
  dim3 grid(R, 7);
  mask_pool_split_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(f_hi), static_cast<const __nv_bfloat16*>(f_lo), mask14, C,
      static_cast<__nv_bfloat16*>(o_hi), static_cast<__nv_bfloat16*>(o_lo));
  return check_launch();
}
