// Device-side building blocks shared by every kernel of libtriplane_b200.
//
// Reference citations are relative to /root/reference/g_nerf/ (VR/ = training/volumetric_rendering/).
// Nothing here is translated from the reference (which is ~40 stock ATen launches per forward,
// SURVEY.md section 2a); these are the fused, register/shared-memory resident equivalents.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace tpr {

constexpr int kC = 32;          // plane channels == decoder inputs
constexpr int kHid = 64;        // decoder hidden width
constexpr int kOutPad = 36;     // 1 sigma + 32 colours, padded to a multiple of 4
constexpr int kHidChunk = 16;   // hidden units kept in registers at a time

// Packed decoder block (floats).  W1 is stored transposed and pre-multiplied by
// weight_gain/3 (the 1/3 is the mean over the three planes, training/triplane.py:126),
// W2 transposed, pre-multiplied by its gain and zero-padded to 36 outputs.
constexpr int kW1tOff = 0;                          // [32][64]
constexpr int kB1Off = kC * kHid;                   // [64]
constexpr int kW2tOff = kB1Off + kHid;              // [64][36]
constexpr int kB2Off = kW2tOff + kHid * kOutPad;    // [36]
constexpr int kDecFloats = kB2Off + kOutPad;        // 4452 floats = 17808 B
static_assert(kDecFloats % 4 == 0, "decoder block must be float4 copyable");

constexpr unsigned kFull = 0xffffffffu;

// ---------------------------------------------------------------------------------------
// deterministic backward (TPR_BWD_DETERMINISTIC): the scratch the decoder-backward kernels use in that mode
// ---------------------------------------------------------------------------------------
// The plane gradient is accumulated in fixed point: every contribution is scaled by 2^e (e from a bound on any texel's sum,
// so nothing overflows 2^62), rounded to int64 and added with integer reductions -- associative, so the result does not
// depend on the order of the samples.  The decoder gradient: every CTA stores its partial sums as one row, and the rows are
// summed in index order.  A launch clamps its grid to kDetMaxRows CTAs.
constexpr int kDetMaxRows = 512;
struct DetScratch {
  int* hdr;                    // [0] e, [1] non-zero: non-finite bound or contribution (the plane gradient becomes NaN),
                               // [2] the bits of the fp32 2^e
  float* rows;                 // [kDetMaxRows][kDecFloats] per-CTA decoder-gradient rows
  unsigned long long* acc;     // [N,3,H,W,32] fixed-point plane gradient (two's complement), zero-initialised
  int n_rows;                  // (host) rows the launch wrote
};

// one fixed-point contribution: v (already x 2^e) rounded to the nearest integer, added as a two's-complement u64
__device__ __forceinline__ void red_add_fixed(unsigned long long* p, float v) {
  long long q;
  asm("cvt.rni.s64.f32 %0, %1;" : "=l"(q) : "f"(v));
  asm volatile("red.global.add.u64 [%0], %1;" ::"l"(p), "l"(q) : "memory");
}
// false for NaN, +-inf and magnitudes the int64 accumulator cannot take
__device__ __forceinline__ bool fixed_ok(float4 v) {
  return fabsf(v.x) < 0x1p62f && fabsf(v.y) < 0x1p62f && fabsf(v.z) < 0x1p62f && fabsf(v.w) < 0x1p62f;
}

// ---------------------------------------------------------------------------------------
// scalar math
// ---------------------------------------------------------------------------------------
// torch.nn.Softplus(beta=1, threshold=20): log1p(exp(x)), identity above the threshold.
// MUFU ex2/lg2 based; absolute error < 3e-7 over the whole range, far inside the 1e-4 gate.
__device__ __forceinline__ float softplus_f(float x) {
  float y = __logf(1.0f + __expf(x));
  return x > 20.0f ? x : y;
}

// sigmoid(x) * 1.002 - 0.001 (training/triplane.py:134)
__device__ __forceinline__ float colour_act(float x) {
  float s = __fdividef(1.0f, 1.0f + __expf(-x));
  return fmaf(s, 1.002f, -0.001f);
}

__device__ __forceinline__ unsigned float_to_ordered(float f) {
  unsigned b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float ordered_to_float(unsigned u) {
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(kFull, v, o));
  return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(kFull, v, o));
  return v;
}
__device__ __forceinline__ double shfl_up_f64(double v, int d) {
  int lo = __double2loint(v), hi = __double2hiint(v);
  lo = __shfl_up_sync(kFull, lo, d);
  hi = __shfl_up_sync(kFull, hi, d);
  return __hiloint2double(hi, lo);
}
__device__ __forceinline__ double shfl_xor_f64(double v, int d) {
  int lo = __double2loint(v), hi = __double2hiint(v);
  lo = __shfl_xor_sync(kFull, lo, d);
  hi = __shfl_xor_sync(kFull, hi, d);
  return __hiloint2double(hi, lo);
}
// exclusive prefix product over lanes (lane 0 gets 1)
__device__ __forceinline__ float warp_excl_prod(float v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    float t = __shfl_up_sync(kFull, v, o);
    if (lane >= o) v *= t;
  }
  float e = __shfl_up_sync(kFull, v, 1);
  return lane == 0 ? 1.0f : e;
}
// exclusive prefix sum over lanes in float64 (lane 0 gets 0)
__device__ __forceinline__ double warp_excl_sum_f64(double v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    double t = shfl_up_f64(v, o);
    if (lane >= o) v += t;
  }
  double e = shfl_up_f64(v, 1);
  return lane == 0 ? 0.0 : e;
}

// ---------------------------------------------------------------------------------------
// Shared-memory row tiles.  A "row" is one sample's 32 floats (128 B): first its plane
// features, later overwritten in place by its 32 colours.  The eight 16-byte chunks of a row
// are XOR-swizzled with (row & 7) -- the same pattern as the UMMA/TMA 128B swizzle -- so both
// access shapes are bank-conflict free: 8 lanes x float4 along one row (gather, colour sum),
// and 32 lanes each walking its own row (decoder, one thread per sample).
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ int row_chunk_off(int row, int chunk) {
  return row * kC + ((chunk ^ (row & 7)) << 2);
}

// ---------------------------------------------------------------------------------------
// a3/a4: project_onto_planes + grid_sample(bilinear, zeros, align_corners=False)
//        VR/renderer.py:39-65.  plane 0 <- (x,y), plane 1 <- (x,z), plane 2 <- (z,x); the first
//        coordinate walks W.  The coordinate arithmetic uses explicitly rounded ops in the
//        reference's order so tap weights are bit-identical to the oracle's (a fused multiply-add
//        here would move weights by ~1e-5 at |ix| ~ 128).
// ---------------------------------------------------------------------------------------
struct Taps {
  int off[4];     // float offset of the tap's texel within its plane (clamped in range)
  float w[4];     // nw, ne, sw, se; zero for taps outside the plane
};

__device__ __forceinline__ void plane_taps(float gu, float gv, int H, int W, Taps& t) {
  float ix = __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(gu, 1.0f), (float)W), -1.0f), 0.5f);
  float iy = __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(gv, 1.0f), (float)H), -1.0f), 0.5f);
  float x0f = floorf(ix), y0f = floorf(iy);
  float wx1 = __fsub_rn(ix, x0f), wy1 = __fsub_rn(iy, y0f);
  float wx0 = __fsub_rn(__fadd_rn(x0f, 1.0f), ix), wy0 = __fsub_rn(__fadd_rn(y0f, 1.0f), iy);
  int x0 = (int)fminf(fmaxf(x0f, -2.0f), (float)(W + 1));
  int y0 = (int)fminf(fmaxf(y0f, -2.0f), (float)(H + 1));
  bool vx0 = (x0 >= 0) & (x0 < W), vx1 = (x0 + 1 >= 0) & (x0 + 1 < W);
  bool vy0 = (y0 >= 0) & (y0 < H), vy1 = (y0 + 1 >= 0) & (y0 + 1 < H);
  int xc0 = min(max(x0, 0), W - 1), xc1 = min(max(x0 + 1, 0), W - 1);
  int yc0 = min(max(y0, 0), H - 1), yc1 = min(max(y0 + 1, 0), H - 1);
  t.off[0] = (yc0 * W + xc0) * kC;
  t.off[1] = (yc0 * W + xc1) * kC;
  t.off[2] = (yc1 * W + xc0) * kC;
  t.off[3] = (yc1 * W + xc1) * kC;
  t.w[0] = (vx0 & vy0) ? __fmul_rn(wx0, wy0) : 0.0f;
  t.w[1] = (vx1 & vy0) ? __fmul_rn(wx1, wy0) : 0.0f;
  t.w[2] = (vx0 & vy1) ? __fmul_rn(wx0, wy1) : 0.0f;
  t.w[3] = (vx1 & vy1) ? __fmul_rn(wx1, wy1) : 0.0f;
}

__device__ __forceinline__ float4 ldg128(const float* p) {
  return __ldg(reinterpret_cast<const float4*>(p));
}

__device__ __forceinline__ void fma4(float4& a, float w, const float4& v) {
  a.x = fmaf(w, v.x, a.x); a.y = fmaf(w, v.y, a.y);
  a.z = fmaf(w, v.z, a.z); a.w = fmaf(w, v.w, a.w);
}

// Sum over the three planes of the bilinear lookups at point (px,py,pz) (already scaled by
// 2/box_warp), for the four channels [4*sub, 4*sub+4).  `img` points at this image's
// [3][H][W][32] block.  All 12 loads are issued before the first use.
__device__ __forceinline__ float4 gather_point(const float* __restrict__ img, int H, int W,
                                               float px, float py, float pz, int sub) {
  Taps t0, t1, t2;
  plane_taps(px, py, H, W, t0);
  plane_taps(px, pz, H, W, t1);
  plane_taps(pz, px, H, W, t2);
  const int plane = H * W * kC;                 // < 2^29 floats (checked on the host)
  const int l0 = sub * 4, l1 = l0 + plane, l2 = l1 + plane;
  float4 v[12];
#pragma unroll
  for (int i = 0; i < 4; ++i) v[i] = ldg128(img + (unsigned)(l0 + t0.off[i]));
#pragma unroll
  for (int i = 0; i < 4; ++i) v[4 + i] = ldg128(img + (unsigned)(l1 + t1.off[i]));
#pragma unroll
  for (int i = 0; i < 4; ++i) v[8 + i] = ldg128(img + (unsigned)(l2 + t2.off[i]));
  float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0, a2 = a0;
#pragma unroll
  for (int i = 0; i < 4; ++i) { fma4(a0, t0.w[i], v[i]); fma4(a1, t1.w[i], v[4 + i]); fma4(a2, t2.w[i], v[8 + i]); }
  return make_float4(a0.x + a1.x + a2.x, a0.y + a1.y + a2.y, a0.z + a1.z + a2.z, a0.w + a1.w + a2.w);
}

// Tap table entry for one (sample, plane): element offsets (plane offset included) and weights.
struct __align__(16) TapEntry { int off[4]; float w[4]; };

// Same as gather_point, but the 12 (offset, weight) pairs come from a shared-memory tap table that one
// lane per (sample, plane) filled beforehand -- the eight lanes of a sample no longer redo that arithmetic.
__device__ __forceinline__ float4 gather_point_taps(const float* __restrict__ img_sub, const TapEntry* __restrict__ te) {
  int4 o[3]; float4 w[3];
#pragma unroll
  for (int p = 0; p < 3; ++p) {
    o[p] = *reinterpret_cast<const int4*>(te[p].off);
    w[p] = *reinterpret_cast<const float4*>(te[p].w);
  }
  float4 v[12];
#pragma unroll
  for (int p = 0; p < 3; ++p) {
    v[4 * p + 0] = ldg128(img_sub + (unsigned)o[p].x);
    v[4 * p + 1] = ldg128(img_sub + (unsigned)o[p].y);
    v[4 * p + 2] = ldg128(img_sub + (unsigned)o[p].z);
    v[4 * p + 3] = ldg128(img_sub + (unsigned)o[p].w);
  }
  float4 a[3];
#pragma unroll
  for (int p = 0; p < 3; ++p) {
    a[p] = make_float4(0.f, 0.f, 0.f, 0.f);
    fma4(a[p], w[p].x, v[4 * p]); fma4(a[p], w[p].y, v[4 * p + 1]); fma4(a[p], w[p].z, v[4 * p + 2]); fma4(a[p], w[p].w, v[4 * p + 3]);
  }
  return make_float4(a[0].x + a[1].x + a[2].x, a[0].y + a[1].y + a[2].y, a[0].z + a[1].z + a[2].z, a[0].w + a[1].w + a[2].w);
}

// One warp gathers the plane features of its 32 samples into shared-memory rows.
// Lane L supplies sample L (point, destination row, validity); `img` (this image's
// [3][H][W][32] block) is warp-uniform.  Eight lanes cooperate on one sample so every load
// instruction fetches four whole 128-byte texels.
__device__ __forceinline__ void gather_chunk(const float* __restrict__ img, int H, int W,
                                             float px, float py, float pz, int row, bool valid,
                                             float* __restrict__ rows, int lane) {
  const int grp = lane >> 3, sub = lane & 7;
#pragma unroll 1
  for (int q = 0; q < 8; ++q) {
    const int src = q * 4 + grp;
    float sx = __shfl_sync(kFull, px, src), sy = __shfl_sync(kFull, py, src), sz = __shfl_sync(kFull, pz, src);
    int srow = __shfl_sync(kFull, row, src);
    bool sv = __shfl_sync(kFull, (int)valid, src) != 0;
    if (sv) {
      float4 f = gather_point(img, H, W, sx, sy, sz, sub);
      *reinterpret_cast<float4*>(rows + row_chunk_off(srow, sub)) = f;
    }
  }
}

// ---------------------------------------------------------------------------------------
// a5/a6: OSGDecoder in fp32 FFMA, one thread per sample (training/triplane.py:124-136,
//        training/networks_stylegan2.py:121-134).  `wsm` is the packed decoder block in shared
//        memory; all weight reads are warp-uniform float4 broadcasts.  x are the SUMMED plane
//        features (1/3 folded into W1).  out[0] = sigma, out[1..32] = colour logits.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void decoder_fp32(const float* __restrict__ wsm, const float* __restrict__ rows, int row,
                                             float (&out)[kOutPad]) {
#pragma unroll
  for (int q = 0; q < kOutPad / 4; ++q) {
    float4 b = *reinterpret_cast<const float4*>(wsm + kB2Off + q * 4);
    out[4 * q] = b.x; out[4 * q + 1] = b.y; out[4 * q + 2] = b.z; out[4 * q + 3] = b.w;
  }
#pragma unroll 1
  for (int hc = 0; hc < kHid / kHidChunk; ++hc) {
    float h[kHidChunk];
    const float* w1 = wsm + kW1tOff + hc * kHidChunk;
#pragma unroll
    for (int q = 0; q < kHidChunk / 4; ++q) {
      float4 b = *reinterpret_cast<const float4*>(wsm + kB1Off + hc * kHidChunk + q * 4);
      h[4 * q] = b.x; h[4 * q + 1] = b.y; h[4 * q + 2] = b.z; h[4 * q + 3] = b.w;
    }
    // the sample's features are re-read from its shared-memory row for every hidden chunk
    // (8 LDS.128 against 512 FFMA) so they never occupy 32 registers across the loop
#pragma unroll
    for (int c = 0; c < kC / 4; ++c) {
      const float4 xv = *reinterpret_cast<const float4*>(rows + row_chunk_off(row, c));
      const float x[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        const int k = c * 4 + kk;
#pragma unroll
        for (int q = 0; q < kHidChunk / 4; ++q) {
          float4 w = *reinterpret_cast<const float4*>(w1 + k * kHid + q * 4);
          h[4 * q] = fmaf(x[kk], w.x, h[4 * q]);
          h[4 * q + 1] = fmaf(x[kk], w.y, h[4 * q + 1]);
          h[4 * q + 2] = fmaf(x[kk], w.z, h[4 * q + 2]);
          h[4 * q + 3] = fmaf(x[kk], w.w, h[4 * q + 3]);
        }
      }
    }
#pragma unroll
    for (int j = 0; j < kHidChunk; ++j) h[j] = softplus_f(h[j]);
    const float* w2 = wsm + kW2tOff + hc * kHidChunk * kOutPad;
#pragma unroll
    for (int j = 0; j < kHidChunk; ++j) {
#pragma unroll
      for (int q = 0; q < kOutPad / 4; ++q) {
        float4 w = *reinterpret_cast<const float4*>(w2 + j * kOutPad + q * 4);
        out[4 * q] = fmaf(h[j], w.x, out[4 * q]);
        out[4 * q + 1] = fmaf(h[j], w.y, out[4 * q + 1]);
        out[4 * q + 2] = fmaf(h[j], w.z, out[4 * q + 2]);
        out[4 * q + 3] = fmaf(h[j], w.w, out[4 * q + 3]);
      }
    }
  }
}

// Decode the sample stored in shared-memory row `row` in place: features -> colours.
// Returns sigma.
__device__ __forceinline__ float decode_row_inplace(const float* __restrict__ wsm,
                                                    float* __restrict__ rows, int row) {
  float out[kOutPad];
  decoder_fp32(wsm, rows, row, out);
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    float4 v = make_float4(colour_act(out[1 + 4 * c]), colour_act(out[2 + 4 * c]),
                           colour_act(out[3 + 4 * c]), colour_act(out[4 + 4 * c]));
    *reinterpret_cast<float4*>(rows + row_chunk_off(row, c)) = v;
  }
  return out[0];
}

// Stage the packed decoder block into shared memory (whole CTA).
__device__ __forceinline__ void stage_decoder(const float* __restrict__ dec, float* wsm) {
  for (int i = threadIdx.x; i < kDecFloats / 4; i += blockDim.x)
    reinterpret_cast<float4*>(wsm)[i] = __ldg(reinterpret_cast<const float4*>(dec) + i);
}

// ---------------------------------------------------------------------------------------
// a9: MipRayMarcher2 interval arithmetic (VR/ray_marcher.py:26-42)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float interval_alpha(float d0, float d1, float s0, float s1) {
  float delta = d1 - d0;
  float dens = softplus_f((s0 + s1) * 0.5f - 1.0f);
  return 1.0f - __expf(-(dens * delta));
}

// One warp turns a ray's S (depth, sigma) pairs, taken in the given order, into the S-1
// compositing weights  w_i = alpha_i * prod_{j<i}(1 - alpha_j + 1e-10).  `w` may alias neither input.
__device__ __forceinline__ void warp_march_weights(const float* z, const float* sg, float* w, int S, int lane) {
  const int n = S - 1;
  const int per = (n + 31) >> 5;
  const int i0 = lane * per;
  float prod = 1.0f;
  for (int e = 0; e < per; ++e) {
    int i = i0 + e;
    if (i < n) {
      float a = interval_alpha(z[i], z[i + 1], sg[i], sg[i + 1]);
      w[i] = a;
      prod *= (1.0f - a + 1e-10f);
    }
  }
  float T = warp_excl_prod(prod, lane);
  for (int e = 0; e < per; ++e) {
    int i = i0 + e;
    if (i < n) {
      float a = w[i];
      w[i] = a * T;
      T *= (1.0f - a + 1e-10f);
    }
  }
}

// ---------------------------------------------------------------------------------------
// a10/a11: importance resampling (VR/renderer.py:194-253), one warp per ray.
// ---------------------------------------------------------------------------------------
// pdf weights from coarse weights: max_pool1d(2,1,pad=1) -> avg_pool1d(2,1) -> +0.01, then drop
// both ends (:205-210).  Only interior entries survive, so no -inf padding is ever read.
__device__ __forceinline__ void warp_smooth_weights(const float* w, float* pw, int nb, int lane) {
  for (int j = lane; j < nb; j += 32) {
    float a = fmaxf(w[j], w[j + 1]), b = fmaxf(w[j + 1], w[j + 2]);
    pw[j] = __fadd_rn(__fmul_rn(__fadd_rn(a, b), 0.5f), 0.01f);
  }
}

// cdf[0..nb] from pdf weights pw[0..nb) (:227-230): (pw+1e-5)/sum, cumulative sum, leading 0.
// Arithmetic contract = oracle/triplane_oracle.py:pdf_to_cdf: the row sum and the running sum are
// accumulated in float64 (exact for this data, hence order independent) and rounded to float32.
__device__ __forceinline__ void warp_cdf(const float* pw, float* cdf, int nb, int lane) {
  const int per = (nb + 31) >> 5;
  const int j0 = lane * per;
  double loc = 0.0;
  for (int e = 0; e < per; ++e) {
    int j = j0 + e;
    if (j < nb) loc += (double)__fadd_rn(pw[j], 1e-5f);
  }
  double tot = loc;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) tot += shfl_xor_f64(tot, o);
  const float totf = (float)tot;
  loc = 0.0;
  for (int e = 0; e < per; ++e) {
    int j = j0 + e;
    if (j < nb) loc += (double)__fdiv_rn(__fadd_rn(pw[j], 1e-5f), totf);
  }
  double run = warp_excl_sum_f64(loc, lane);
  for (int e = 0; e < per; ++e) {
    int j = j0 + e;
    if (j < nb) {
      run += (double)__fdiv_rn(__fadd_rn(pw[j], 1e-5f), totf);
      cdf[j + 1] = (float)run;
    }
  }
  if (lane == 0) cdf[0] = 0.0f;
}

// inverse-CDF draw for one u (:240-252).  bins are read through `bin(i)`.
template <typename BinFn>
__device__ __forceinline__ float invert_cdf(const float* cdf, int nb, float uu, BinFn bin, int& inds) {
  int lo = 0, hi = nb + 1;                 // first index with cdf[i] > u  (searchsorted right=True)
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    if (cdf[mid] <= uu) lo = mid + 1; else hi = mid;
  }
  inds = lo;
  int below = max(lo - 1, 0), above = min(lo, nb);
  float cb = cdf[below], ca = cdf[above];
  float bb = bin(below), ba = bin(above);
  float denom = __fsub_rn(ca, cb);
  if (denom < 1e-5f) denom = 1.0f;
  float t = __fdiv_rn(__fsub_rn(uu, cb), denom);
  return __fadd_rn(bb, __fmul_rn(t, __fsub_rn(ba, bb)));
}

// ---------------------------------------------------------------------------------------
// a12: unify_samples = per-ray sort by depth (VR/renderer.py:157-167).
// Bitonic network over 32*E keys held E per lane in blocked order (position = lane*E + slot);
// exchanges at distance < E stay in registers, the rest are warp shuffles.  Ties are broken
// by original index, so the result equals a stable sort.
// ---------------------------------------------------------------------------------------
template <int E>
__device__ __forceinline__ void warp_bitonic_sort(float (&key)[E], int (&idx)[E], int lane) {
#pragma unroll
  for (int k = 2; k <= 32 * E; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      if (j < E) {
#pragma unroll
        for (int e = 0; e < E; ++e) {
          int f = e ^ j;
          if (f > e) {
            int p = lane * E + e;
            bool asc = (p & k) == 0;
            bool lt = (key[f] < key[e]) || (key[f] == key[e] && idx[f] < idx[e]);
            if (lt == asc) {
              float tk = key[e]; key[e] = key[f]; key[f] = tk;
              int ti = idx[e]; idx[e] = idx[f]; idx[f] = ti;
            }
          }
        }
      } else {
        const int lj = j / E;
#pragma unroll
        for (int e = 0; e < E; ++e) {
          float ok = __shfl_xor_sync(kFull, key[e], lj);
          int oi = __shfl_xor_sync(kFull, idx[e], lj);
          int p = lane * E + e;
          bool asc = (p & k) == 0;
          bool lower = (p & j) == 0;
          bool other_lt = (ok < key[e]) || (ok == key[e] && oi < idx[e]);
          // the lower position keeps the minimum when ascending, the maximum when descending
          bool take = (lower == asc) ? other_lt : !other_lt;
          if (take) { key[e] = ok; idx[e] = oi; }
        }
      }
    }
  }
}

}  // namespace tpr
