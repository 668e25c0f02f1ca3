// Backward pass of ImportanceRenderer.forward (SURVEY.md section 8(f) row 3) for sm_100a: gradients of the rendered
// (rgb, depth, weight_sum) with respect to the tri-planes and the four OSGDecoder tensors -- what the reference's
// training step back-propagates through the renderer (training/training_loop.py:335,377).
//
// What is differentiated (citations relative to /root/reference/g_nerf/, VR/ = training/volumetric_rendering/):
//   * the importance depths are constants: the reference produces them under torch.no_grad() and detaches the coarse
//     weights (VR/renderer.py:198,210), and the coarse depths depend on the jitter only (VR/renderer.py:169-192);
//     ray origins / directions come from the camera and carry no gradient.  So the graph is
//       planes, decoder -> (colour, sigma) of the S = Dc + Df samples of a ray (VR/renderer.py:142-148)
//                       -> sort by depth (VR/renderer.py:157-167) -> final march (VR/ray_marcher.py:25-57).
//   * the first march (coarse weights) only feeds the resampling, i.e. nothing.
//
// Kernels, none of which stores per-sample activations of the decoder (the decoder's backward of the product path is
// decode_backward_tc_kernel in tpr_backward_tc.cu -- tcgen05; the mma.sync kernel below is its A/B partner, TPR_BWD_IMPL=hmma,
// and the fall-back for devices / shapes the tcgen05 kernel refuses):
//   points_kernel           sample positions origin + depth * direction of all S samples of every ray
//   (tpr_run_model)         colours and densities of those points: the forward's tcgen05 point-query kernel
//   march_backward_kernel   one warp per ray: sort, march, and the march's backward -> per sample d(loss)/d(sigma) and
//                           the composite weight omega of its colour (d(loss)/d(colour_c) = 2 * g_rgb_c * omega)
//   decode_backward_kernel  per tile of 64 samples: re-gather the features, layer 1 forward, the decoder's backward
//                           (three small GEMMs per sample tile + two outer-product GEMMs for the weight gradients, all
//                           on mma.sync m16n8k8 TF32 with the 3xTF32 split, fp32 accumulation), then the bilinear
//                           scatter of d(loss)/d(features) into the packed plane gradient with 128-bit reductions
//                           (red.global.add.v4.f32: one texel = one 128-byte line = 8 lanes).
// (DESIGN.md section 4.)
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <stdlib.h>
#include "triplane_b200.h"
#include "tpr_device.cuh"

namespace tpr {
namespace bwd {

// ---------------------------------------------------------------------------------------------------------
// sample positions (VR/renderer.py:105,123), in the forward's order: ray-major, coarse samples then importance samples
// ---------------------------------------------------------------------------------------------------------
__global__ void points_kernel(const float* __restrict__ origins, const float* __restrict__ dirs,
                              const float* __restrict__ dc, const float* __restrict__ df, int Dc, int Df,
                              long long n_rays_total, float* __restrict__ pts) {
  const int S = Dc + Df;
  const long long total = n_rays_total * S;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long g = i / S;
    const int k = (int)(i - g * S);
    const float d = k < Dc ? __ldg(dc + g * Dc + k) : __ldg(df + g * Df + (k - Dc));
    pts[3 * i + 0] = __fadd_rn(__ldg(origins + 3 * g + 0), __fmul_rn(d, __ldg(dirs + 3 * g + 0)));
    pts[3 * i + 1] = __fadd_rn(__ldg(origins + 3 * g + 1), __fmul_rn(d, __ldg(dirs + 3 * g + 1)));
    pts[3 * i + 2] = __fadd_rn(__ldg(origins + 3 * g + 2), __fmul_rn(d, __ldg(dirs + 3 * g + 2)));
  }
}

// ---------------------------------------------------------------------------------------------------------
// march backward: one warp per ray
// ---------------------------------------------------------------------------------------------------------
struct MarchArgs {
  const float* dc; const float* df; int Dc, Df;
  const float* sigma;            // [rays, S]
  const float* colours;          // [rays, S, 32], or (chunked != 0) [rays, 8, S, 4] as tpr_render_train keeps them
  int chunked;
  const float* g_rgb;            // [rays, 32]
  const float* g_depth;          // [rays]
  const float* g_wsum;           // [rays]
  const float* range;            // [2]: the forward's (min, max) of all depths (VR/ray_marcher.py:50)
  int white_back;
  long long n_rays;
  float* gsig;                   // [rays, S]   d(loss)/d(sigma), sample order
  float* omega;                  // [rays, S]   composite weight of the sample's colour
};

__device__ __forceinline__ float warp_excl_suffix_sum(float v, int lane) {
  float incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float t = __shfl_down_sync(kFull, incl, o);
    if (lane + o < 32) incl += t;
  }
  return incl - v;
}

template <int E>
__global__ void __launch_bounds__(128, 8) march_backward_kernel(const MarchArgs a) {
  extern __shared__ float sm[];
  const int S = a.Dc + a.Df, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  float* z = sm + wid * 7 * S; float* sg = z + S; float* q = sg + S;
  float* zs = q + S; float* ss = zs + S; float* qs = ss + S; int* idx = reinterpret_cast<int*>(qs + S);
  float* a2s = sm + 4 * 7 * S + wid * 32;          // 2 x the ray's upstream rgb gradient (shared memory: 32 registers less per
                                                   // thread = 10 instead of 6 resident CTAs, and the kernel waits for DRAM)
  const bool vec = (S & 3) == 0 && (a.Dc & 3) == 0; // float4 reads of the depth rows are aligned
  const float lo = __ldg(a.range), hi = __ldg(a.range + 1);
  for (long long g = blockIdx.x * 4ll + wid; g < a.n_rays; g += gridDim.x * 4ll) {
    // upstream gradient of rgb (x2: VR/ray_marcher.py:55)
    float sumA2 = 0.0f;
    if (lane < 8) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(a.g_rgb + g * 32) + lane);
      const float4 w = make_float4(2.0f * v.x, 2.0f * v.y, 2.0f * v.z, 2.0f * v.w);
      *reinterpret_cast<float4*>(a2s + 4 * lane) = w;
      sumA2 = (w.x + w.y) + (w.z + w.w);
    }
    sumA2 = warp_sum(sumA2);
    __syncwarp();
    const float B = __ldg(a.g_depth + g), C = __ldg(a.g_wsum + g);
    for (int p = lane; p < S; p += 32) {
      z[p] = p < a.Dc ? __ldg(a.dc + g * a.Dc + p) : __ldg(a.df + g * a.Df + (p - a.Dc));
      sg[p] = __ldg(a.sigma + g * S + p);
      // sample-major rows: float4 c4 of sample p at row + c4; chunk-major: at chunk c4's run of the ray + p (coalesced over lanes)
      const float4* row = reinterpret_cast<const float4*>(a.colours + g * S * 32) + (a.chunked ? p : p * 8);
      const int cstep = a.chunked ? S : 1;
      float acc = 0.0f;
#pragma unroll
      for (int c4 = 0; c4 < 8; ++c4) {
        const float4 v = __ldg(row + c4 * cstep);
        const float4 w = *reinterpret_cast<const float4*>(a2s + 4 * c4);
        acc = fmaf(w.x, v.x, acc); acc = fmaf(w.y, v.y, acc);
        acc = fmaf(w.z, v.z, acc); acc = fmaf(w.w, v.w, acc);
      }
      q[p] = acc;                                   // sum_c d(loss)/d(rgb_raw_c) * colour_c
    }
    __syncwarp();
    // sort by depth (VR/renderer.py:157-167): rank = number of smaller depths, ties by sample index (a stable sort).  The
    // coarse depths of a ray ascend (stratified: VR/renderer.py:199-224), so a coarse sample's rank among them is its index and
    // an importance sample's is an upper bound found by bisection; only the Df importance depths are compared one by one.
    // Fast path: importance depths counted with strict compares, four per shared-memory read; two EQUAL importance depths would
    // then share a rank, which the rank sum detects -- the exact loop (ties by index) runs again only for such a ray.
    bool ascending = true;
    for (int p = lane; p + 1 < a.Dc; p += 32) ascending = ascending && (z[p] <= z[p + 1]);
    ascending = __all_sync(kFull, ascending);
    int cnt[E];
    bool exact = !(ascending && vec);
    if (!exact) {
      int rsum = 0;
#pragma unroll
      for (int e = 0; e < E; ++e) {
        const int p = lane + 32 * e;
        cnt[e] = 0;
        if (p < S) {
          const float zp = z[p];
          int c = p;
          if (p >= a.Dc) {
            int lo_i = 0, hi_i = a.Dc;                      // first coarse index whose depth is > zp
            while (lo_i < hi_i) { const int mid = (lo_i + hi_i) >> 1; if (z[mid] <= zp) lo_i = mid + 1; else hi_i = mid; }
            c = lo_i;
          }
          for (int j = a.Dc; j < S; j += 4) {
            const float4 v = *reinterpret_cast<const float4*>(z + j);
            c += (int)(v.x < zp) + (int)(v.y < zp) + (int)(v.z < zp) + (int)(v.w < zp);
          }
          cnt[e] = c;
          rsum += c;
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) rsum += __shfl_xor_sync(kFull, rsum, o);
      exact = rsum != S * (S - 1) / 2;                      // (warp-uniform)
    }
    if (exact) {
#pragma unroll
      for (int e = 0; e < E; ++e) {
        const int p = lane + 32 * e;
        cnt[e] = 0;
        if (p < S) {
          const float zp = z[p];
          int c = 0;
          for (int j = 0; j < S; ++j) { const float v = z[j]; c += (int)((v < zp) || (v == zp && j < p)); }
          cnt[e] = c;
        }
      }
    }
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int p = lane + 32 * e;
      if (p < S) { zs[cnt[e]] = z[p]; ss[cnt[e]] = sg[p]; qs[cnt[e]] = q[p]; idx[cnt[e]] = p; }
    }
    __syncwarp();
    // blocked: position p = lane * E + e
    float key[E + 1], sgm[E + 1], qq[E + 1];
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int p = lane * E + e;
      key[e] = p < S ? zs[p] : 0.0f; sgm[e] = p < S ? ss[p] : 0.0f; qq[e] = p < S ? qs[p] : 0.0f;
    }
    key[E] = __shfl_down_sync(kFull, key[0], 1); sgm[E] = __shfl_down_sync(kFull, sgm[0], 1); qq[E] = __shfl_down_sync(kFull, qq[0], 1);
    // forward march (VR/ray_marcher.py:26-46)
    float al[E], ex[E], om1[E], dm[E], sx[E], T[E], w[E];
    float prod = 1.0f;
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int p = lane * E + e;
      const bool valid = p + 1 < S;
      const float delta = key[e + 1] - key[e];
      const float x = (sgm[e] + sgm[e + 1]) * 0.5f - 1.0f;
      const float t = __expf(x);
      const float dens = x > 20.0f ? x : __logf(1.0f + t);
      sx[e] = x > 20.0f ? 1.0f : __fdividef(t, 1.0f + t);      // softplus'(x)
      ex[e] = valid ? __expf(-(dens * delta)) : 1.0f;
      al[e] = valid ? 1.0f - ex[e] : 0.0f;
      om1[e] = 1.0f - al[e] + 1e-10f;
      dm[e] = (key[e] + key[e + 1]) * 0.5f;
      if (valid) prod *= om1[e];
    }
    float Tr = warp_excl_prod(prod, lane);
    float wsum = 0.0f, dnum = 0.0f;
#pragma unroll
    for (int e = 0; e < E; ++e) {
      T[e] = Tr; w[e] = al[e] * Tr;
      if (lane * E + e + 1 < S) Tr *= om1[e];
      wsum += w[e]; dnum = fmaf(w[e], dm[e], dnum);
    }
    wsum = warp_sum(wsum); dnum = warp_sum(dnum);
    const float depth_raw = dnum / wsum;
    // nan_to_num + clamp (VR/ray_marcher.py:49-50): the gradient passes only where the depth is inside the range
    const bool pass = depth_raw >= lo && depth_raw <= hi;
    const float bscale = pass ? B / wsum : 0.0f;
    const float wb = a.white_back ? sumA2 : 0.0f;               // rgb += 1 - sum(w) (VR/ray_marcher.py:52-53)
    float gw[E], u[E], lane_tot = 0.0f;
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const bool valid = lane * E + e + 1 < S;
      gw[e] = valid ? 0.5f * (qq[e] + qq[e + 1]) - wb + C + (pass ? bscale * (dm[e] - depth_raw) : 0.0f) : 0.0f;
      u[e] = gw[e] * w[e];
      lane_tot += u[e];
    }
    float run = warp_excl_suffix_sum(lane_tot, lane);           // sum of u over all later lanes
    float gx[E];
#pragma unroll
    for (int e = E - 1; e >= 0; --e) {
      const bool valid = lane * E + e + 1 < S;
      // w_i = alpha_i T_i, T_j = prod_{k<j} (1 - alpha_k + 1e-10):  d/d(alpha_i) = gw_i T_i - sum_{j>i} gw_j w_j / (1 - alpha_i + 1e-10)
      const float galpha = gw[e] * T[e] - run / om1[e];
      run += u[e];
      const float delta = key[e + 1] - key[e];
      gx[e] = valid ? galpha * delta * ex[e] * sx[e] : 0.0f;   // alpha = 1 - exp(-softplus(x) delta)
    }
    float gx_prev = __shfl_up_sync(kFull, gx[E - 1], 1), w_prev = __shfl_up_sync(kFull, w[E - 1], 1);
    if (lane == 0) { gx_prev = 0.0f; w_prev = 0.0f; }
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int p = lane * E + e;
      if (p < S) {
        const float gxp = e == 0 ? gx_prev : gx[e > 0 ? e - 1 : 0], wp = e == 0 ? w_prev : w[e > 0 ? e - 1 : 0];
        a.gsig[g * S + idx[p]] = 0.5f * (gxp + gx[e]);           // sigma_mid = (sigma_i + sigma_{i+1}) / 2
        a.omega[g * S + idx[p]] = 0.5f * (wp + w[e]);            // colour_mid likewise (VR/ray_marcher.py:27)
      }
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------------------------
// decoder backward + plane-gradient scatter
// ---------------------------------------------------------------------------------------------------------
constexpr int kT = 64;                  // samples per tile
constexpr int kBT = 256;                // threads per CTA: 8 warps = 4 row blocks of 16 samples x 2 warps (column halves)
constexpr int FS = 36, HS = 72, YS = 44, W1S = 72, W2S = kOutPad;    // shared-memory row strides (floats)
static_assert(W2S == 36, "W2t B-fragment loads assume a row stride of 36 floats");

// ~108 KB: two CTAs (16 warps) per SM.  The decoder weights are kept pre-split into their TF32 hi and lo parts.
struct __align__(16) Smem {
  float w1t[2][kC * W1S];               // [hi, lo][k][j]   (W1 * gain / 3)
  float w2t[2][kHid * W2S + 40];        // [hi, lo][j][o]   (W2 * gain), then finite padding for the K = 36..39 tail reads
  float b1[kHid];
  float F[kT * FS];                     // summed plane features
  float H[kT * HS];                     // softplus(layer 1)
  float GA[kT * HS];                    // d/d(layer-1 pre-activation)
  float GY[kT * YS];                    // d/d(decoder outputs): [0] sigma, [1..32] colour logits, [33..43] = 0
  float GF[kT * FS];                    // d/d(features)
  uint32_t tap_off[kT * 12];            // float offset of each tap's texel inside its image
  float tap_w[kT * 12];
  int simg[kT];
};

struct DecArgs {
  const float* planes; int H, W;        // packed [N,3,H,W,32]
  const float* dec;                     // packed decoder
  const float* pts;                     // [T,3]
  const float* colours;                 // [T,32], or (col_chunked != 0) [rays, 8, S, 4]
  int col_chunked;
  const float* features;                // [T,32] summed plane features kept by the forward, or NULL: gather them again
  const float* gsig; const float* omega;// [T] (point queries: omega unused)
  const float* g_rgb;                   // [rays,32]; point queries: [T,32] or NULL (sigma only)
  long long total, pts_per_img; int S;
  float box_scale;
  float* g_planes;                      // packed, zero-initialised
  float* g_dec;                         // [kDecFloats], zero-initialised
  int debug;                            // bit 0: no plane-gradient scatter, bit 1: no weight-gradient phase (the caller does not want
                                        // that gradient; TPR_BWD_DEBUG ORs into it for profiling A/B runs)
};
// DET (deterministic mode): the plane gradient goes to g_acc in fixed point (scale 2^e from det_hdr), the decoder gradient to
// this CTA's row of dec_rows (a separate type, so that the default kernels' parameter block stays as it is)
struct DetDecArgs : DecArgs {
  unsigned long long* g_acc; float* dec_rows; int* det_hdr;
};

__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x) & 0xffffe000u;          // the tensor core reads the top 19 bits of an fp32 register
  lo = __float_as_uint(x - __uint_as_float(hi));
}
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
// 3xTF32: x = hi + lo; a.b ~ a_lo.b_hi + a_hi.b_lo + a_hi.b_hi (small terms first)
__device__ __forceinline__ void mma3(float (&d)[4], const uint32_t (&ah)[4], const uint32_t (&al)[4], const uint32_t (&bh)[2],
                                     const uint32_t (&bl)[2]) {
  mma_tf32(d, al, bh);
  mma_tf32(d, ah, bl);
  mma_tf32(d, ah, bh);
}
template <bool FAST>
__device__ __forceinline__ void split_op(float x, uint32_t& hi, uint32_t& lo) {
  if (FAST) { asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hi) : "f"(x)); lo = 0u; }
  else split_tf32(x, hi, lo);
}
__device__ __forceinline__ void pair_sync(int id) { asm volatile("bar.sync %0, 64;" ::"r"(id) : "memory"); }

// FAST = false: 3xTF32 (fp32-grade gradients, the parity mode).  FAST = true (decoder_precision = 'bf16', the caller's
// reduced-precision mode): operands rounded to TF32 (round to nearest), one HMMA per product.
// POINT = true: point queries (ImportanceRenderer.run_model under autograd), as in decode_backward_tc_kernel: colours and g_rgb
// rows per point, GY colour = g_rgb x 1.002 x s(1-s), no omega; g_rgb == NULL reads no colours (sigma only).
// DET = true: the deterministic mode (DecArgs::g_acc).
template <bool FAST, bool POINT, bool DET = false, class Args = DecArgs>
__global__ void __launch_bounds__(kBT, 2) decode_backward_kernel(const Args a) {
  extern __shared__ uint8_t smem_raw[];
  Smem& s = *reinterpret_cast<Smem*>(smem_raw + ((16u - ((uint32_t)__cvta_generic_to_shared(smem_raw) & 15u)) & 15u));
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;           // mma fragment coordinates
  const int grp = lane >> 3, sub = lane & 7;       // gather: 8 lanes per sample
  const int mt = warp >> 1, hf = warp & 1;         // row block of 16 samples, column half
  const int row0 = mt * 16;
  const bool want_col = !POINT || a.g_rgb != nullptr;
  // ---- stage the decoder, split once
  for (int i = tid; i < kC * kHid; i += kBT) {
    const int k = i >> 6, j = i & 63;
    uint32_t hi, lo; split_op<FAST>(__ldg(a.dec + kW1tOff + i), hi, lo);
    s.w1t[0][k * W1S + j] = __uint_as_float(hi); s.w1t[1][k * W1S + j] = __uint_as_float(lo);
  }
  for (int i = tid; i < kHid * W2S + 40; i += kBT) {
    const float v = i < kHid * W2S ? __ldg(a.dec + kW2tOff + i) : (i - kHid * W2S < kOutPad ? __ldg(a.dec + kB2Off + i - kHid * W2S) : 0.0f);
    uint32_t hi, lo; split_op<FAST>(v, hi, lo);
    s.w2t[0][i] = __uint_as_float(hi); s.w2t[1][i] = __uint_as_float(lo);
  }
  if (tid < kHid) s.b1[tid] = __ldg(a.dec + kB1Off + tid);
  for (int i = tid; i < kT * (YS - 33); i += kBT) { const int r = i / (YS - 33); s.GY[r * YS + 33 + (i - r * (YS - 33))] = 0.0f; }
  __syncthreads();

  // weight-gradient accumulators of this warp: one 16-row block of gW2t (5 column blocks) or of gW1t (4 column blocks)
  float pacc[5][4];
#pragma unroll
  for (int i = 0; i < 5; ++i) { pacc[i][0] = pacc[i][1] = pacc[i][2] = pacc[i][3] = 0.0f; }
  float bacc = 0.0f;                               // tid < 64: gb1[tid]; 64 <= tid < 104: gb2[tid - 64]
  const size_t img_stride = (size_t)3 * a.H * a.W * kC;
  const long long n_tiles = (a.total + kT - 1) / kT;

  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long gs0 = tile * kT;
    const long long n0 = gs0 / a.pts_per_img, rem0 = gs0 - n0 * a.pts_per_img;
    const long long ray0 = POINT ? 0 : gs0 / a.S;
    const int rr0 = POINT ? 0 : (int)(gs0 - ray0 * a.S);
    // ---- taps of this warp's 8 samples x 3 planes (VR/renderer.py:39-65)
    if (lane < 24) {
      const int sl = lane / 3, p = lane - sl * 3, sr = row0 + 8 * hf + sl;
      const long long gs = gs0 + sr;
      Taps tp;
      int n = 0;
      if (gs < a.total) {
        const float px = __fmul_rn(__ldg(a.pts + 3 * gs + 0), a.box_scale), py = __fmul_rn(__ldg(a.pts + 3 * gs + 1), a.box_scale),
                    pz = __fmul_rn(__ldg(a.pts + 3 * gs + 2), a.box_scale);
        plane_taps(p == 2 ? pz : px, p == 0 ? py : (p == 1 ? pz : px), a.H, a.W, tp);      // (x,y) (x,z) (z,x)
        long long r = rem0 + sr; n = (int)n0;
        while (r >= a.pts_per_img) { r -= a.pts_per_img; ++n; }
      } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) { tp.off[k] = 0; tp.w[k] = 0.0f; }
      }
      const int po = p * a.H * a.W * kC;
      *reinterpret_cast<uint4*>(s.tap_off + sr * 12 + p * 4) = make_uint4((uint32_t)(tp.off[0] + po), (uint32_t)(tp.off[1] + po),
                                                                          (uint32_t)(tp.off[2] + po), (uint32_t)(tp.off[3] + po));
      *reinterpret_cast<float4*>(s.tap_w + sr * 12 + p * 4) = make_float4(tp.w[0], tp.w[1], tp.w[2], tp.w[3]);
      if (p == 0) s.simg[sr] = n;
    }
    __syncwarp();
    // ---- gather: F = sum over planes and taps (the plane mean's 1/3 is folded into W1t)
#pragma unroll 1
    for (int it = 0; it < 2; ++it) {
      const int sr = row0 + 8 * hf + it * 4 + grp;
      const long long gsf = gs0 + sr;
      const bool kept = !POINT && a.features != nullptr;        // (point queries: always gathered again)
      const float4* img = reinterpret_cast<const float4*>(a.planes + (size_t)s.simg[sr] * img_stride) + sub;
      float4 v[12];
      float4 fk = make_float4(0.f, 0.f, 0.f, 0.f);
      if (kept) {
        if (gsf < a.total) fk = __ldg(reinterpret_cast<const float4*>(a.features + gsf * 32) + sub);
      } else {
#pragma unroll
        for (int k = 0; k < 12; ++k) v[k] = __ldg(img + (s.tap_off[sr * 12 + k] >> 2));
      }
      // ---- upstream gradient of the decoder outputs of this sample (loads overlap the texel fetches)
      const long long gs = gs0 + sr;
      float gy[4] = {0.f, 0.f, 0.f, 0.f};
      float gs_sig = 0.0f;
      if (gs < a.total) gs_sig = __ldg(a.gsig + gs);
      if (gs < a.total && want_col) {
        const long long ray = POINT ? gs : ray0 + (unsigned)(rr0 + sr) / (unsigned)a.S;      // the row of g_rgb
        const float4 col = (!POINT && a.col_chunked)
            ? __ldg(reinterpret_cast<const float4*>(a.colours + ray * a.S * 32) + sub * a.S + (gs - ray * a.S))
            : __ldg(reinterpret_cast<const float4*>(a.colours + gs * 32) + sub);
        const float4 A = __ldg(reinterpret_cast<const float4*>(a.g_rgb + ray * 32) + sub);
        // rgb*2-1 (VR/ray_marcher.py:55), sigmoid*1.002 (training/triplane.py:134)
        const float om = POINT ? 1.002f : __ldg(a.omega + gs) * (2.0f * 1.002f);
        const float cc[4] = {col.x, col.y, col.z, col.w}, aa[4] = {A.x, A.y, A.z, A.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float sv = (cc[k] + 0.001f) * (1.0f / 1.002f);           // sigmoid(logit)
          gy[k] = aa[k] * om * sv * (1.0f - sv);
        }
      }
      float* gyr = s.GY + sr * YS;
#pragma unroll
      for (int k = 0; k < 4; ++k) gyr[1 + 4 * sub + k] = gy[k];
      if (sub == 0) gyr[0] = gs_sig;
      float4 acc = fk;
      if (!kept) {
#pragma unroll
        for (int k = 0; k < 12; ++k) {
          const float w = s.tap_w[sr * 12 + k];
          acc.x = fmaf(w, v[k].x, acc.x); acc.y = fmaf(w, v[k].y, acc.y); acc.z = fmaf(w, v[k].z, acc.z); acc.w = fmaf(w, v[k].w, acc.w);
        }
      }
      *reinterpret_cast<float4*>(s.F + sr * FS + 4 * sub) = acc;
    }
    pair_sync(1 + mt);                             // F and GY of the 16 rows are complete

    // ---- layer 1 forward for rows row0 + {g, g+8}, hidden units [32 hf, 32 hf + 32): a = F . W1t + b1.
    //      Four column blocks are accumulated side by side and the three TF32 passes are issued block by block, so that
    //      consecutive HMMAs never depend on each other (each accumulator chain is 12 HMMAs long).
    float sgd[4][4];                               // softplus'(a) = sigmoid(a), later d/d(a)
    {
      float acc[4][4];
#pragma unroll
      for (int n4 = 0; n4 < 4; ++n4) {
        const int nt = 4 * hf + n4;
        acc[n4][0] = acc[n4][2] = s.b1[8 * nt + 2 * t]; acc[n4][1] = acc[n4][3] = s.b1[8 * nt + 2 * t + 1];
      }
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        uint32_t ah[4], al[4];
        const float* f0 = s.F + (row0 + g) * FS + 8 * ks + t;
        split_op<FAST>(f0[0], ah[0], al[0]); split_op<FAST>(f0[8 * FS], ah[1], al[1]);
        split_op<FAST>(f0[4], ah[2], al[2]); split_op<FAST>(f0[8 * FS + 4], ah[3], al[3]);
        uint32_t bh[4][2], bl[4][2];
#pragma unroll
        for (int n4 = 0; n4 < 4; ++n4) {
          const int o0 = (8 * ks + t) * W1S + 8 * (4 * hf + n4) + g;
          bh[n4][0] = __float_as_uint(s.w1t[0][o0]); bh[n4][1] = __float_as_uint(s.w1t[0][o0 + 4 * W1S]);
          bl[n4][0] = __float_as_uint(s.w1t[1][o0]); bl[n4][1] = __float_as_uint(s.w1t[1][o0 + 4 * W1S]);
        }
#pragma unroll
        for (int n4 = 0; n4 < 4; ++n4) if (!FAST) mma_tf32(acc[n4], al, bh[n4]);
#pragma unroll
        for (int n4 = 0; n4 < 4; ++n4) if (!FAST) mma_tf32(acc[n4], ah, bl[n4]);
#pragma unroll
        for (int n4 = 0; n4 < 4; ++n4) mma_tf32(acc[n4], ah, bh[n4]);
      }
#pragma unroll
      for (int n4 = 0; n4 < 4; ++n4) {
        const int nt = 4 * hf + n4;
        float h[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float e = __expf(acc[n4][i]), d = 1.0f + e;
          h[i] = acc[n4][i] > 20.0f ? acc[n4][i] : __logf(d);         // Softplus(beta=1, threshold=20)
          sgd[n4][i] = acc[n4][i] > 20.0f ? 1.0f : __fdividef(e, d);
        }
        *reinterpret_cast<float2*>(s.H + (row0 + g) * HS + 8 * nt + 2 * t) = make_float2(h[0], h[1]);
        *reinterpret_cast<float2*>(s.H + (row0 + g + 8) * HS + 8 * nt + 2 * t) = make_float2(h[2], h[3]);
      }
    }
    // ---- d/d(hidden) = GY . W2 (K = 40 outputs, 33 real), times softplus' -> d/d(a)
    {
      float acc[4][4];
#pragma unroll
      for (int n4 = 0; n4 < 4; ++n4) { acc[n4][0] = acc[n4][1] = acc[n4][2] = acc[n4][3] = 0.0f; }
#pragma unroll
      for (int ks = 0; ks < 5; ++ks) {
        uint32_t ah[4], al[4];
        const float* y0 = s.GY + (row0 + g) * YS + 8 * ks + t;
        split_op<FAST>(y0[0], ah[0], al[0]); split_op<FAST>(y0[8 * YS], ah[1], al[1]);
        split_op<FAST>(y0[4], ah[2], al[2]); split_op<FAST>(y0[8 * YS + 4], ah[3], al[3]);
        uint32_t bh[4][2], bl[4][2];
#pragma unroll
        for (int n4 = 0; n4 < 4; ++n4) {
          const int o0 = (8 * (4 * hf + n4) + g) * W2S + 8 * ks + t;
          bh[n4][0] = __float_as_uint(s.w2t[0][o0]); bh[n4][1] = __float_as_uint(s.w2t[0][o0 + 4]);
          bl[n4][0] = __float_as_uint(s.w2t[1][o0]); bl[n4][1] = __float_as_uint(s.w2t[1][o0 + 4]);
        }
#pragma unroll
        for (int n4 = 0; n4 < 4; ++n4) if (!FAST) mma_tf32(acc[n4], al, bh[n4]);
#pragma unroll
        for (int n4 = 0; n4 < 4; ++n4) if (!FAST) mma_tf32(acc[n4], ah, bl[n4]);
#pragma unroll
        for (int n4 = 0; n4 < 4; ++n4) mma_tf32(acc[n4], ah, bh[n4]);
      }
#pragma unroll
      for (int n4 = 0; n4 < 4; ++n4) {
        const int nt = 4 * hf + n4;
#pragma unroll
        for (int i = 0; i < 4; ++i) sgd[n4][i] *= acc[n4][i];
        *reinterpret_cast<float2*>(s.GA + (row0 + g) * HS + 8 * nt + 2 * t) = make_float2(sgd[n4][0], sgd[n4][1]);
        *reinterpret_cast<float2*>(s.GA + (row0 + g + 8) * HS + 8 * nt + 2 * t) = make_float2(sgd[n4][2], sgd[n4][3]);
      }
    }
    pair_sync(1 + mt);                             // GA of the 16 rows (both column halves) is complete
    // ---- d/d(features) = GA . W1t^T, channels [16 hf, 16 hf + 16).  The K index (hidden unit) is permuted inside every
    //      block of eight (k' = t <-> 2t, k' = t+4 <-> 2t+1) on both operands, so that each is one 64-bit load.
    //      Even and odd K blocks go to separate accumulators (four independent chains).
    {
      float acc[2][2][4];
#pragma unroll
      for (int n2 = 0; n2 < 2; ++n2)
#pragma unroll
        for (int par = 0; par < 2; ++par) { acc[n2][par][0] = acc[n2][par][1] = acc[n2][par][2] = acc[n2][par][3] = 0.0f; }
#pragma unroll
      for (int q2 = 0; q2 < 4; ++q2) {
        uint32_t ah[2][4], al[2][4], bh[2][2][2], bl[2][2][2];
#pragma unroll
        for (int par = 0; par < 2; ++par) {
          const int q = 2 * q2 + par;
          const float2 a01 = *reinterpret_cast<const float2*>(s.GA + (row0 + g) * HS + 8 * q + 2 * t);
          const float2 a23 = *reinterpret_cast<const float2*>(s.GA + (row0 + g + 8) * HS + 8 * q + 2 * t);
          split_op<FAST>(a01.x, ah[par][0], al[par][0]); split_op<FAST>(a23.x, ah[par][1], al[par][1]);
          split_op<FAST>(a01.y, ah[par][2], al[par][2]); split_op<FAST>(a23.y, ah[par][3], al[par][3]);
#pragma unroll
          for (int n2 = 0; n2 < 2; ++n2) {
            const int o0 = (8 * (2 * hf + n2) + g) * W1S + 8 * q + 2 * t;
            const float2 wh = *reinterpret_cast<const float2*>(s.w1t[0] + o0), wl = *reinterpret_cast<const float2*>(s.w1t[1] + o0);
            bh[par][n2][0] = __float_as_uint(wh.x); bh[par][n2][1] = __float_as_uint(wh.y);
            bl[par][n2][0] = __float_as_uint(wl.x); bl[par][n2][1] = __float_as_uint(wl.y);
          }
        }
#pragma unroll
        for (int par = 0; par < 2; ++par)
#pragma unroll
          for (int n2 = 0; n2 < 2; ++n2) if (!FAST) mma_tf32(acc[n2][par], al[par], bh[par][n2]);
#pragma unroll
        for (int par = 0; par < 2; ++par)
#pragma unroll
          for (int n2 = 0; n2 < 2; ++n2) if (!FAST) mma_tf32(acc[n2][par], ah[par], bl[par][n2]);
#pragma unroll
        for (int par = 0; par < 2; ++par)
#pragma unroll
          for (int n2 = 0; n2 < 2; ++n2) mma_tf32(acc[n2][par], ah[par], bh[par][n2]);
      }
#pragma unroll
      for (int n2 = 0; n2 < 2; ++n2) {
        const int nt = 2 * hf + n2;
        *reinterpret_cast<float2*>(s.GF + (row0 + g) * FS + 8 * nt + 2 * t) =
            make_float2(acc[n2][0][0] + acc[n2][1][0], acc[n2][0][1] + acc[n2][1][1]);
        *reinterpret_cast<float2*>(s.GF + (row0 + g + 8) * FS + 8 * nt + 2 * t) =
            make_float2(acc[n2][0][2] + acc[n2][1][2], acc[n2][0][3] + acc[n2][1][3]);
      }
    }
    __syncthreads();                                // F, H, GA, GY, GF of all 64 samples are in shared memory

    // ---- scatter d/d(features) to the twelve texels of each sample: the transpose of the bilinear gather
#pragma unroll 1
    for (int it = 0; it < 2; ++it) {
      const int sr = row0 + 8 * hf + it * 4 + grp;
      if constexpr (DET) {
        // deterministic: GF x 2^e, four fixed-point reductions per lane and texel
        if (a.debug & 1) continue;
        const float fx = __int_as_float(__ldg(a.det_hdr + 2));
        float4 gf = *reinterpret_cast<const float4*>(s.GF + sr * FS + 4 * sub);
        gf = make_float4(gf.x * fx, gf.y * fx, gf.z * fx, gf.w * fx);
        if (!fixed_ok(gf)) a.det_hdr[1] = 1;
        unsigned long long* img = a.g_acc + (size_t)s.simg[sr] * img_stride + 4 * sub;
#pragma unroll
        for (int k = 0; k < 12; ++k) {
          const float w = s.tap_w[sr * 12 + k];
          if (w != 0.0f) {
            unsigned long long* t = img + s.tap_off[sr * 12 + k];
            red_add_fixed(t, w * gf.x); red_add_fixed(t + 1, w * gf.y); red_add_fixed(t + 2, w * gf.z); red_add_fixed(t + 3, w * gf.w);
          }
        }
        continue;
      }
      const float4 gf = *reinterpret_cast<const float4*>(s.GF + sr * FS + 4 * sub);
      float4* img = reinterpret_cast<float4*>(a.g_planes + (size_t)s.simg[sr] * img_stride) + sub;
#pragma unroll
      for (int k = 0; k < 12; ++k) {
        const float w = s.tap_w[sr * 12 + k];
        if (w != 0.0f && !(a.debug & 1)) atomicAdd(img + (s.tap_off[sr * 12 + k] >> 2), make_float4(w * gf.x, w * gf.y, w * gf.z, w * gf.w));
      }
    }
    // ---- weight gradients: sums over the tile's 64 samples of H (x) GY (gW2t [64 x 40]: warps 0-3, 16 rows x 5 column
    //      blocks each) and F (x) GA (gW1t [32 x 64]: warps 4-7, 16 rows x 4 column blocks each).  The A fragment of a
    //      K step is loaded and split once for all column blocks of the warp.
    if (!(a.debug & 2)) {
      const bool second = warp < 4;                                  // gW2t
      const int pm = second ? warp : (warp - 4) >> 1;
      const int pn0 = second ? 0 : 4 * ((warp - 4) & 1);
      const float* As = second ? s.H : s.F; const int as = second ? HS : FS;
      const float* Bs = second ? s.GY : s.GA; const int bs = second ? YS : HS;
      const float* ap = As + t * as + 16 * pm + g;
      const float* bp = Bs + t * bs + 8 * pn0 + g;
#pragma unroll 2
      for (int ks = 0; ks < kT / 8; ++ks) {
        uint32_t ah[4], al[4], bh[5][2], bl[5][2];
        split_op<FAST>(ap[0], ah[0], al[0]); split_op<FAST>(ap[8], ah[1], al[1]);
        split_op<FAST>(ap[4 * as], ah[2], al[2]); split_op<FAST>(ap[4 * as + 8], ah[3], al[3]);
#pragma unroll
        for (int i = 0; i < 4; ++i) { split_op<FAST>(bp[8 * i], bh[i][0], bl[i][0]); split_op<FAST>(bp[4 * bs + 8 * i], bh[i][1], bl[i][1]); }
        if (second) { split_op<FAST>(bp[32], bh[4][0], bl[4][0]); split_op<FAST>(bp[4 * bs + 32], bh[4][1], bl[4][1]); }
#pragma unroll
        for (int i = 0; i < 4; ++i) if (!FAST) mma_tf32(pacc[i], al, bh[i]);
        if (second) if (!FAST) mma_tf32(pacc[4], al, bh[4]);
#pragma unroll
        for (int i = 0; i < 4; ++i) if (!FAST) mma_tf32(pacc[i], ah, bl[i]);
        if (second) if (!FAST) mma_tf32(pacc[4], ah, bl[4]);
#pragma unroll
        for (int i = 0; i < 4; ++i) mma_tf32(pacc[i], ah, bh[i]);
        if (second) mma_tf32(pacc[4], ah, bh[4]);
        ap += 8 * as; bp += 8 * bs;
      }
    }
    if (a.debug & 2) {
    } else if (tid < kHid) {
      float acc = 0.0f;
#pragma unroll 8
      for (int r = 0; r < kT; ++r) acc += s.GA[r * HS + tid];
      bacc += acc;
    } else if (tid < kHid + 40) {
      float acc = 0.0f;
#pragma unroll 8
      for (int r = 0; r < kT; ++r) acc += s.GY[r * YS + tid - kHid];
      bacc += acc;
    }
    __syncthreads();                                // the tile buffers are rewritten by the next tile
  }

  // ---- flush this CTA's partial weight gradients
  if (a.debug & 2) return;
  if constexpr (DET) {
    // deterministic: every element has one owning thread, which stores it into the CTA's row
    float* drow = a.dec_rows + (size_t)blockIdx.x * kDecFloats;
    const bool second = warp < 4;
    const int pm = second ? warp : (warp - 4) >> 1;
    const int pn0 = second ? 0 : 4 * ((warp - 4) & 1);
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      if (i < 4 || second) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const int m = 16 * pm + g + (r >> 1) * 8, n = 8 * (pn0 + i) + 2 * t + (r & 1);
          if (!second) drow[kW1tOff + m * kHid + n] = pacc[i][r];
          else if (n < kOutPad) drow[kW2tOff + m * kOutPad + n] = pacc[i][r];
        }
      }
    }
    if (tid < kHid) drow[kB1Off + tid] = bacc;
    else if (tid < kHid + kOutPad) drow[kB2Off + tid - kHid] = bacc;
    return;
  }
  {
    const bool second = warp < 4;
    const int pm = second ? warp : (warp - 4) >> 1;
    const int pn0 = second ? 0 : 4 * ((warp - 4) & 1);
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      if (i < 4 || second) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const int m = 16 * pm + g + (r >> 1) * 8, n = 8 * (pn0 + i) + 2 * t + (r & 1);
          if (!second) atomicAdd(a.g_dec + kW1tOff + m * kHid + n, pacc[i][r]);             // gW1t[k = m][j = n]
          else if (n < kOutPad) atomicAdd(a.g_dec + kW2tOff + m * kOutPad + n, pacc[i][r]);  // gW2t[j = m][o = n]
        }
      }
    }
  }
  if (tid < kHid) atomicAdd(a.g_dec + kB1Off + tid, bacc);
  else if (tid < kHid + kOutPad) atomicAdd(a.g_dec + kB2Off + tid - kHid, bacc);
}

// deterministic mode, after the decoder-backward kernel: the fixed-point accumulator -> the fp32 packed plane gradient (NaN
// everywhere when the bound or a contribution was not finite), and the per-CTA rows summed in index order in fp64, rounded once
__global__ void det_planes_kernel(const long long* __restrict__ acc, long long n4, const int* __restrict__ hdr, float* __restrict__ out) {
  const double inv = ldexp(1.0, -__ldg(hdr));
  const bool bad = __ldg(hdr + 1) != 0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const longlong2 u = __ldg(reinterpret_cast<const longlong2*>(acc) + 2 * i), v = __ldg(reinterpret_cast<const longlong2*>(acc) + 2 * i + 1);
    float4 r = make_float4(__double2float_rn((double)u.x * inv), __double2float_rn((double)u.y * inv),
                           __double2float_rn((double)v.x * inv), __double2float_rn((double)v.y * inv));
    if (bad) r = make_float4(__int_as_float(0x7fffffff), __int_as_float(0x7fffffff), __int_as_float(0x7fffffff), __int_as_float(0x7fffffff));
    reinterpret_cast<float4*>(out)[i] = r;
  }
}
__global__ void det_rows_kernel(const float* __restrict__ rows, int n_rows, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= kDecFloats) return;
  double sum = 0.0;
  for (int r = 0; r < n_rows; ++r) sum += (double)__ldg(rows + (size_t)r * kDecFloats + i);
  out[i] = (float)sum;
}

// packed decoder gradient -> gradients of the module's raw tensors (training/networks_stylegan2.py:118-127: the runtime gains)
__global__ void unpack_decoder_grad_kernel(const float* __restrict__ gd, float g_w1, float g_b1, float g_w2, float g_b2,
                                           float* __restrict__ w1, float* __restrict__ b1, float* __restrict__ w2,
                                           float* __restrict__ b2) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < kHid * kC) { const int j = i / kC, k = i - j * kC; w1[i] = gd[kW1tOff + k * kHid + j] * (g_w1 * (1.0f / 3.0f)); }
  if (i < kHid) b1[i] = gd[kB1Off + i] * g_b1;
  if (i < TPR_OUT * kHid) { const int o = i / kHid, j = i - o * kHid; w2[i] = gd[kW2tOff + j * kOutPad + o] * g_w2; }
  if (i < TPR_OUT) b2[i] = gd[kB2Off + i] * g_b2;
}

}  // namespace bwd

// ---------------------------------------------------------------------------------------------------------
// launchers (called from the C ABI in triplane_b200.cu); each returns a cudaError_t
// ---------------------------------------------------------------------------------------------------------
int launch_bwd_points(const float* origins, const float* dirs, const float* dc, const float* df, int Dc, int Df,
                      long long n_rays_total, float* pts, int sms, cudaStream_t st) {
  const long long total = n_rays_total * (Dc + Df);
  long long blocks = (total + 255) / 256;
  if (blocks > (long long)sms * 32) blocks = (long long)sms * 32;
  bwd::points_kernel<<<(unsigned)blocks, 256, 0, st>>>(origins, dirs, dc, df, Dc, Df, n_rays_total, pts);
  return (int)cudaGetLastError();
}

int launch_bwd_march(const float* dc, const float* df, int Dc, int Df, const float* sigma, const float* colours, int col_chunked,
                     const float* g_rgb, const float* g_depth, const float* g_wsum, const float* range, int white_back,
                     long long n_rays_total, float* gsig, float* omega, int sms, cudaStream_t st) {
  bwd::MarchArgs a;
  a.dc = dc; a.df = df; a.Dc = Dc; a.Df = Df; a.sigma = sigma; a.colours = colours; a.chunked = col_chunked; a.g_rgb = g_rgb; a.g_depth = g_depth;
  a.g_wsum = g_wsum; a.range = range; a.white_back = white_back; a.n_rays = n_rays_total; a.gsig = gsig; a.omega = omega;
  const int S = Dc + Df;
  const size_t smem = (size_t)4 * (7 * S + 32) * sizeof(float);
  long long blocks = (n_rays_total + 3) / 4;
  if (blocks > (long long)sms * 16) blocks = (long long)sms * 16;
  const int E = (S + 31) / 32;
  if (E <= 1) bwd::march_backward_kernel<1><<<(unsigned)blocks, 128, smem, st>>>(a);
  else if (E <= 2) bwd::march_backward_kernel<2><<<(unsigned)blocks, 128, smem, st>>>(a);
  else if (E <= 3) bwd::march_backward_kernel<3><<<(unsigned)blocks, 128, smem, st>>>(a);
  else if (E <= 4) bwd::march_backward_kernel<4><<<(unsigned)blocks, 128, smem, st>>>(a);
  else if (E <= 6) bwd::march_backward_kernel<6><<<(unsigned)blocks, 128, smem, st>>>(a);
  else bwd::march_backward_kernel<8><<<(unsigned)blocks, 128, smem, st>>>(a);
  return (int)cudaGetLastError();
}

// point != 0: point queries (see decode_backward_kernel); det != NULL: the deterministic mode, as in launch_bwd_decode_tc
// (the caller has run launch_det_bound)
int launch_bwd_decode(const float* planes, int H, int W, const float* dec, const float* pts, const float* colours, int col_chunked,
                      const float* features, const float* gsig, const float* omega, const float* g_rgb, long long total, long long pts_per_img, int S,
                      int point, float box_scale, float* g_planes, float* g_dec, int fast, int skip, DetScratch* det, int sms, cudaStream_t st) {
  bwd::DetDecArgs a;
  a.planes = planes; a.H = H; a.W = W; a.dec = dec; a.pts = pts; a.colours = colours; a.col_chunked = col_chunked; a.features = features; a.gsig = gsig; a.omega = omega;
  a.g_rgb = g_rgb; a.total = total; a.pts_per_img = pts_per_img; a.S = S; a.box_scale = box_scale; a.g_planes = g_planes;
  a.g_dec = g_dec;
  a.g_acc = det ? det->acc : nullptr; a.dec_rows = det ? det->rows : nullptr; a.det_hdr = det ? det->hdr : nullptr;
  { const char* e = getenv("TPR_BWD_DEBUG"); a.debug = skip | (e ? atoi(e) : 0); }
  const size_t smem = sizeof(bwd::Smem) + 16;
  using bwd::DecArgs; using bwd::DetDecArgs;
  void (*kern)(const DecArgs) = point ? (fast ? bwd::decode_backward_kernel<true, true> : bwd::decode_backward_kernel<false, true>)
                                      : (fast ? bwd::decode_backward_kernel<true, false> : bwd::decode_backward_kernel<false, false>);
  void (*kern_det)(const DetDecArgs) =
      point ? (fast ? bwd::decode_backward_kernel<true, true, true, DetDecArgs> : bwd::decode_backward_kernel<false, true, true, DetDecArgs>)
            : (fast ? bwd::decode_backward_kernel<true, false, true, DetDecArgs> : bwd::decode_backward_kernel<false, false, true, DetDecArgs>);
  cudaError_t e = det ? cudaFuncSetAttribute(kern_det, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                      : cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  const long long n_tiles = (total + bwd::kT - 1) / bwd::kT;
  long long grid = n_tiles < 2 * sms ? n_tiles : 2 * sms;      // two CTAs per SM
  if (det) {
    if (grid > kDetMaxRows) grid = kDetMaxRows;
    det->n_rows = (int)grid;
    if (!(skip & 2) && (e = cudaMemsetAsync(det->rows, 0, (size_t)grid * kDecFloats * sizeof(float), st)) != cudaSuccess) return (int)e;
    kern_det<<<(unsigned)grid, bwd::kBT, smem, st>>>(a);
    return (int)cudaGetLastError();
  }
  kern<<<(unsigned)grid, bwd::kBT, smem, st>>>(a);
  return (int)cudaGetLastError();
}

// deterministic mode: the outputs from det (either output may be NULL)
int launch_det_finish(const DetScratch* det, long long n_plane_floats, float* g_planes, float* g_dec, int sms, cudaStream_t st) {
  if (g_planes) {
    const long long n4 = n_plane_floats / 4;
    long long blocks = (n4 + 255) / 256;
    if (blocks > (long long)sms * 16) blocks = (long long)sms * 16;
    bwd::det_planes_kernel<<<(unsigned)blocks, 256, 0, st>>>(reinterpret_cast<const long long*>(det->acc), n4, det->hdr, g_planes);
  }
  if (g_dec) bwd::det_rows_kernel<<<(kDecFloats + 255) / 256, 256, 0, st>>>(det->rows, det->n_rows, g_dec);
  return (int)cudaGetLastError();
}

int launch_unpack_decoder_grad(const float* gd, float g_w1, float g_b1, float g_w2, float g_b2, float* w1, float* b1, float* w2,
                               float* b2, cudaStream_t st) {
  bwd::unpack_decoder_grad_kernel<<<(TPR_OUT * kHid + 255) / 256, 256, 0, st>>>(gd, g_w1, g_b1, g_w2, g_b2, w1, b1, w2, b2);
  return (int)cudaGetLastError();
}

}  // namespace tpr
