// libtriplane_b200.so -- kernels + C ABI (include/triplane_b200.h).
//
// Reference citations are relative to /root/reference/g_nerf/ (VR/ = training/volumetric_rendering/).
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>
#include <mutex>
#include <string>
#include <vector>

#include "triplane_b200.h"
#include "tpr_device.cuh"
#include "tpr_render.cuh"
#include "tpr_host.h"

namespace tpr {

// warp-specialised tensor-core render path (tpr_render_ws.cu)
int ws_rays_per_group(int Dc, int Df, int mode);
bool ws_keeps_samples(int Dc, int Df);
int launch_render_ws(RenderArgs a, int mode, int sms, int smem_optin, long long n_img, long long n_rays, cudaStream_t st);
// tpr_run_model_ws.cu
int launch_run_model_ws(const float* planes, long long n_img, long long plane_sets, int H, int W, const float* dec, const float* xyz,
                        long long n_pts, float box_scale, float* rgb, float* sigma, int mode, int sms, int smem_optin, cudaStream_t st);

// tpr_backward.cu
int launch_bwd_points(const float* origins, const float* dirs, const float* dc, const float* df, int Dc, int Df,
                      long long n_rays_total, float* pts, int sms, cudaStream_t st);
int launch_bwd_march(const float* dc, const float* df, int Dc, int Df, const float* sigma, const float* colours, int col_chunked,
                     const float* g_rgb, const float* g_depth, const float* g_wsum, const float* range, long long group_rays,
                     int white_back, long long n_rays_total, float* gsig, float* omega, int sms, cudaStream_t st);
int launch_bwd_decode(const float* planes, int H, int W, const float* dec, const float* pts, const float* colours, int col_chunked,
                      const float* features, const float* gsig, const float* omega, const float* g_rgb, long long total, long long pts_per_img,
                      int n_sets, int S, int point, float box_scale, float* g_planes, float* g_dec, int fast, int skip, DetScratch* det, int sms,
                      cudaStream_t st);
int launch_det_finish(const DetScratch* det, long long n_plane_floats, float* g_planes, float* g_dec, int sms, cudaStream_t st);
// tpr_backward_tc.cu: the decoder backward on tcgen05 (returns -1 if it cannot run here)
int launch_bwd_decode_tc(const float* planes, int H, int W, const float* dec, const float* pts, const float* colours, int col_chunked,
                         const float* features, const float* gsig, const float* omega, const float* g_rgb, long long total,
                         long long pts_per_img, int n_sets, int S, int point, float box_scale, float* g_planes, float* g_dec,
                         float* scale_buf, DetScratch* det, int sms, int smem_optin, cudaStream_t st);
int launch_det_bound(const float* dec, const float* gsig, const float* g_rgb, long long total, int n_sets, int S, int point,
                     float* scale_buf, DetScratch* det, int sms, cudaStream_t st);
int launch_unpack_decoder_grad(const float* gd, float g_w1, float g_b1, float g_w2, float g_b2, float* w1, float* b1, float* w2,
                               float* b2, cudaStream_t st);

// =======================================================================================
// layout preparation
// =======================================================================================
// [P][32][HW] -> [P][HW][32]; one CTA transposes a 32-channel x 32-pixel tile through smem.
__global__ void __launch_bounds__(256) pack_planes_kernel(const float* __restrict__ src, float* __restrict__ dst,
                                                          int hw, int tiles_per_plane) {
  __shared__ float tile[32][33];
  const int plane = blockIdx.x / tiles_per_plane;
  const int p0 = (blockIdx.x - plane * tiles_per_plane) * 32;
  const float* s = src + (size_t)plane * kC * hw;
  float* d = dst + (size_t)plane * kC * hw;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 8 rows of 32
#pragma unroll
  for (int c = ty; c < 32; c += 8) {
    int p = p0 + tx;
    tile[c][tx] = p < hw ? s[(size_t)c * hw + p] : 0.0f;
  }
  __syncthreads();
#pragma unroll
  for (int pp = ty; pp < 32; pp += 8) {
    int p = p0 + pp;
    if (p < hw) d[(size_t)p * kC + tx] = tile[tx][pp];
  }
}

// [P][HW][32] -> [P][32][HW]: the adjoint (plane gradients back to the backbone's layout)
__global__ void __launch_bounds__(256) unpack_planes_kernel(const float* __restrict__ src, float* __restrict__ dst,
                                                            int hw, int tiles_per_plane) {
  __shared__ float tile[32][33];
  const int plane = blockIdx.x / tiles_per_plane;
  const int p0 = (blockIdx.x - plane * tiles_per_plane) * 32;
  const float* s = src + (size_t)plane * kC * hw;
  float* d = dst + (size_t)plane * kC * hw;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
  for (int pp = ty; pp < 32; pp += 8) {
    const int p = p0 + pp;
    tile[pp][tx] = p < hw ? s[(size_t)p * kC + tx] : 0.0f;
  }
  __syncthreads();
#pragma unroll
  for (int c = ty; c < 32; c += 8) {
    const int p = p0 + tx;
    if (p < hw) d[(size_t)c * hw + p] = tile[tx][c];
  }
}

__global__ void pack_decoder_kernel(const float* __restrict__ w1, const float* __restrict__ b1,
                                    const float* __restrict__ w2, const float* __restrict__ b2,
                                    float g_w1, float g_b1, float g_w2, float g_b2, float* __restrict__ out) {
  for (int i = threadIdx.x + blockIdx.x * blockDim.x; i < kDecFloats; i += blockDim.x * gridDim.x) {
    float v;
    if (i < kB1Off) {                       // W1t[k][j] = W1[j][k] * gain / 3
      int k = i / kHid, j = i - k * kHid;
      v = __fmul_rn(w1[j * kC + k], g_w1) * (1.0f / 3.0f);
    } else if (i < kW2tOff) {
      v = b1[i - kB1Off] * g_b1;
    } else if (i < kB2Off) {                // W2t[j][o] = W2[o][j] * gain
      int r = i - kW2tOff;
      int j = r / kOutPad, o = r - j * kOutPad;
      v = o < TPR_OUT ? w2[o * kHid + j] * g_w2 : 0.0f;
    } else {
      int o = i - kB2Off;
      v = o < TPR_OUT ? b2[o] * g_b2 : 0.0f;
    }
    out[i] = v;
  }
}

// =======================================================================================
// a1: RaySampler.forward (VR/ray_sampler.py:36-61), one thread per ray
// =======================================================================================
__global__ void ray_sample_kernel(const float* __restrict__ c2w, const float* __restrict__ K, int res, long long total,
                                  float* __restrict__ origins, float* __restrict__ dirs) {
  const long long m_per = (long long)res * res;
  for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < total; g += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(g / m_per);
    const int m = (int)(g - n * m_per);
    const int py = m / res, pxi = m - py * res;       // x fastest (:44)
    const float* A = c2w + n * 16;
    const float* k = K + n * 9;
    const float fx = k[0], sk = k[1], cx = k[2], fy = k[4], cy = k[5];
    const float inv = 1.0f / (float)res, half = 0.5f / (float)res;
    const float xc = __fadd_rn(__fmul_rn((float)pxi, inv), half);
    const float yc = __fadd_rn(__fmul_rn((float)py, inv), half);
    // (x - cx + cy*sk/fy - sk*y/fy) / fx   and   (y - cy) / fy    (:51-52)
    float xl = __fsub_rn(__fadd_rn(__fsub_rn(xc, cx), __fdiv_rn(__fmul_rn(cy, sk), fy)), __fdiv_rn(__fmul_rn(sk, yc), fy));
    xl = __fdiv_rn(xl, fx);
    const float yl = __fdiv_rn(__fsub_rn(yc, cy), fy);
    float d[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      float acc = __fmul_rn(A[i * 4 + 0], xl);
      acc = __fadd_rn(acc, __fmul_rn(A[i * 4 + 1], yl));
      acc = __fadd_rn(acc, A[i * 4 + 2]);
      acc = __fadd_rn(acc, A[i * 4 + 3]);
      d[i] = __fsub_rn(acc, A[i * 4 + 3]);            // minus camera position (:58)
    }
    float nrm = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(d[0], d[0]), __fmul_rn(d[1], d[1])), __fmul_rn(d[2], d[2])));
    nrm = fmaxf(nrm, 1e-12f);                          // F.normalize eps (:59)
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      dirs[g * 3 + i] = __fdiv_rn(d[i], nrm);
      origins[g * 3 + i] = A[i * 4 + 3];
    }
  }
}

// =======================================================================================
// a7 stand-alone: sample_stratified (VR/renderer.py:169-192), one thread per depth
// =======================================================================================
__global__ void sample_stratified_kernel(const RenderArgs a, long long total, float* __restrict__ depths) {
  const bool per_ray = a.rs != nullptr;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long g = i / a.Dc;
    const int k = (int)(i - g * a.Dc);
    depths[i] = coarse_depth(a, k, a.jitter[i], per_ray ? a.rs[g] : a.ray_start, per_ray ? a.re[g] : a.ray_end, per_ray);
  }
}

// =======================================================================================
// a14: get_ray_limits_box (VR/math_utils.py:46-98), one thread per ray
// =======================================================================================
__global__ void ray_limits_box_kernel(const float* __restrict__ o, const float* __restrict__ d, long long n, float side,
                                      float* __restrict__ tmin_out, float* __restrict__ tmax_out) {
  for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < n; g += (long long)gridDim.x * blockDim.x) {
    const float lo = -0.5f * side, hi = 0.5f * side;
    float inv[3], org[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) { org[i] = o[g * 3 + i]; inv[i] = __fdiv_rn(1.0f, d[g * 3 + i]); }
    bool valid = true;
    // slab test in the reference's order: x, then y, then z
    float tmin = __fmul_rn(__fsub_rn(inv[0] < 0 ? hi : lo, org[0]), inv[0]);
    float tmax = __fmul_rn(__fsub_rn(inv[0] < 0 ? lo : hi, org[0]), inv[0]);
    float tymin = __fmul_rn(__fsub_rn(inv[1] < 0 ? hi : lo, org[1]), inv[1]);
    float tymax = __fmul_rn(__fsub_rn(inv[1] < 0 ? lo : hi, org[1]), inv[1]);
    if (tmin > tymax || tymin > tmax) valid = false;
    tmin = fmaxf(tmin, tymin); tmax = fminf(tmax, tymax);
    float tzmin = __fmul_rn(__fsub_rn(inv[2] < 0 ? hi : lo, org[2]), inv[2]);
    float tzmax = __fmul_rn(__fsub_rn(inv[2] < 0 ? lo : hi, org[2]), inv[2]);
    if (tmin > tzmax || tzmin > tmax) valid = false;
    tmin = fmaxf(tmin, tzmin); tmax = fminf(tmax, tzmax);
    tmin_out[g] = valid ? tmin : -1.0f;
    tmax_out[g] = valid ? tmax : -2.0f;
  }
}

// =======================================================================================
// a8 / a5: run_model and the stand-alone decoder.  Each warp owns a private 32-row tile.
// =======================================================================================
constexpr int kRmThreads = 256;
constexpr int kRmWarps = kRmThreads / 32;

template <bool kFromFeatures>
__global__ void __launch_bounds__(kRmThreads) run_model_kernel(
    const float* __restrict__ planes, int H, int W, const float* __restrict__ dec,
    const float* __restrict__ in /* xyz [N,P,3] or features [N,3,P,32] */, long long n_img, long long n_pts,
    float box_scale, float* __restrict__ rgb, float* __restrict__ sigma, long long plane_sets /* image n reads set n % plane_sets */) {
  extern __shared__ __align__(16) float smem[];
  float* wsm = smem;
  float* rows = smem + kDecFloats + (threadIdx.x >> 5) * 32 * kC;
  stage_decoder(dec, wsm);
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const long long chunks_per_img = (n_pts + 31) >> 5;       // a chunk never straddles two images
  const long long n_chunks = n_img * chunks_per_img;
  const size_t img_stride = (size_t)3 * H * W * kC;
  for (long long chunk = blockIdx.x * (long long)kRmWarps + (threadIdx.x >> 5); chunk < n_chunks;
       chunk += (long long)gridDim.x * kRmWarps) {
    const long long n = chunk / chunks_per_img;
    const long long p0 = (chunk - n * chunks_per_img) * 32;
    const int nvalid = (int)min(32LL, n_pts - p0);
    const bool valid = lane < nvalid;
    const long long g = n * n_pts + p0 + lane;
    if (!kFromFeatures) {
      float px = 0.f, py = 0.f, pz = 0.f;
      if (valid) {
        px = __fmul_rn(in[g * 3 + 0], box_scale);       // (2/box_warp) * coordinates (VR/renderer.py:61)
        py = __fmul_rn(in[g * 3 + 1], box_scale);
        pz = __fmul_rn(in[g * 3 + 2], box_scale);
      }
      gather_chunk(planes + (size_t)(n % plane_sets) * img_stride, H, W, px, py, pz, lane, valid, rows, lane);
    } else {
      // features [N,3,P,32]: sum the three planes' rows, eight lanes per sample
      const int grp = lane >> 3, sub = lane & 7;
#pragma unroll 2
      for (int q = 0; q < 8; ++q) {
        const int r = q * 4 + grp;
        if (r < nvalid) {
          const float* f0 = in + (n * 3 * n_pts + p0 + r) * kC + sub * 4;
          float4 a = ldg128(f0), b = ldg128(f0 + n_pts * kC), c = ldg128(f0 + 2 * n_pts * kC);
          *reinterpret_cast<float4*>(rows + row_chunk_off(r, sub)) =
              make_float4(a.x + b.x + c.x, a.y + b.y + c.y, a.z + b.z + c.z, a.w + b.w + c.w);
        }
      }
    }
    __syncwarp();
    float sg = 0.f;
    if (valid) sg = decode_row_inplace(wsm, rows, lane);
    __syncwarp();
    if (valid) sigma[g] = sg;
    if (rgb != nullptr) {
      // the 32 rows of this chunk are contiguous in rgb[N,P,32]: store them fully coalesced
      float4* dst = reinterpret_cast<float4*>(rgb + (n * n_pts + p0) * kC);
#pragma unroll
      for (int it = 0; it < 8; ++it) {
        const int f = it * 32 + lane, r = f >> 3, c = f & 7;
        if (r < nvalid) dst[f] = *reinterpret_cast<const float4*>(rows + row_chunk_off(r, c));
      }
    }
    __syncwarp();
  }
}

// =======================================================================================
// a13: the fused ImportanceRenderer.forward.  One persistent CTA per SM slot walks tiles of R
// rays.  Per tile:   A  coarse depths -> gather -> decoder          (warp per 32 samples)
//                    B  coarse march -> smoothed pdf -> CDF -> fine depths   (warp per ray)
//                    C  gather -> decoder for the fine samples      (warp per 32 samples)
//                    D  sort 2D samples, final march, colour sum    (warp per ray)
// Per-sample features and colours live only in shared memory (one 128-byte row per sample).
// =======================================================================================
struct TileSmem {
  float* wsm;     // packed decoder
  float* col;     // [R*S][32]  features, then colours
  float* dep;     // [R*S]
  float* sig;     // [R*S]
  float* wa;      // [R*S]  coarse weights        | omega (phase D)
  float* wb;      // [R*S]  pdf weights           | sorted index (phase D, as int)
  float* wc;      // [R*S]  cdf
  float* ray;     // [R][8]: origin xyz, dir xyz, start, end
};

// gather + decode `n_samp` = nr*Dx samples of the tile; sample s -> ray s/Dx, slot off + s%Dx
__device__ __forceinline__ void tile_pass(const RenderArgs& a, const TileSmem& sm, const float* __restrict__ img,
                                          int nr, int Dx, int off, int S) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int n_samp = nr * Dx;
  for (int c0 = warp * 32; c0 < n_samp; c0 += nwarps * 32) {
    const int s = c0 + lane;
    const bool valid = s < n_samp;
    int row = 0; float px = 0.f, py = 0.f, pz = 0.f;
    if (valid) {
      const int r = s / Dx;
      row = r * S + off + (s - r * Dx);
      const float d = sm.dep[row];
      const float* ry = sm.ray + r * 8;
      // origin + depth * direction (VR/renderer.py:105,123), then * 2/box_warp (:61)
      px = __fmul_rn(__fadd_rn(ry[0], __fmul_rn(d, ry[3])), a.box_scale);
      py = __fmul_rn(__fadd_rn(ry[1], __fmul_rn(d, ry[4])), a.box_scale);
      pz = __fmul_rn(__fadd_rn(ry[2], __fmul_rn(d, ry[5])), a.box_scale);
    }
    gather_chunk(img, a.H, a.W, px, py, pz, row, valid, sm.col, lane);
    __syncwarp();
    if (valid) sm.sig[row] = decode_row_inplace(sm.wsm, sm.col, row);
  }
}

template <int E>
__device__ __forceinline__ void ray_composite(const RenderArgs& a, const TileSmem& sm, int r, long long g, int n, int S,
                                              float& mn, float& mx) {
  const int lane = threadIdx.x & 31;
  float* om = sm.wa + r * S;
  int* oi = reinterpret_cast<int*>(sm.wb + r * S);
  float wsum, dnum;
  warp_sort_and_weights<E, false>(sm.dep + r * S, sm.sig + r * S, om, oi, S, lane, wsum, dnum, mn, mx);
  __syncwarp();
  // colour sum: lane = channel
  const int rowbase = r * S;
  float acc0 = 0.f, acc1 = 0.f;
  int p = 0;
  for (; p + 1 < S; p += 2) {
    const int r0 = rowbase + oi[p], r1 = rowbase + oi[p + 1];
    acc0 = fmaf(om[p], sm.col[r0 * kC + ((((lane >> 2) ^ (r0 & 7)) << 2) | (lane & 3))], acc0);
    acc1 = fmaf(om[p + 1], sm.col[r1 * kC + ((((lane >> 2) ^ (r1 & 7)) << 2) | (lane & 3))], acc1);
  }
  if (p < S) {
    const int r0 = rowbase + oi[p];
    acc0 = fmaf(om[p], sm.col[r0 * kC + ((((lane >> 2) ^ (r0 & 7)) << 2) | (lane & 3))], acc0);
  }
  float c = acc0 + acc1;
  if (a.white_back) c = c + 1.0f - wsum;              // VR/ray_marcher.py:52-53
  long long cstride;
  float* px = rgb_ptr(a, g, n, cstride);
  px[lane * cstride] = c * 2.0f - 1.0f;                              // :55
  if (lane == 0) {
    a.depth[g] = dnum / wsum;                         // NaN -> inf and the clamp happen in finish_kernel
    a.wsum[g] = wsum;
  }
}

template <int E>   // sort width: 32*E >= Dc + Df
__global__ void __launch_bounds__(kRenderMaxThreads, 1) render_kernel(const RenderArgs a) {
  extern __shared__ __align__(16) float smem[];
  const int R = a.R, Dc = a.Dc, Df = a.Df, S = Dc + Df;
  TileSmem sm;
  sm.wsm = smem;
  sm.col = sm.wsm + kDecFloats;
  sm.dep = sm.col + (size_t)R * S * kC;
  sm.sig = sm.dep + R * S;
  sm.wa = sm.sig + R * S;
  sm.wb = sm.wa + R * S;
  sm.wc = sm.wb + R * S;
  sm.ray = sm.wc + R * S;
  __shared__ unsigned range_sm[2];
  if (threadIdx.x == 0) { range_sm[0] = 0xffffffffu; range_sm[1] = 0u; }
  stage_decoder(a.dec, sm.wsm);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const bool per_ray = a.rs != nullptr;
  const size_t img_stride = (size_t)3 * a.H * a.W * kC;
  float mn = __int_as_float(0x7f800000), mx = -__int_as_float(0x7f800000);
  float smn = mn, smx = mx;                           // running depth range of the current clamp slot
  int cur_slot = 0;

  for (long long tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    // a tile is R consecutive rays of ONE image, so the plane block is CTA-uniform
    const long long n = tile / a.tiles_per_img;
    const long long m0 = (tile - n * a.tiles_per_img) * R;
    const long long g0 = n * a.rays_per_img + m0;
    const int nr = (int)min((long long)R, a.rays_per_img - m0);
    const float* img = a.planes + (size_t)(n % a.plane_sets) * img_stride;
    if (range_slot(a, (int)n) != cur_slot) { range_fold(a, cur_slot, smn, smx, mn, mx, lane); cur_slot = range_slot(a, (int)n); }
    __syncthreads();                                   // previous tile fully consumed
    // ---- rays
    if (threadIdx.x < nr * 6) {
      const int r = threadIdx.x / 6, c = threadIdx.x - r * 6;
      const long long g = g0 + r;
      sm.ray[r * 8 + c] = c < 3 ? a.origins[g * 3 + c] : a.dirs[g * 3 + c - 3];
      if (c == 0) {
        sm.ray[r * 8 + 6] = per_ray ? a.rs[g] : a.ray_start;
        sm.ray[r * 8 + 7] = per_ray ? a.re[g] : a.ray_end;
      }
    }
    __syncthreads();
    // ---- coarse depths (the jitter block of a tile is contiguous in HBM)
    for (int s = threadIdx.x; s < nr * Dc; s += blockDim.x) {
      const int r = s / Dc, k = s - r * Dc;
      const float jit = __ldg(a.jitter + g0 * Dc + s);
      sm.dep[r * S + k] = coarse_depth(a, k, jit, sm.ray[r * 8 + 6], sm.ray[r * 8 + 7], per_ray);
    }
    __syncthreads();
    const int n_pass = Df > 0 ? 2 : 1;
#pragma unroll 1
    for (int pass = 0; pass < n_pass; ++pass) {
      if (pass == 1) {
        // ---- B: importance resampling, one warp per ray
        for (int r = warp; r < nr; r += nwarps)
          warp_resample_ray(a, sm.dep + r * S, sm.sig + r * S, sm.wa + r * S, sm.wb + r * S, sm.wc + r * S,
                            sm.dep + r * S + Dc, g0 + r, lane, a.u + (g0 + r) * Df);
        __syncthreads();
      }
      // ---- A / C: gather + decode the coarse (pass 0) or fine (pass 1) samples
      tile_pass(a, sm, img, nr, pass == 0 ? Dc : Df, pass == 0 ? 0 : Dc, S);
      __syncthreads();
      if (a.noise_c != nullptr) {     // density_noise (VR/renderer.py:146)
        if (pass == 0) add_density_noise(a, a.noise_c, sm.sig, S, 0, Dc, nr * Dc, g0, 1, threadIdx.x, blockDim.x);
        else add_density_noise(a, a.noise_f, sm.sig, S, Dc, Df, nr * Df, g0, 1, threadIdx.x, blockDim.x);
        __syncthreads();
      }
    }
    // ---- D: merge + final march
    for (int r = warp; r < nr; r += nwarps) ray_composite<E>(a, sm, r, g0 + r, (int)n, S, smn, smx);
  }
  range_fold(a, cur_slot, smn, smx, mn, mx, lane);
  mn = warp_min(mn); mx = warp_max(mx);
  if (lane == 0 && mn <= mx) {
    atomicMin(&range_sm[0], float_to_ordered(mn));
    atomicMax(&range_sm[1], float_to_ordered(mx));
  }
  __syncthreads();
  if (threadIdx.x == 0 && range_sm[0] <= range_sm[1]) {
    atomicMin(a.range_enc + 0, range_sm[0]);
    atomicMax(a.range_enc + 1, range_sm[1]);
  }
}

// n_slots < 0: `enc` is just the two range words (tpr_ray_march); otherwise the render scratch block
__global__ void range_init_kernel(unsigned* enc, int n_slots) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    enc[0] = 0xffffffffu; enc[1] = 0u;
    if (n_slots >= 0)
      for (int i = 0; i < 16; ++i) reinterpret_cast<long long*>(reinterpret_cast<char*>(enc) + 64)[i] = 0;   // phase counters
  }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_slots; i += gridDim.x * blockDim.x) {
    enc[kRangeSlotOff + 2 * i] = 0xffffffffu; enc[kRangeSlotOff + 2 * i + 1] = 0u;
  }
}

// decode the (min,max) and optionally apply nan_to_num(inf) + clamp (VR/ray_marcher.py:49-50)
// rays_per_slot > 0: ray i clamps against the range of slot i / rays_per_slot instead of the call-wide one
__global__ void finish_kernel(const unsigned* __restrict__ enc, float* __restrict__ range_out,
                              float* __restrict__ depth, long long n, int do_clamp, long long rays_per_slot) {
  const float glo = ordered_to_float(enc[0]), ghi = ordered_to_float(enc[1]);
  if (blockIdx.x == 0 && threadIdx.x == 0 && range_out) { range_out[0] = glo; range_out[1] = ghi; }
  if (!do_clamp) return;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float lo = glo, hi = ghi;
    if (rays_per_slot > 0) {
      const long long s = i / rays_per_slot;
      lo = ordered_to_float(enc[kRangeSlotOff + 2 * s]); hi = ordered_to_float(enc[kRangeSlotOff + 2 * s + 1]);
    }
    float d = depth[i];
    if (d != d) d = __int_as_float(0x7f800000);
    depth[i] = fminf(fmaxf(d, lo), hi);
  }
}

__global__ void clamp_depth_kernel(float* __restrict__ depth, long long n, const float* __restrict__ range) {
  const float lo = range[0], hi = range[1];
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float d = depth[i];
    if (d != d) d = __int_as_float(0x7f800000);
    depth[i] = fminf(fmaxf(d, lo), hi);
  }
}

// copy one GPU's rendered outputs into the peers' gather buffers (plain stores through peer-mapped pointers)
__global__ void peer_scatter_kernel(const PeerSinks peers, const float* __restrict__ rgb, const float* __restrict__ depth,
                                    const float* __restrict__ wsum, long long n_rays) {
  const long long n4 = n_rays * (kC / 4);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(rgb)[i];
    for (int p = 0; p < peers.n; ++p) reinterpret_cast<float4*>(peers.rgb[p])[i] = v;
    if (i < n_rays) {
      const float d = depth[i], w = wsum[i];
      for (int p = 0; p < peers.n; ++p) { peers.depth[p][i] = d; peers.wsum[p][i] = w; }
    }
  }
}

// =======================================================================================
// a9 stand-alone: MipRayMarcher2.forward, one warp per ray, samples in the given order
// =======================================================================================
__global__ void __launch_bounds__(256) ray_march_kernel(const float* __restrict__ colors, const float* __restrict__ dens,
                                                        const float* __restrict__ depths, long long n_rays, int S, int C,
                                                        int white_back, float* __restrict__ rgb, float* __restrict__ depth,
                                                        float* __restrict__ weights, unsigned* __restrict__ range_enc) {
  const int lane = threadIdx.x & 31;
  float mn = __int_as_float(0x7f800000), mx = -mn;
  for (long long g = blockIdx.x * 8LL + (threadIdx.x >> 5); g < n_rays; g += gridDim.x * 8LL) {
    const float* z = depths + g * S;
    const float* sg = dens + g * S;
    float* w = weights + g * (S - 1);
    warp_march_weights(z, sg, w, S, lane);
    __syncwarp();
    float wsum = 0.f, dnum = 0.f;
    for (int i = lane; i < S - 1; i += 32) {
      wsum += w[i];
      dnum = fmaf(w[i], (z[i] + z[i + 1]) * 0.5f, dnum);
    }
    for (int i = lane; i < S; i += 32) { mn = fminf(mn, z[i]); mx = fmaxf(mx, z[i]); }
    wsum = warp_sum(wsum); dnum = warp_sum(dnum);
    const float* col = colors + g * (long long)S * C;
    for (int c = lane; c < C; c += 32) {
      float acc = 0.f;
      for (int i = 0; i < S - 1; ++i) acc = fmaf(w[i], (col[(long long)i * C + c] + col[(long long)(i + 1) * C + c]) * 0.5f, acc);
      if (white_back) acc = acc + 1.0f - wsum;
      rgb[g * C + c] = acc * 2.0f - 1.0f;
    }
    if (lane == 0) depth[g] = dnum / wsum;
  }
  mn = warp_min(mn); mx = warp_max(mx);
  if (lane == 0 && mn <= mx) {
    atomicMin(range_enc + 0, float_to_ordered(mn));
    atomicMax(range_enc + 1, float_to_ordered(mx));
  }
}

// =======================================================================================
// a10/a11 stand-alone, one warp per ray (same device functions as the fused kernel)
// =======================================================================================
constexpr int kPdfWarps = 4;
// mode 0: sample_importance(z_vals [R,S], weights [R,S-1]);  mode 1: sample_pdf(bins, weights [R,nb])
__global__ void __launch_bounds__(kPdfWarps * 32) resample_kernel(
    int mode, const float* __restrict__ zin, int z_stride, const float* __restrict__ win, const float* __restrict__ u,
    long long n_rays, int S_or_nb, int K, float* __restrict__ samples, int* __restrict__ inds_out) {
  extern __shared__ __align__(16) float smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int cap = (mode == 0 ? S_or_nb : S_or_nb + 2);
  float* z = smem + warp * 4 * cap;
  float* w = z + cap; float* pw = w + cap; float* cdf = pw + cap;
  for (long long g = blockIdx.x * (long long)kPdfWarps + warp; g < n_rays; g += (long long)gridDim.x * kPdfWarps) {
    int nb;
    if (mode == 0) {
      const int S = S_or_nb;
      nb = S - 3;
      for (int i = lane; i < S; i += 32) z[i] = zin[g * z_stride + i];
      for (int i = lane; i < S - 1; i += 32) w[i] = win[g * (S - 1) + i];
      __syncwarp();
      warp_smooth_weights(w, pw, nb, lane);
    } else {
      nb = S_or_nb;
      for (int i = lane; i < nb + 1; i += 32) z[i] = zin[g * z_stride + i];
      for (int i = lane; i < nb; i += 32) pw[i] = win[g * nb + i];
    }
    __syncwarp();
    warp_cdf(pw, cdf, nb, lane);
    __syncwarp();
    for (int j = lane; j < K; j += 32) {
      int inds; float smp;
      const float uu = u[g * K + j];
      if (mode == 0) smp = invert_cdf(cdf, nb, uu, [&](int i) { return __fmul_rn(0.5f, __fadd_rn(z[i], z[i + 1])); }, inds);
      else smp = invert_cdf(cdf, nb, uu, [&](int i) { return z[i]; }, inds);
      samples[g * K + j] = smp;
      if (inds_out) inds_out[g * K + j] = inds;
    }
    __syncwarp();
  }
}

// =======================================================================================
// host side
// =======================================================================================
static thread_local std::string g_err;

// (shared with the other translation units through tpr_host.h)
int fail(int code, const char* msg) { g_err = msg; return code; }
int cuda_fail(cudaError_t e, const char* what) {
  g_err = std::string(what) + ": " + cudaGetErrorString(e);
  (void)cudaGetLastError();                 // clear the (non-sticky) error so later calls start clean
  return (int)e > 0 ? (int)e : 999;
}
#define TPR_CHECK_LAUNCH(what)                                   \
  do {                                                           \
    cudaError_t e__ = cudaGetLastError();                        \
    if (e__ != cudaSuccess) return cuda_fail(e__, what);         \
  } while (0)

DeviceInfo device_info() {
  static std::mutex mu;
  static DeviceInfo cache[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return DeviceInfo();
  std::lock_guard<std::mutex> lk(mu);
  if (!cache[dev].ok) {
    cudaDeviceGetAttribute(&cache[dev].sms, cudaDevAttrMultiProcessorCount, dev);
    cudaDeviceGetAttribute(&cache[dev].smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    cache[dev].ok = cache[dev].sms > 0;
  }
  return cache[dev];
}

static int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return v && *v ? atoi(v) : dflt;
}

// Operand scheme of the tcgen05 decoder for a TPR_MLP_* flag (the kernels' MODE): 1 = bf16 operands (the PSNR mode),
// 2 = 2xFP16 (x = hi + lo in fp16, three products: the fp32-grade mode; it replaced 3xTF32, see tpr_ws.cuh).
static int tc_mode(int flags) { return flags == TPR_MLP_BF16 ? 1 : 2; }

int grid_for(long long work_items, int per_block, int sms, int waves) {
  long long blocks = (work_items + per_block - 1) / per_block;
  long long cap = (long long)sms * waves;
  if (blocks > cap) blocks = cap;
  return (int)(blocks < 1 ? 1 : blocks);
}

// shared-memory bytes of render_kernel for R rays of S samples
static size_t render_smem_bytes(int R, int S) {
  return sizeof(float) * ((size_t)kDecFloats + (size_t)R * S * kC + (size_t)5 * R * S + (size_t)R * 8);
}

}  // namespace tpr

using namespace tpr;

extern "C" {

int tpr_abi_version(void) { return TPR_ABI_VERSION; }
const char* tpr_last_error(void) { return g_err.c_str(); }

size_t tpr_packed_planes_bytes(int64_t n_img, int32_t height, int32_t width) {
  if (n_img < 0 || height <= 0 || width <= 0) return 0;
  return (size_t)n_img * TPR_PLANES * TPR_CHANNELS * height * width * sizeof(float);
}

int tpr_pack_planes(const float* planes_nchw, int64_t n_img, int32_t height, int32_t width, float* planes_packed,
                    void* stream) {
  if (!planes_nchw || !planes_packed) return fail(TPR_E_NULL, "tpr_pack_planes: NULL pointer");
  if (n_img <= 0 || height <= 0 || width <= 0 || (int64_t)height * width > (1 << 26))
    return fail(TPR_E_SHAPE, "tpr_pack_planes: bad shape");
  const int hw = height * width;
  const int tiles = (hw + 31) / 32;
  const long long blocks = (long long)n_img * TPR_PLANES * tiles;
  if (blocks > 0x7fffffffLL) return fail(TPR_E_SHAPE, "tpr_pack_planes: too many tiles");
  pack_planes_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(planes_nchw, planes_packed, hw, tiles);
  TPR_CHECK_LAUNCH("pack_planes_kernel");
  return 0;
}

int tpr_unpack_planes(const float* planes_packed, int64_t n_img, int32_t height, int32_t width, float* planes_nchw,
                      void* stream) {
  if (!planes_nchw || !planes_packed) return fail(TPR_E_NULL, "tpr_unpack_planes: NULL pointer");
  if (n_img <= 0 || height <= 0 || width <= 0 || (int64_t)height * width > (1 << 26))
    return fail(TPR_E_SHAPE, "tpr_unpack_planes: bad shape");
  const int hw = height * width;
  const int tiles = (hw + 31) / 32;
  const long long blocks = (long long)n_img * TPR_PLANES * tiles;
  if (blocks > 0x7fffffffLL) return fail(TPR_E_SHAPE, "tpr_unpack_planes: too many tiles");
  unpack_planes_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(planes_packed, planes_nchw, hw, tiles);
  TPR_CHECK_LAUNCH("unpack_planes_kernel");
  return 0;
}

size_t tpr_packed_decoder_bytes(void) { return kDecFloats * sizeof(float); }

int tpr_pack_decoder(const float* w1, const float* b1, const float* w2, const float* b2, float w1_gain, float b1_gain,
                     float w2_gain, float b2_gain, float* decoder_packed, void* stream) {
  if (!w1 || !b1 || !w2 || !b2 || !decoder_packed) return fail(TPR_E_NULL, "tpr_pack_decoder: NULL pointer");
  pack_decoder_kernel<<<5, 256, 0, (cudaStream_t)stream>>>(w1, b1, w2, b2, w1_gain, b1_gain, w2_gain, b2_gain,
                                                           decoder_packed);
  TPR_CHECK_LAUNCH("pack_decoder_kernel");
  return 0;
}

int tpr_ray_sample(const float* cam2world, const float* intrinsics, int64_t n_img, int32_t resolution, float* origins,
                   float* dirs, void* stream) {
  if (!cam2world || !intrinsics || !origins || !dirs) return fail(TPR_E_NULL, "tpr_ray_sample: NULL pointer");
  if (n_img <= 0 || resolution <= 0 || resolution > 16384) return fail(TPR_E_SHAPE, "tpr_ray_sample: bad shape");
  DeviceInfo di = device_info();
  if (!di.ok) return fail(TPR_E_DEVICE, "tpr_ray_sample: no CUDA device");
  const long long total = (long long)n_img * resolution * resolution;
  ray_sample_kernel<<<grid_for(total, 256, di.sms, 16), 256, 0, (cudaStream_t)stream>>>(cam2world, intrinsics, resolution,
                                                                                       total, origins, dirs);
  TPR_CHECK_LAUNCH("ray_sample_kernel");
  return 0;
}

int tpr_ray_limits_box(const float* origins, const float* dirs, int64_t n_rays, float box_side_length, float* t_min,
                       float* t_max, void* stream) {
  if (!origins || !dirs || !t_min || !t_max) return fail(TPR_E_NULL, "tpr_ray_limits_box: NULL pointer");
  if (n_rays <= 0) return fail(TPR_E_SHAPE, "tpr_ray_limits_box: n_rays <= 0");
  DeviceInfo di = device_info();
  if (!di.ok) return fail(TPR_E_DEVICE, "tpr_ray_limits_box: no CUDA device");
  ray_limits_box_kernel<<<grid_for(n_rays, 256, di.sms, 16), 256, 0, (cudaStream_t)stream>>>(origins, dirs, n_rays,
                                                                                            box_side_length, t_min, t_max);
  TPR_CHECK_LAUNCH("ray_limits_box_kernel");
  return 0;
}

// the depth-sampling constants of RenderArgs, derived exactly as torch derives them from the python floats
static void set_depth_constants(RenderArgs& a, const TprOptions* opt) {
  const int Dc = opt->depth_resolution;
  a.ray_start = (float)opt->ray_start; a.ray_end = (float)opt->ray_end;                 // torch.linspace casts to float32
  a.lin_step = (a.ray_end - a.ray_start) / (float)(Dc - 1);                             // torch.linspace step, float32
  a.jitter_scale = (float)((opt->ray_end - opt->ray_start) / (Dc - 1));                 // python float (VR/renderer.py:189)
  a.inv_start = (float)(1.0 / opt->ray_start); a.inv_end = (float)(1.0 / opt->ray_end); // python floats (:181)
  a.Dc = Dc; a.disparity = opt->disparity_space_sampling;
}

int tpr_sample_stratified(const float* jitter, int64_t n_rays, const float* ray_start_per_ray, const float* ray_end_per_ray,
                          const TprOptions* opt, float* depths, void* stream) {
  if (!jitter || !opt || !depths) return fail(TPR_E_NULL, "tpr_sample_stratified: NULL pointer");
  if ((ray_start_per_ray == nullptr) != (ray_end_per_ray == nullptr))
    return fail(TPR_E_NULL, "tpr_sample_stratified: per-ray limits need both start and end");
  if (n_rays <= 0 || opt->depth_resolution < 2) return fail(TPR_E_SHAPE, "tpr_sample_stratified: need n_rays > 0, depth_resolution >= 2");
  DeviceInfo di = device_info();
  if (!di.ok) return fail(TPR_E_DEVICE, "tpr_sample_stratified: no CUDA device");
  RenderArgs a;
  memset(&a, 0, sizeof(a));
  set_depth_constants(a, opt);
  a.jitter = jitter; a.rs = ray_start_per_ray; a.re = ray_end_per_ray;
  const long long total = (long long)n_rays * opt->depth_resolution;
  sample_stratified_kernel<<<grid_for(total, 256, di.sms, 16), 256, 0, (cudaStream_t)stream>>>(a, total, depths);
  TPR_CHECK_LAUNCH("sample_stratified_kernel");
  return 0;
}

// plane_sets: image n reads plane set n % plane_sets (tpr_run_model: plane_sets = n_img; the render backward re-evaluates
// frame-batched samples with the forward's plane_sets)
static int launch_run_model(bool from_features, const float* planes, int64_t n_img, int64_t plane_sets, int32_t H, int32_t W,
                            const float* dec, const float* in, int64_t n_pts, double box_warp, float* rgb, float* sigma,
                            int32_t flags, void* stream) {
  if (!dec || !in || !sigma) return fail(TPR_E_NULL, "run_model: NULL pointer");
  if (!from_features && !planes) return fail(TPR_E_NULL, "run_model: NULL planes");
  if (n_img <= 0 || n_pts <= 0) return fail(TPR_E_SHAPE, "run_model: empty input");
  if (!from_features && (H <= 0 || W <= 0 || (int64_t)H * W > (1 << 24))) return fail(TPR_E_SHAPE, "run_model: bad plane size");
  if (!from_features && !(box_warp > 0.0)) return fail(TPR_E_OPTION, "run_model: box_warp must be > 0");
  if (flags != TPR_MLP_FP32 && flags != TPR_MLP_BF16 && flags != TPR_MLP_FFMA)
    return fail(TPR_E_OPTION, "run_model: unknown decoder flag");
  DeviceInfo di = device_info();
  if (!di.ok) return fail(TPR_E_DEVICE, "run_model: no CUDA device");
  const float box_scale = (float)(2.0 / box_warp);      // python float (VR/renderer.py:61)
  // Point queries with enough points to fill the GPU run the warp-specialised tensor-core kernel (2xFP16 operand pairs in the fp32
  // mode, bf16 operands in the bf16 mode); small queries, pre-gathered features (tpr_decode) and TPR_MLP_FFMA run the
  // fp32 FFMA kernel below, whose 32-point chunks spread over the SMs at any size.
  if (!from_features && flags != TPR_MLP_FFMA && (long long)n_img * n_pts >= env_int("TPR_RM_WS_MIN_POINTS", 1 << 16) &&
      !env_int("TPR_FORCE_FFMA", 0)) {
    int rc = launch_run_model_ws(planes, n_img, plane_sets, H, W, dec, in, n_pts, box_scale, rgb, sigma, tc_mode(flags), di.sms,
                                 di.smem_optin, (cudaStream_t)stream);
    if (rc > 0) return cuda_fail((cudaError_t)rc, "run_model_ws_kernel");
    if (rc == 0) return 0;
  }
  const size_t smem = sizeof(float) * (kDecFloats + kRmWarps * 32 * kC);
  static std::once_flag once[2];
  cudaError_t attr_err = cudaSuccess;
  std::call_once(once[from_features ? 1 : 0], [&] {
    attr_err = from_features
                   ? cudaFuncSetAttribute(run_model_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                   : cudaFuncSetAttribute(run_model_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  });
  if (attr_err != cudaSuccess) return cuda_fail(attr_err, "cudaFuncSetAttribute(run_model_kernel)");
  const long long total = (long long)n_img * n_pts;
  const int grid = grid_for(total, kRmThreads, di.sms, env_int("TPR_RM_WAVES", 3));
  if (from_features)
    run_model_kernel<true><<<grid, kRmThreads, smem, (cudaStream_t)stream>>>(nullptr, 0, 0, dec, in, n_img, n_pts, 0.f, rgb, sigma, 1);
  else
    run_model_kernel<false><<<grid, kRmThreads, smem, (cudaStream_t)stream>>>(planes, H, W, dec, in, n_img, n_pts, box_scale, rgb, sigma,
                                                                          plane_sets);
  TPR_CHECK_LAUNCH("run_model_kernel");
  return 0;
}

int tpr_run_model(const float* planes_packed, int64_t n_img, int32_t height, int32_t width, const float* decoder_packed,
                  const float* xyz, int64_t n_pts, double box_warp, float* rgb, float* sigma, int32_t flags, void* stream) {
  return launch_run_model(false, planes_packed, n_img, n_img, height, width, decoder_packed, xyz, n_pts, box_warp, rgb, sigma,
                          flags, stream);
}

int tpr_decode(const float* features, int64_t n_img, int64_t n_pts, const float* decoder_packed, float* rgb, float* sigma,
               int32_t flags, void* stream) {
  if (!rgb) return fail(TPR_E_NULL, "tpr_decode: NULL rgb");
  return launch_run_model(true, nullptr, n_img, 1, 0, 0, decoder_packed, features, n_pts, 1.0, rgb, sigma, flags, stream);
}

// [0..8) call-wide depth range, [64..192) phase counters, from byte 256 one (min, max) pair per depth-clamp slot
size_t tpr_render_scratch_bytes(int64_t n_img, int64_t, const TprOptions* opt) {
  const int64_t k = opt ? opt->depth_clamp_group : 0;
  const int64_t slots = (k > 0 && n_img > 0) ? (n_img + k - 1) / k : 0;
  return (size_t)(512 + 8 * slots);
}

// pick rays-per-CTA and threads for render_kernel
static void render_config(int Dc, int Df, int smem_optin, int& R, int& threads, size_t& smem) {
  const int S = Dc + Df;
  const int budget = env_int("TPR_SMEM_BUDGET", 112 * 1024);      // two CTAs per SM
  R = env_int("TPR_RAYS_PER_CTA", 0);
  if (R <= 0) {
    R = 8;
    while (R > 1 && (int)render_smem_bytes(R, S) > budget) --R;
  }
  while (R > 1 && (int)render_smem_bytes(R, S) > smem_optin) --R;
  smem = render_smem_bytes(R, S);
  threads = env_int("TPR_THREADS", 0);
  if (threads <= 0) {
    const int dmax = Dc > Df ? Dc : Df;
    int warps = (R * dmax + 31) / 32;
    if (warps < 4) warps = 4;
    if (warps > 16) warps = 16;
    threads = warps * 32;
  }
  if (threads > kRenderMaxThreads) threads = kRenderMaxThreads;
  threads = (threads + 31) / 32 * 32;
}

// The body of tpr_render.  `phases`: kRangeInit resets the running depth range in `scratch` before rendering,
// kFinish decodes it (and clamps when clamp_depth != 0) afterwards.  tpr_render_host renders image by image
// against ONE running range and finishes once.
enum { kRangeInit = 1, kFinish = 2 };
static int render_impl(const float* planes_packed, int64_t n_img, int32_t height, int32_t width, const float* decoder_packed,
                       const float* origins, const float* dirs, int64_t n_rays, const float* jitter, const float* u,
                       const float* ray_start_per_ray, const float* ray_end_per_ray, const TprOptions* opt, float* rgb,
                       float* depth, float* weight_sum, float* fine_depths, int32_t* fine_inds, float* depth_range_io,
                       int32_t clamp_depth, void* scratch, size_t scratch_bytes, void* stream, int phases,
                       const TprPeerSinks* peers = nullptr, float* sample_colours = nullptr, float* sample_sigma = nullptr,
                       int32_t* samples_saved = nullptr, float* sample_features = nullptr) {
  if (!planes_packed || !decoder_packed || !origins || !dirs || !jitter || !opt || !rgb || !depth || !weight_sum || !scratch)
    return fail(TPR_E_NULL, "tpr_render: NULL pointer");
  if ((ray_start_per_ray == nullptr) != (ray_end_per_ray == nullptr))
    return fail(TPR_E_NULL, "tpr_render: per-ray limits need both start and end");
  const int Dc = opt->depth_resolution, Df = opt->depth_resolution_importance;
  if (n_img <= 0 || n_rays <= 0 || height <= 0 || width <= 0 || (int64_t)height * width > (1 << 24))
    return fail(TPR_E_SHAPE, "tpr_render: bad shape");
  if (Dc < 2 || Df < 0 || Dc + Df > TPR_MAX_SAMPLES) return fail(TPR_E_SHAPE, "tpr_render: depth resolutions out of range");
  if (Df > 0 && Dc < 4) return fail(TPR_E_SHAPE, "tpr_render: importance sampling needs depth_resolution >= 4");
  if (Df > 0 && !u) return fail(TPR_E_NULL, "tpr_render: NULL u with depth_resolution_importance > 0");
  if (!(opt->box_warp > 0.0)) return fail(TPR_E_OPTION, "tpr_render: box_warp must be > 0");
  if (opt->flags != TPR_MLP_FP32 && opt->flags != TPR_MLP_BF16 && opt->flags != TPR_MLP_FFMA)
    return fail(TPR_E_OPTION, "tpr_render: unknown decoder flag");
  if (scratch_bytes < tpr_render_scratch_bytes(n_img, n_rays, opt)) return fail(TPR_E_SCRATCH, "tpr_render: scratch too small");
  if (n_img >= (1ll << 31)) return fail(TPR_E_SHAPE, "tpr_render: too many images");
  if (opt->plane_sets < 0 || (opt->plane_sets > 0 && n_img % opt->plane_sets != 0))
    return fail(TPR_E_SHAPE, "tpr_render: n_img must be a multiple of plane_sets");
  if (opt->depth_clamp_group < 0) return fail(TPR_E_OPTION, "tpr_render: depth_clamp_group < 0");
  if (opt->output_layout != TPR_LAYOUT_CHANNELS_LAST && opt->output_layout != TPR_LAYOUT_CHANNELS_FIRST)
    return fail(TPR_E_OPTION, "tpr_render: unknown output_layout");
  // the reference's disparity branch (VR/renderer.py:174-181) divides python floats; with per-ray tensors it fails on shapes
  if (ray_start_per_ray && opt->disparity_space_sampling)
    return fail(TPR_E_OPTION, "tpr_render: disparity_space_sampling takes scalar ray limits, not per-ray ('auto') limits");
  if (!ray_start_per_ray && opt->disparity_space_sampling && !(opt->ray_start > 0.0 && opt->ray_end > 0.0))
    return fail(TPR_E_OPTION, "tpr_render: disparity_space_sampling needs ray_start > 0 and ray_end > 0");
  if (opt->density_noise < 0.0) return fail(TPR_E_OPTION, "tpr_render: density_noise < 0");
  if (opt->density_noise > 0.0 && (!opt->density_noise_coarse || (Df > 0 && !opt->density_noise_fine)))
    return fail(TPR_E_NULL, "tpr_render: density_noise > 0 needs the standard-normal draws (density_noise_coarse / _fine)");
  DeviceInfo di = device_info();
  if (!di.ok) return fail(TPR_E_DEVICE, "tpr_render: no CUDA device");

  RenderArgs a;
  memset(&a, 0, sizeof(a));
  a.planes = planes_packed; a.H = height; a.W = width; a.dec = decoder_packed;
  a.origins = origins; a.dirs = dirs; a.jitter = jitter; a.u = u;
  a.rs = ray_start_per_ray; a.re = ray_end_per_ray;
  a.n_rays_total = (long long)n_img * n_rays; a.rays_per_img = n_rays;
  set_depth_constants(a, opt);
  a.box_scale = (float)(2.0 / opt->box_warp);                                           // python float (VR/renderer.py:61)
  a.Df = Df; a.white_back = opt->white_back;
  a.plane_sets = opt->plane_sets > 0 ? opt->plane_sets : (int)n_img;
  a.nchw = opt->output_layout == TPR_LAYOUT_CHANNELS_FIRST;
  a.clamp_group = opt->depth_clamp_group;
  if (opt->density_noise > 0.0) {                                                       // VR/renderer.py:146
    a.noise_c = opt->density_noise_coarse; a.noise_f = opt->density_noise_fine; a.density_noise = (float)opt->density_noise;
  }
  const int n_slots = a.clamp_group > 0 ? (int)((n_img + a.clamp_group - 1) / a.clamp_group) : 0;
  a.rgb = rgb; a.depth = depth; a.wsum = weight_sum; a.fine_depths = fine_depths; a.fine_inds = fine_inds;
  a.range_enc = reinterpret_cast<unsigned*>(scratch);
  if (peers) {
    if (peers->n_peers < 0 || peers->n_peers > TPR_MAX_PEERS) return fail(TPR_E_SHAPE, "tpr_render_peers: n_peers out of range");
    if (clamp_depth) return fail(TPR_E_OPTION, "tpr_render_peers: the depth clamp needs the all-reduced range; pass clamp_depth = 0");
    a.peers.n = peers->n_peers;
    for (int p = 0; p < peers->n_peers; ++p) {
      if (!peers->rgb[p] || !peers->depth[p] || !peers->weight_sum[p]) return fail(TPR_E_NULL, "tpr_render_peers: NULL peer pointer");
      a.peers.rgb[p] = peers->rgb[p]; a.peers.depth[p] = peers->depth[p]; a.peers.wsum[p] = peers->weight_sum[p];
    }
  }
  {
    // column grouping needs the rays to be a square image with x fastest (what RaySampler produces); the caller
    // can say so through tile_width, otherwise it is inferred from a perfect-square ray count
    int w = opt->tile_width;
    if (w == 0) { w = (int)llround(sqrt((double)n_rays)); if ((long long)w * w != n_rays) w = 0; }
    if (w < 0 || env_int("TPR_NO_COLUMN_TILES", 0)) w = 0;
    a.col_w = w;
  }
  a.variant = env_int("TPR_WS_VARIANT", 0);
  // cp.async.bulk for the per-group jitter / u rows: built, parity-clean, and measured SLOWER than the 4-byte cp.async prefetch
  // (config 2, same box: 2.266 vs 2.218 ms; equal at 96+96) -- one thread issuing 16 small bulk copies per group costs its warp
  // more than 3 fire-and-forget LDGSTS per thread cost all of them.  Opt-in for A/B: TPR_WS_VARIANT bit 6.
  a.bulk_inputs = (a.variant & 64) && (Dc % 4 == 0) && (Df % 4 == 0) && ((uintptr_t)jitter % 16 == 0) &&
                  (Df == 0 || (uintptr_t)u % 16 == 0);
  a.dbg = env_int("TPR_PHASE_TIMING", 0) ? reinterpret_cast<long long*>(reinterpret_cast<char*>(scratch) + 64) : nullptr;
  cudaStream_t st = (cudaStream_t)stream;
  if (phases & kRangeInit) {
    range_init_kernel<<<n_slots > 256 ? (n_slots + 255) / 256 : 1, n_slots > 0 ? 256 : 1, 0, st>>>(a.range_enc, n_slots);
    TPR_CHECK_LAUNCH("range_init_kernel");
  }

  // Dispatch: the warp-specialised tcgen05 kernel whenever the sample counts fit its TMEM colour-slot pool (every depth
  // pair any G-NeRF configuration uses), else -- or with TPR_MLP_FFMA -- the fp32 FFMA kernel, which takes any S <= 256.
  bool done = false;
  if (opt->flags != TPR_MLP_FFMA && !env_int("TPR_FORCE_FFMA", 0) && ws_rays_per_group(Dc, Df, tc_mode(opt->flags)) > 0) {
    const bool keep = sample_colours && sample_sigma && ws_keeps_samples(Dc, Df) && !a.dbg;
    if (keep) { a.sample_colours = sample_colours; a.sample_sigma = sample_sigma; a.sample_features = sample_features; }   // (only this kernel can keep them)
    if (keep) {                                   // profiling A/B only (results of the backward are then garbage): skip one of the kept streams
      const int dbg = env_int("TPR_TRAIN_DEBUG", 0);
      if (dbg & 1) a.sample_colours = nullptr;
      if (dbg & 2) a.sample_features = nullptr;
    }
    int rc = launch_render_ws(a, tc_mode(opt->flags), di.sms, di.smem_optin, n_img, n_rays, st);
    if (rc > 0) return cuda_fail((cudaError_t)rc, "render_ws_kernel");
    done = rc == 0;                       // < 0: does not fit shared memory, fall through
    a.sample_colours = nullptr; a.sample_sigma = nullptr; a.sample_features = nullptr;
  }
  if (samples_saved) *samples_saved = (done && sample_colours && sample_sigma && ws_keeps_samples(Dc, Df) && !a.dbg) ? 1 : 0;
  const bool kernel_stores_to_peers = done;     // only the warp-specialised kernel has the peer stores in its epilogue
  if (!done) {
    void (*kern)(const RenderArgs) = (Dc + Df <= 64) ? render_kernel<2> : (Dc + Df <= 128) ? render_kernel<4> : render_kernel<8>;
    cudaFuncAttributes fa;
    {
      cudaError_t e = cudaFuncGetAttributes(&fa, kern);
      if (e != cudaSuccess) return cuda_fail(e, "cudaFuncGetAttributes(render_kernel): no sm_100a image for this device?");
    }
    const int smem_cap = di.smem_optin - (int)fa.sharedSizeBytes;      // static smem counts against the opt-in limit
    int R, threads; size_t smem;
    render_config(Dc, Df, smem_cap, R, threads, smem);
    if ((int)smem > smem_cap) return fail(TPR_E_SHAPE, "tpr_render: sample count does not fit shared memory");
    {
      // per device and cheap; set on every call rather than caching per device
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(render_kernel)");
    }
    a.R = R;
    a.tiles_per_img = (n_rays + R - 1) / R;
    a.n_tiles = a.tiles_per_img * n_img;
    int occ = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, smem);
    if (occ < 1) occ = 1;
    long long grid = (long long)di.sms * occ;
    if (grid > a.n_tiles) grid = a.n_tiles;
    kern<<<(unsigned)grid, threads, smem, st>>>(a);
    TPR_CHECK_LAUNCH("render_kernel");
  }
  if (a.peers.n > 0 && !kernel_stores_to_peers) {
    // sample counts that do not fit the warp-specialised kernel: forward this GPU's outputs after the render
    peer_scatter_kernel<<<grid_for(a.n_rays_total * kC, 256, di.sms, 8), 256, 0, st>>>(a.peers, rgb, depth, weight_sum, a.n_rays_total);
    TPR_CHECK_LAUNCH("peer_scatter_kernel");
  }
  if (phases & kFinish) {
    finish_kernel<<<grid_for(a.n_rays_total, 256, di.sms, 4), 256, 0, st>>>(a.range_enc, depth_range_io, depth, a.n_rays_total,
                                                                            clamp_depth, (long long)a.clamp_group * n_rays);
    TPR_CHECK_LAUNCH("finish_kernel");
  }
  return 0;
}

int tpr_render(const float* planes_packed, int64_t n_img, int32_t height, int32_t width, const float* decoder_packed,
               const float* origins, const float* dirs, int64_t n_rays, const float* jitter, const float* u,
               const float* ray_start_per_ray, const float* ray_end_per_ray, const TprOptions* opt, float* rgb,
               float* depth, float* weight_sum, float* fine_depths, int32_t* fine_inds, float* depth_range_io,
               int32_t clamp_depth, void* scratch, size_t scratch_bytes, void* stream) {
  return render_impl(planes_packed, n_img, height, width, decoder_packed, origins, dirs, n_rays, jitter, u, ray_start_per_ray,
                     ray_end_per_ray, opt, rgb, depth, weight_sum, fine_depths, fine_inds, depth_range_io, clamp_depth, scratch,
                     scratch_bytes, stream, kRangeInit | kFinish);
}

int tpr_render_train(const float* planes_packed, int64_t n_img, int32_t height, int32_t width, const float* decoder_packed,
                     const float* origins, const float* dirs, int64_t n_rays, const float* jitter, const float* u,
                     const float* ray_start_per_ray, const float* ray_end_per_ray, const TprOptions* opt, float* rgb,
                     float* depth, float* weight_sum, float* fine_depths, float* depth_range_io, float* sample_colours,
                     float* sample_sigma, float* sample_features, int32_t* samples_saved, void* scratch, size_t scratch_bytes,
                     void* stream) {
  if (!sample_colours || !sample_sigma || !samples_saved) return fail(TPR_E_NULL, "tpr_render_train: NULL pointer");
  if (opt && opt->depth_resolution_importance > 0 && !fine_depths) return fail(TPR_E_NULL, "tpr_render_train: NULL fine_depths");
  return render_impl(planes_packed, n_img, height, width, decoder_packed, origins, dirs, n_rays, jitter, u, ray_start_per_ray,
                     ray_end_per_ray, opt, rgb, depth, weight_sum, fine_depths, nullptr, depth_range_io, 1, scratch, scratch_bytes,
                     stream, kRangeInit | kFinish, nullptr, sample_colours, sample_sigma, samples_saved, sample_features);
}

int tpr_render_peers(const float* planes_packed, int64_t n_img, int32_t height, int32_t width, const float* decoder_packed,
                     const float* origins, const float* dirs, int64_t n_rays, const float* jitter, const float* u,
                     const float* ray_start_per_ray, const float* ray_end_per_ray, const TprOptions* opt, float* rgb,
                     float* depth, float* weight_sum, float* depth_range_io, void* scratch, size_t scratch_bytes,
                     const TprPeerSinks* peers, void* stream) {
  if (!peers) return fail(TPR_E_NULL, "tpr_render_peers: NULL peers");
  return render_impl(planes_packed, n_img, height, width, decoder_packed, origins, dirs, n_rays, jitter, u, ray_start_per_ray,
                     ray_end_per_ray, opt, rgb, depth, weight_sum, nullptr, nullptr, depth_range_io, 0, scratch,
                     scratch_bytes, stream, kRangeInit | kFinish, peers);
}

// peer-mappable gather buffers (see the header): the one place the library owns device memory, with explicit
// create / destroy.  cudaIpc* needs a cudaMalloc allocation whose base address is the exported pointer, which a
// sub-allocating caller (PyTorch's caching allocator) cannot promise.
int tpr_peer_alloc(size_t bytes, void** dev_ptr, unsigned char* handle_out) {
  if (!dev_ptr || !handle_out) return fail(TPR_E_NULL, "tpr_peer_alloc: NULL pointer");
  if (bytes == 0) return fail(TPR_E_SHAPE, "tpr_peer_alloc: zero bytes");
  static_assert(sizeof(cudaIpcMemHandle_t) == TPR_PEER_HANDLE_BYTES, "handle size");
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, bytes);
  if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(peer buffer)");
  cudaIpcMemHandle_t h;
  e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) { cudaFree(p); return cuda_fail(e, "cudaIpcGetMemHandle"); }
  memcpy(handle_out, &h, sizeof(h));
  *dev_ptr = p;
  return 0;
}
int tpr_peer_open(const unsigned char* handle, void** dev_ptr) {
  if (!handle || !dev_ptr) return fail(TPR_E_NULL, "tpr_peer_open: NULL pointer");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  void* p = nullptr;
  cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
  if (e != cudaSuccess) return cuda_fail(e, "cudaIpcOpenMemHandle (no NVLink / PCIe peer access between these GPUs?)");
  *dev_ptr = p;
  return 0;
}
int tpr_peer_close(void* dev_ptr) {
  if (!dev_ptr) return fail(TPR_E_NULL, "tpr_peer_close: NULL pointer");
  cudaError_t e = cudaIpcCloseMemHandle(dev_ptr);
  return e == cudaSuccess ? 0 : cuda_fail(e, "cudaIpcCloseMemHandle");
}
int tpr_peer_free(void* dev_ptr) {
  if (!dev_ptr) return fail(TPR_E_NULL, "tpr_peer_free: NULL pointer");
  cudaError_t e = cudaFree(dev_ptr);
  return e == cudaSuccess ? 0 : cuda_fail(e, "cudaFree(peer buffer)");
}

// ---------------------------------------------------------------------------------------------------------
// The same forward with HOST buffers: planes / rays come from (pinned) host memory, outputs land in host memory.
// One image's planes are 25 MB and take longer to cross PCIe than to render, so the images are pipelined over
// three streams -- copy-in (H2D of image i+1), the caller's stream (repack + render of image i), copy-out (D2H of
// image i-1) -- with the raw planes double buffered.  The global depth clamp (VR/ray_marcher.py:50) needs every
// image, so depth is clamped and copied back last.
// ---------------------------------------------------------------------------------------------------------
namespace {
struct HostPipe {
  cudaStream_t in = nullptr, out = nullptr;
  std::vector<cudaEvent_t> ev;
  bool ok = false;
};
std::mutex g_pipe_mu;
HostPipe g_pipe[64];

// streams / events of the current device (created on first use; the only per-device state the library keeps)
HostPipe* host_pipe(int n_events) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  std::lock_guard<std::mutex> lk(g_pipe_mu);
  HostPipe& p = g_pipe[dev];
  if (!p.ok) {
    if (cudaStreamCreateWithFlags(&p.in, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    if (cudaStreamCreateWithFlags(&p.out, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    p.ok = true;
  }
  while ((int)p.ev.size() < n_events) {
    cudaEvent_t e;
    if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    p.ev.push_back(e);
  }
  return &p;
}

struct HostWs { size_t raw, packed, rays, rgb, depth, wsum, scratch, total; };
HostWs host_ws_layout(int64_t n_img, int32_t H, int32_t W, int64_t n_rays) {
  auto up = [](size_t x) { return (x + 1023) & ~(size_t)1023; };
  HostWs w;
  const size_t img = (size_t)TPR_PLANES * TPR_CHANNELS * H * W * sizeof(float);
  size_t o = 0;
  w.raw = o; o += 2 * up(img);
  w.packed = o; o += 2 * up(img);
  w.rays = o; o += up((size_t)n_img * n_rays * 6 * sizeof(float));
  w.rgb = o; o += up((size_t)n_img * n_rays * TPR_CHANNELS * sizeof(float));
  w.depth = o; o += up((size_t)n_img * n_rays * sizeof(float));
  w.wsum = o; o += up((size_t)n_img * n_rays * sizeof(float));
  w.scratch = o; o += 1024;
  w.total = o;
  return w;
}
}  // namespace

size_t tpr_render_host_workspace_bytes(int64_t n_img, int32_t height, int32_t width, int64_t n_rays) {
  if (n_img <= 0 || height <= 0 || width <= 0 || n_rays <= 0) return 0;
  return host_ws_layout(n_img, height, width, n_rays).total;
}

#define TPR_CUDA(call, what)                                       \
  do {                                                             \
    cudaError_t e__ = (call);                                      \
    if (e__ != cudaSuccess) return cuda_fail(e__, what);           \
  } while (0)

int tpr_render_host(const float* planes_host, int64_t n_img, int32_t height, int32_t width, const float* decoder_packed,
                    const float* origins_host, const float* dirs_host, int64_t n_rays, const float* jitter, const float* u,
                    const TprOptions* opt, float* rgb_host, float* depth_host, float* weight_sum_host, float* depth_range_io,
                    void* workspace, size_t workspace_bytes, void* stream) {
  if (!planes_host || !decoder_packed || !origins_host || !dirs_host || !jitter || !opt || !rgb_host || !weight_sum_host || !workspace)
    return fail(TPR_E_NULL, "tpr_render_host: NULL pointer");
  if (!depth_host && !depth_range_io) return fail(TPR_E_NULL, "tpr_render_host: deferred depth (depth_host = NULL) needs depth_range_io");
  if (n_img <= 0 || n_rays <= 0 || height <= 0 || width <= 0 || (int64_t)height * width > (1 << 24))
    return fail(TPR_E_SHAPE, "tpr_render_host: bad shape");
  if (opt->depth_resolution_importance > 0 && !u) return fail(TPR_E_NULL, "tpr_render_host: NULL u");
  if (opt->plane_sets != 0 && opt->plane_sets != n_img)
    return fail(TPR_E_OPTION, "tpr_render_host: plane_sets must be 0 (every image brings its own planes across PCIe)");
  if (opt->depth_clamp_group != 0) return fail(TPR_E_OPTION, "tpr_render_host: depth_clamp_group must be 0");
  const HostWs w = host_ws_layout(n_img, height, width, n_rays);
  if (workspace_bytes < w.total) return fail(TPR_E_SCRATCH, "tpr_render_host: workspace too small");
  // One caller at a time per process while the pipeline is ENQUEUED: the copy streams and the events are per-device state
  // shared by every caller.  A cudaStreamWaitEvent captures the event's most recent record at the time of the call, so once
  // this call's record / wait pairs are enqueued a later caller re-recording the same events cannot disturb them.
  static std::mutex enqueue_mu;
  std::lock_guard<std::mutex> enqueue_lock(enqueue_mu);
  HostPipe* hp = host_pipe((int)(2 * n_img + 4));
  if (!hp) return fail(TPR_E_DEVICE, "tpr_render_host: cannot create copy streams / events");
  cudaStream_t st = (cudaStream_t)stream;
  char* ws = reinterpret_cast<char*>(workspace);
  const size_t img_floats = (size_t)TPR_PLANES * TPR_CHANNELS * height * width, img_bytes = img_floats * sizeof(float);
  const size_t img_stride = (img_bytes + 1023) & ~(size_t)1023;
  float* d_orig = reinterpret_cast<float*>(ws + w.rays);
  float* d_dirs = d_orig + (size_t)n_img * n_rays * 3;
  float* d_rgb = reinterpret_cast<float*>(ws + w.rgb);
  float* d_depth = reinterpret_cast<float*>(ws + w.depth);
  float* d_wsum = reinterpret_cast<float*>(ws + w.wsum);
  const int Dc = opt->depth_resolution, Df = opt->depth_resolution_importance;
  // events: [0] entry fence, [1..2] raw buffer free, [3] all copied out, [4+2i] image i copied in, [5+2i] image i rendered
  cudaEvent_t* ev = hp->ev.data();

  // the workspace may still be in use by earlier work on the caller's stream (a previous call)
  TPR_CUDA(cudaEventRecord(ev[0], st), "cudaEventRecord");
  TPR_CUDA(cudaStreamWaitEvent(hp->in, ev[0], 0), "cudaStreamWaitEvent");
  TPR_CUDA(cudaStreamWaitEvent(hp->out, ev[0], 0), "cudaStreamWaitEvent");
  const size_t ray_bytes = (size_t)n_img * n_rays * 3 * sizeof(float);
  TPR_CUDA(cudaMemcpyAsync(d_orig, origins_host, ray_bytes, cudaMemcpyHostToDevice, hp->in), "cudaMemcpyAsync(origins)");
  TPR_CUDA(cudaMemcpyAsync(d_dirs, dirs_host, ray_bytes, cudaMemcpyHostToDevice, hp->in), "cudaMemcpyAsync(dirs)");
  for (int64_t i = 0; i < n_img; ++i) {
    const int b = (int)(i & 1);
    float* raw = reinterpret_cast<float*>(ws + w.raw + b * img_stride);
    float* packed = reinterpret_cast<float*>(ws + w.packed + b * img_stride);
    if (i >= 2) TPR_CUDA(cudaStreamWaitEvent(hp->in, ev[1 + b], 0), "cudaStreamWaitEvent");      // repack of image i-2 done
    TPR_CUDA(cudaMemcpyAsync(raw, planes_host + (size_t)i * img_floats, img_bytes, cudaMemcpyHostToDevice, hp->in),
             "cudaMemcpyAsync(planes)");
    TPR_CUDA(cudaEventRecord(ev[4 + 2 * i], hp->in), "cudaEventRecord");
    TPR_CUDA(cudaStreamWaitEvent(st, ev[4 + 2 * i], 0), "cudaStreamWaitEvent");
    int rc = tpr_pack_planes(raw, 1, height, width, packed, st);
    if (rc != 0) return rc;
    TPR_CUDA(cudaEventRecord(ev[1 + b], st), "cudaEventRecord");
    const size_t ro = (size_t)i * n_rays;
    TprOptions oi = *opt;                          // this image's slice of the density-noise draws
    if (opt->density_noise > 0.0 && opt->density_noise_coarse) oi.density_noise_coarse = opt->density_noise_coarse + ro * Dc;
    if (opt->density_noise > 0.0 && opt->density_noise_fine) oi.density_noise_fine = opt->density_noise_fine + ro * Df;
    rc = render_impl(packed, 1, height, width, decoder_packed, d_orig + ro * 3, d_dirs + ro * 3, n_rays, jitter + ro * Dc,
                     u ? u + ro * Df : nullptr, nullptr, nullptr, &oi, d_rgb + ro * TPR_CHANNELS, d_depth + ro, d_wsum + ro,
                     nullptr, nullptr, nullptr, 0, ws + w.scratch, 1024, st, i == 0 ? kRangeInit : 0);
    if (rc != 0) return rc;
    TPR_CUDA(cudaEventRecord(ev[5 + 2 * i], st), "cudaEventRecord");
    TPR_CUDA(cudaStreamWaitEvent(hp->out, ev[5 + 2 * i], 0), "cudaStreamWaitEvent");
    TPR_CUDA(cudaMemcpyAsync(rgb_host + ro * TPR_CHANNELS, d_rgb + ro * TPR_CHANNELS, (size_t)n_rays * TPR_CHANNELS * sizeof(float),
                             cudaMemcpyDeviceToHost, hp->out), "cudaMemcpyAsync(rgb)");
    TPR_CUDA(cudaMemcpyAsync(weight_sum_host + ro, d_wsum + ro, (size_t)n_rays * sizeof(float), cudaMemcpyDeviceToHost, hp->out),
             "cudaMemcpyAsync(weight_sum)");
  }
  DeviceInfo di = device_info();
  const long long total = (long long)n_img * n_rays;
  // depth_host = NULL: the caller shards rays over GPUs and owes the clamp an all-reduced range -- only decode this GPU's
  // range; tpr_render_host_depth finishes the job
  finish_kernel<<<grid_for(total, 256, di.sms, 4), 256, 0, st>>>(reinterpret_cast<unsigned*>(ws + w.scratch), depth_range_io,
                                                                 d_depth, total, depth_host ? 1 : 0, 0);
  TPR_CHECK_LAUNCH("finish_kernel");
  if (depth_host)
    TPR_CUDA(cudaMemcpyAsync(depth_host, d_depth, (size_t)total * sizeof(float), cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(depth)");
  // the caller's stream completes only when every output has landed
  TPR_CUDA(cudaEventRecord(ev[3], hp->out), "cudaEventRecord");
  TPR_CUDA(cudaStreamWaitEvent(st, ev[3], 0), "cudaStreamWaitEvent");
  return 0;
}

int tpr_render_host_depth(void* workspace, size_t workspace_bytes, int64_t n_img, int32_t height, int32_t width, int64_t n_rays,
                          const float* depth_range, float* depth_host, void* stream) {
  if (!workspace || !depth_range || !depth_host) return fail(TPR_E_NULL, "tpr_render_host_depth: NULL pointer");
  if (n_img <= 0 || n_rays <= 0 || height <= 0 || width <= 0) return fail(TPR_E_SHAPE, "tpr_render_host_depth: bad shape");
  const HostWs w = host_ws_layout(n_img, height, width, n_rays);
  if (workspace_bytes < w.total) return fail(TPR_E_SCRATCH, "tpr_render_host_depth: workspace too small");
  DeviceInfo di = device_info();
  if (!di.ok) return fail(TPR_E_DEVICE, "tpr_render_host_depth: no CUDA device");
  cudaStream_t st = (cudaStream_t)stream;
  float* d_depth = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + w.depth);
  const long long total = (long long)n_img * n_rays;
  clamp_depth_kernel<<<grid_for(total, 256, di.sms, 4), 256, 0, st>>>(d_depth, total, depth_range);
  TPR_CHECK_LAUNCH("clamp_depth_kernel");
  TPR_CUDA(cudaMemcpyAsync(depth_host, d_depth, (size_t)total * sizeof(float), cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(depth)");
  return 0;
}

int tpr_clamp_depth(float* depth, int64_t n, const float* depth_range, void* stream) {
  if (!depth || !depth_range) return fail(TPR_E_NULL, "tpr_clamp_depth: NULL pointer");
  if (n <= 0) return fail(TPR_E_SHAPE, "tpr_clamp_depth: n <= 0");
  DeviceInfo di = device_info();
  if (!di.ok) return fail(TPR_E_DEVICE, "tpr_clamp_depth: no CUDA device");
  clamp_depth_kernel<<<grid_for(n, 256, di.sms, 4), 256, 0, (cudaStream_t)stream>>>(depth, n, depth_range);
  TPR_CHECK_LAUNCH("clamp_depth_kernel");
  return 0;
}

int tpr_ray_march(const float* colors, const float* densities, const float* depths, int64_t n_rays, int32_t n_samples,
                  int32_t n_channels, int32_t white_back, float* rgb, float* depth, float* weights, float* depth_range,
                  int32_t clamp_depth, void* stream) {
  if (!colors || !densities || !depths || !rgb || !depth || !weights || !depth_range)
    return fail(TPR_E_NULL, "tpr_ray_march: NULL pointer");
  if (n_rays <= 0 || n_samples < 2 || n_channels <= 0) return fail(TPR_E_SHAPE, "tpr_ray_march: bad shape");
  DeviceInfo di = device_info();
  if (!di.ok) return fail(TPR_E_DEVICE, "tpr_ray_march: no CUDA device");
  cudaStream_t st = (cudaStream_t)stream;
  // depth_range[2..3] hold the encoded (min,max) until finish_kernel decodes them into [0..1]
  unsigned* enc = reinterpret_cast<unsigned*>(depth_range) + 2;
  range_init_kernel<<<1, 1, 0, st>>>(enc, -1);
  TPR_CHECK_LAUNCH("range_init_kernel");
  ray_march_kernel<<<grid_for(n_rays, 8, di.sms, 8), 256, 0, st>>>(colors, densities, depths, n_rays, n_samples, n_channels,
                                                                   white_back, rgb, depth, weights, enc);
  TPR_CHECK_LAUNCH("ray_march_kernel");
  finish_kernel<<<grid_for(n_rays, 256, di.sms, 4), 256, 0, st>>>(enc, depth_range, depth, n_rays, clamp_depth, 0);
  TPR_CHECK_LAUNCH("finish_kernel");
  return 0;
}

static int launch_resample(int mode, const float* z, int z_stride, const float* w, const float* u, int64_t n_rays, int S_or_nb,
                           int K, float* samples, int32_t* inds, void* stream) {
  if (!z || !w || !u || !samples) return fail(TPR_E_NULL, "resample: NULL pointer");
  if (n_rays <= 0 || K <= 0) return fail(TPR_E_SHAPE, "resample: empty input");
  if (mode == 0 && (S_or_nb < 4 || S_or_nb > 4096)) return fail(TPR_E_SHAPE, "tpr_sample_importance: need 4 <= n_samples <= 4096");
  if (mode == 1 && (S_or_nb < 1 || S_or_nb > 4096)) return fail(TPR_E_SHAPE, "tpr_sample_pdf: need 1 <= n_weights <= 4096");
  DeviceInfo di = device_info();
  if (!di.ok) return fail(TPR_E_DEVICE, "resample: no CUDA device");
  const int cap = mode == 0 ? S_or_nb : S_or_nb + 2;
  const size_t smem = sizeof(float) * 4 * cap * kPdfWarps;
  if (smem > 48 * 1024) {
    static std::once_flag once;
    std::call_once(once, [&] { cudaFuncSetAttribute(resample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, di.smem_optin); });
  }
  resample_kernel<<<grid_for(n_rays, kPdfWarps, di.sms, 16), kPdfWarps * 32, smem, (cudaStream_t)stream>>>(
      mode, z, z_stride, w, u, n_rays, S_or_nb, K, samples, inds);
  TPR_CHECK_LAUNCH("resample_kernel");
  return 0;
}

int tpr_sample_importance(const float* z_vals, const float* weights, const float* u, int64_t n_rays, int32_t n_samples,
                          int32_t n_importance, float* samples, int32_t* inds, void* stream) {
  return launch_resample(0, z_vals, n_samples, weights, u, n_rays, n_samples, n_importance, samples, inds, stream);
}

int tpr_sample_pdf(const float* bins, int32_t bins_stride, const float* weights, const float* u, int64_t n_rays,
                   int32_t n_weights, int32_t n_importance, float* samples, int32_t* inds, void* stream) {
  if (bins_stride < n_weights + 1) return fail(TPR_E_SHAPE, "tpr_sample_pdf: bins_stride < n_weights + 1");
  return launch_resample(1, bins, bins_stride, weights, u, n_rays, n_weights, n_importance, samples, inds, stream);
}

// ---------------------------------------------------------------------------------------
// backward of tpr_render (kernels: tpr_backward.cu)
// ---------------------------------------------------------------------------------------
static size_t align256(size_t n) { return (n + 255) & ~(size_t)255; }
size_t tpr_render_backward_scratch_bytes(int64_t n_img, int64_t n_rays, int32_t n_samples) {
  if (n_img <= 0 || n_rays <= 0 || n_samples <= 0) return 0;
  const size_t T = (size_t)n_img * (size_t)n_rays * (size_t)n_samples;
  // points [T,3], colours [T,32], sigma [T], g_sigma [T], omega [T], the operand scale of the tcgen05 decoder backward
  return align256(T * 12) + align256(T * 128) + 3 * align256(T * 4) + 256;
}

// TPR_BWD_DETERMINISTIC: [256 B: DetScratch::hdr][kDetMaxRows decoder rows][int64 accumulator [P,3,H,W,32]]; P = the plane
// sets (tpr_render_backward with plane_sets > 0), else the images
size_t tpr_backward_deterministic_scratch_bytes(int64_t n_img, int32_t height, int32_t width) {
  if (n_img <= 0 || height <= 0 || width <= 0) return 0;
  return 256 + align256((size_t)kDetMaxRows * kDecFloats * sizeof(float)) +
         align256((size_t)n_img * 3 * (size_t)height * (size_t)width * kC * sizeof(long long));
}
static DetScratch det_scratch(void* scratch, size_t base) {
  uint8_t* q = (uint8_t*)scratch + base;
  DetScratch d;
  d.hdr = (int*)q; q += 256;
  d.rows = (float*)q; q += align256((size_t)kDetMaxRows * kDecFloats * sizeof(float));
  d.acc = (unsigned long long*)q;
  d.n_rows = 0;
  return d;
}

// The decoder backward of both entry points: tcgen05 + TMEM, warp-specialised (tpr_backward_tc.cu) first; the mma.sync kernel
// when it refuses (fewer than 128 samples per image, too little shared memory) or with TPR_BWD_IMPL=hmma (A/B runs).  The outputs
// are zeroed here.  det != NULL: the deterministic mode, its outputs converted after the kernel.  n_sets: the plane sets in
// planes_packed / g_planes_packed (image n = sample / pts_per_img reads and scatters to set n % n_sets).
static int decoder_backward(const float* planes_packed, int n_sets, int32_t height, int32_t width, const float* dec, const float* pts,
                            const float* colours, int col_chunked, const float* features, const float* gsig, const float* omega,
                            const float* g_rgb, long long total, long long pts_per_img, int S, int point, float box_scale, int fast,
                            float* g_planes_packed, float* g_decoder_packed, float* scale_buf, void* scratch, DetScratch* det,
                            const DeviceInfo& di, cudaStream_t st) {
  const size_t plane_floats = (size_t)n_sets * 3 * height * width * kC;
  cudaError_t e = cudaSuccess;
  if (g_planes_packed) e = det ? cudaMemsetAsync(det->acc, 0, plane_floats * sizeof(long long), st)
                               : cudaMemsetAsync(g_planes_packed, 0, plane_floats * sizeof(float), st);
  if (e == cudaSuccess && g_decoder_packed && !det) e = cudaMemsetAsync(g_decoder_packed, 0, kDecFloats * sizeof(float), st);
  if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
  const char* impl = getenv("TPR_BWD_IMPL");
  int rc = -1;
  if (!(impl && strcmp(impl, "hmma") == 0)) {
    rc = launch_bwd_decode_tc(planes_packed, height, width, dec, pts, colours, col_chunked, features, gsig, omega, g_rgb, total,
                              pts_per_img, n_sets, S, point, box_scale, g_planes_packed, g_decoder_packed, scale_buf, det, di.sms,
                              di.smem_optin, st);
    if (rc > 0) return cuda_fail((cudaError_t)rc, "decode_backward_tc_kernel");
  }
  if (rc != 0) {
    if (det) {
      rc = launch_det_bound(dec, gsig, g_rgb, total, n_sets, S, point, scale_buf, det, di.sms, st);
      if (rc != 0) return cuda_fail((cudaError_t)rc, "det_bound_kernel");
    }
    float* g_dec_out = g_decoder_packed ? g_decoder_packed : reinterpret_cast<float*>(scratch);      // (never written when skipped)
    rc = launch_bwd_decode(planes_packed, height, width, dec, pts, colours, col_chunked, features, gsig, omega, g_rgb, total,
                           pts_per_img, n_sets, S, point, box_scale, g_planes_packed, g_dec_out, fast,
                           (g_planes_packed ? 0 : 1) | (g_decoder_packed ? 0 : 2), det, di.sms, st);
    if (rc != 0) return cuda_fail((cudaError_t)rc, "decode_backward_kernel");
  }
  if (det) {
    rc = launch_det_finish(det, (long long)plane_floats, g_planes_packed, g_decoder_packed, di.sms, st);
    if (rc != 0) return cuda_fail((cudaError_t)rc, "det_planes_kernel");
  }
  return 0;
}

int tpr_march_backward(const float* depths_coarse, const float* depths_fine, int32_t dc, int32_t df, const float* sigma,
                       const float* colours, const float* g_rgb, const float* g_depth, const float* g_weight_sum,
                       const float* depth_range, int32_t white_back, int64_t n_rays_total, float* g_sigma, float* omega,
                       void* stream) {
  if (!depths_coarse || !sigma || !colours || !g_rgb || !g_depth || !g_weight_sum || !depth_range || !g_sigma || !omega ||
      (df > 0 && !depths_fine))
    return fail(TPR_E_NULL, "tpr_march_backward: NULL pointer");
  if (n_rays_total <= 0 || dc < 2 || df < 0 || dc + df > TPR_MAX_SAMPLES) return fail(TPR_E_SHAPE, "tpr_march_backward: bad shape");
  DeviceInfo di = device_info();
  if (!di.ok) return fail(TPR_E_DEVICE, "tpr_march_backward: no CUDA device");
  const int rc = launch_bwd_march(depths_coarse, depths_fine, dc, df, sigma, colours, 0, g_rgb, g_depth, g_weight_sum, depth_range, 0,
                                  white_back, n_rays_total, g_sigma, omega, di.sms, (cudaStream_t)stream);
  if (rc != 0) return cuda_fail((cudaError_t)rc, "march_backward_kernel");
  return 0;
}

int tpr_render_backward(const float* planes_packed, int64_t n_img, int32_t height, int32_t width, const float* decoder_packed,
                        const float* origins, const float* dirs, int64_t n_rays, const float* depths_coarse,
                        const float* depths_fine, const float* depth_range, const TprOptions* opt, const float* g_rgb,
                        const float* g_depth, const float* g_weight_sum, const float* sample_colours, const float* sample_sigma,
                        const float* sample_features, float* g_planes_packed, float* g_decoder_packed, void* scratch, size_t scratch_bytes, void* stream) {
  if ((sample_colours == nullptr) != (sample_sigma == nullptr))
    return fail(TPR_E_NULL, "tpr_render_backward: sample_colours and sample_sigma come together");
  if (!planes_packed || !decoder_packed || !origins || !dirs || !depths_coarse || !depth_range || !opt || !g_rgb || !g_depth ||
      !g_weight_sum || (!g_planes_packed && !g_decoder_packed) || !scratch)
    return fail(TPR_E_NULL, "tpr_render_backward: NULL pointer");
  const int Dc = opt->depth_resolution, Df = opt->depth_resolution_importance, S = Dc + Df;
  if (Df > 0 && !depths_fine) return fail(TPR_E_NULL, "tpr_render_backward: depths_fine is NULL but depth_resolution_importance > 0");
  if (n_img <= 0 || n_rays <= 0 || height <= 0 || width <= 0 || Dc < 2 || Df < 0 || S > TPR_MAX_SAMPLES)
    return fail(TPR_E_SHAPE, "tpr_render_backward: bad shape");
  if ((long long)3 * height * width * kC >= (1ll << 32)) return fail(TPR_E_SHAPE, "tpr_render_backward: planes too large");
  if (n_img >= (1ll << 31)) return fail(TPR_E_SHAPE, "tpr_render_backward: too many images");
  if (opt->plane_sets < 0 || (opt->plane_sets > 0 && n_img % opt->plane_sets != 0))
    return fail(TPR_E_SHAPE, "tpr_render_backward: n_img must be a multiple of plane_sets");
  if (opt->depth_clamp_group < 0) return fail(TPR_E_OPTION, "tpr_render_backward: depth_clamp_group < 0");
  if (opt->depth_clamp_group > 0 && n_img * n_rays >= (1ll << 32))
    return fail(TPR_E_SHAPE, "tpr_render_backward: depth_clamp_group needs fewer than 2^32 rays");
  const int P = opt->plane_sets > 0 ? opt->plane_sets : (int)n_img;
  if (!(opt->box_warp > 0)) return fail(TPR_E_OPTION, "tpr_render_backward: box_warp must be > 0");
  const bool det = (opt->flags & TPR_BWD_DETERMINISTIC) != 0;
  const int32_t mlp = opt->flags & ~TPR_BWD_DETERMINISTIC;
  if (mlp != TPR_MLP_FP32 && mlp != TPR_MLP_BF16 && mlp != TPR_MLP_FFMA)
    return fail(TPR_E_OPTION, "tpr_render_backward: unknown flag");
  const size_t base_bytes = tpr_render_backward_scratch_bytes(n_img, n_rays, S);
  if (scratch_bytes < base_bytes + (det ? tpr_backward_deterministic_scratch_bytes(P, height, width) : 0))
    return fail(TPR_E_SCRATCH, "tpr_render_backward: scratch too small");
  DeviceInfo di = device_info();
  if (!di.ok) return fail(TPR_E_DEVICE, "tpr_render_backward: no CUDA device");
  cudaStream_t st = (cudaStream_t)stream;
  const long long rays = (long long)n_img * n_rays;
  const size_t T = (size_t)rays * S;
  uint8_t* p = (uint8_t*)scratch;
  float* pts = (float*)p; p += align256(T * 12);
  float* colours = (float*)p; p += align256(T * 128);
  float* sigma = (float*)p; p += align256(T * 4);
  float* gsig = (float*)p; p += align256(T * 4);
  float* omega = (float*)p; p += align256(T * 4);
  float* scale_buf = (float*)p;
  int rc = launch_bwd_points(origins, dirs, depths_coarse, depths_fine, Dc, Df, rays, pts, di.sms, st);
  if (rc != 0) return cuda_fail((cudaError_t)rc, "points_kernel");
  const float* col_in = sample_colours; const float* sig_in = sample_sigma;
  const int col_chunked = sample_colours != nullptr ? 1 : 0;      // tpr_render_train's layout; recomputed colours are sample-major
  if (!col_in) {
    // not kept by the forward (tpr_render_train): colours and densities of every sample through the forward's point query
    // (VR/renderer.py:142-148)
    rc = launch_run_model(false, planes_packed, n_img, P, height, width, decoder_packed, pts, (int64_t)n_rays * S, opt->box_warp,
                          colours, sigma, mlp, stream);
    if (rc != 0) return rc;
    col_in = colours; sig_in = sigma;
  }
  // a group of k >= n_img cameras is the whole call: min(k, n_img) rays_per_img keeps the group size <= the rays (< 2^32)
  const long long group_rays = opt->depth_clamp_group > 0 ? (opt->depth_clamp_group < n_img ? (long long)opt->depth_clamp_group : (long long)n_img) * n_rays : 0;
  rc = launch_bwd_march(depths_coarse, depths_fine, Dc, Df, sig_in, col_in, col_chunked, g_rgb, g_depth, g_weight_sum, depth_range,
                        group_rays, opt->white_back, rays, gsig, omega, di.sms, st);
  if (rc != 0) return cuda_fail((cudaError_t)rc, "march_backward_kernel");
  DetScratch ds = det_scratch(scratch, base_bytes);
  return decoder_backward(planes_packed, P, height, width, decoder_packed, pts, col_in, col_chunked, sample_features, gsig, omega,
                          g_rgb, (long long)T, (long long)n_rays * S, S, 0, (float)(2.0 / opt->box_warp), mlp == TPR_MLP_BF16,
                          g_planes_packed, g_decoder_packed, scale_buf, scratch, det ? &ds : nullptr, di, st);
}

// ---------------------------------------------------------------------------------------
// backward of tpr_run_model (ImportanceRenderer.run_model under autograd): the decoder backward kernels of tpr_render_backward
// in their point-query mode -- no march, no sort; the features are gathered again
// ---------------------------------------------------------------------------------------
size_t tpr_run_model_backward_scratch_bytes(int64_t n_img, int64_t n_pts) {
  if (n_img <= 0 || n_pts <= 0) return 0;
  // a zero g_sigma row [T] (used when g_sigma is NULL), the operand scale of the tcgen05 decoder backward
  return align256((size_t)n_img * (size_t)n_pts * 4) + 256;
}

int tpr_run_model_backward(const float* planes_packed, int64_t n_img, int32_t height, int32_t width, const float* decoder_packed,
                           const float* xyz, int64_t n_pts, double box_warp, const float* rgb, const float* g_rgb,
                           const float* g_sigma, int32_t flags, float* g_planes_packed, float* g_decoder_packed, void* scratch,
                           size_t scratch_bytes, void* stream) {
  if (g_rgb && !rgb) return fail(TPR_E_NULL, "tpr_run_model_backward: g_rgb needs the forward's rgb");
  if (!g_rgb && !g_sigma) return fail(TPR_E_NULL, "tpr_run_model_backward: g_rgb and g_sigma are both NULL");
  if (!planes_packed || !decoder_packed || !xyz || (!g_planes_packed && !g_decoder_packed) || !scratch)
    return fail(TPR_E_NULL, "tpr_run_model_backward: NULL pointer");
  if (n_img <= 0 || n_pts <= 0 || height <= 0 || width <= 0) return fail(TPR_E_SHAPE, "tpr_run_model_backward: bad shape");
  if ((long long)3 * height * width * kC >= (1ll << 32)) return fail(TPR_E_SHAPE, "tpr_run_model_backward: planes too large");
  if (!(box_warp > 0)) return fail(TPR_E_OPTION, "tpr_run_model_backward: box_warp must be > 0");
  const bool det = (flags & TPR_BWD_DETERMINISTIC) != 0;
  flags &= ~TPR_BWD_DETERMINISTIC;
  if (flags != TPR_MLP_FP32 && flags != TPR_MLP_BF16 && flags != TPR_MLP_FFMA)
    return fail(TPR_E_OPTION, "tpr_run_model_backward: unknown decoder flag");
  const size_t base_bytes = tpr_run_model_backward_scratch_bytes(n_img, n_pts);
  if (scratch_bytes < base_bytes + (det ? tpr_backward_deterministic_scratch_bytes(n_img, height, width) : 0))
    return fail(TPR_E_SCRATCH, "tpr_run_model_backward: scratch too small");
  DeviceInfo di = device_info();
  if (!di.ok) return fail(TPR_E_DEVICE, "tpr_run_model_backward: no CUDA device");
  cudaStream_t st = (cudaStream_t)stream;
  const long long T = (long long)n_img * n_pts;
  float* zero_gsig = (float*)scratch;
  float* scale_buf = (float*)((uint8_t*)scratch + align256((size_t)T * 4));
  if (!g_sigma) {
    const cudaError_t e = cudaMemsetAsync(zero_gsig, 0, (size_t)T * sizeof(float), st);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
  }
  const float* gsig = g_sigma ? g_sigma : zero_gsig;
  const float box_scale = (float)(2.0 / box_warp);      // python float (VR/renderer.py:61)
  DetScratch ds = det_scratch(scratch, base_bytes);
  return decoder_backward(planes_packed, (int)n_img, height, width, decoder_packed, xyz, rgb, 0, nullptr, gsig, nullptr, g_rgb, T, n_pts, 1, 1,
                          box_scale, flags == TPR_MLP_BF16, g_planes_packed, g_decoder_packed, scale_buf, scratch, det ? &ds : nullptr,
                          di, st);
}

int tpr_unpack_decoder_grad(const float* g_decoder_packed, float w1_gain, float b1_gain, float w2_gain, float b2_gain, float* g_w1,
                            float* g_b1, float* g_w2, float* g_b2, void* stream) {
  if (!g_decoder_packed || !g_w1 || !g_b1 || !g_w2 || !g_b2) return fail(TPR_E_NULL, "tpr_unpack_decoder_grad: NULL pointer");
  const int rc = launch_unpack_decoder_grad(g_decoder_packed, w1_gain, b1_gain, w2_gain, b2_gain, g_w1, g_b1, g_w2, g_b2,
                                            (cudaStream_t)stream);
  if (rc != 0) return cuda_fail((cudaError_t)rc, "unpack_decoder_grad_kernel");
  return 0;
}

}  // extern "C"
