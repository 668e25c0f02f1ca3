// Decoder backward + plane-gradient scatter of the renderer's backward pass on tcgen05 (sm_100a), warp-specialised.
// Replaces the mma.sync (HMMA) kernel of tpr_backward.cu: all five GEMMs of the decoder's backward run on the 5th-gen tensor
// cores with 2xFP16 operands (x = hi + lo in fp16, three products, fp32 accumulation in TMEM -- the forward's scheme, see
// tpr_ws.cuh), the per-sample gradients never leave the SM, and loading / MMA issue / epilogues / atomic scatter overlap.
//
// Per tile of 128 samples (TMEM lane = sample):
//   G1  A  = F . W1t + b1            M = samples, N = 64,  K = 32   (layer 1 forward again: H = softplus(A), S' = sigmoid(A))
//   G2  GH = GYc . W2c               M = samples, N = 64,  K = 32   (d/d hidden from the 32 colour logits; the sigma column of
//                                                                   GY is a rank-1 term added by the epilogue in fp32)
//       GA = GH (.) S'
//   G3  GF = GA . W1t^T              M = samples, N = 32,  K = 64   (d/d features -> scattered to the 12 texels of the sample)
//   WG  [GA ; H]^T . [F | GYc | gs]  M = 128 (64 hidden of GA stacked on 64 hidden of H), K = 128 samples:
//         rows 0..63   x F columns   = gW1t^T        rows 64..127 x GYc columns = gW2t (colour columns)
//         rows 0..63   x ones column = gb1           rows 64..127 x gsig column = gW2t (sigma column)
//       accumulated in TMEM over ALL tiles of the CTA and flushed once.  The operands of WG are the SAME shared-memory
//       tiles G1-G3 use: a tile stored as [sample rows][128 bytes of fp16] with the 128-byte swizzle is K-major for a GEMM
//       whose K runs along the row and MN-major for one whose K runs over the rows (instruction descriptor bits 15 / 16).
//       The inputs of a tile are three swizzle atoms 16 KB apart, [F lo | GYc lo], [F hi | GYc hi], [gsig hi, lo, one]: one B
//       operand of N = 144 for the hi half of [GA ; H] and of N = 80 (from the second atom) for its lo half -- two MMAs per 16
//       samples (every MMA re-reads its 4 KB A slice from shared memory, so few wide MMAs beat many narrow ones).
//
// What bounds it (profiles/r02_scatter_shapes.json, TPR_BWD_PROFILE=1): the scatter.  12 texels x 128 bytes of
// red.global.add per sample run at ~6 TB/s when the gradient of one image's planes (25 MB) is L2 resident -- the tiles are
// handed out so that all CTAs work on the same image -- which is 3.1-3.3 ms for config 2's 151 M lines.
//
// Gradient-side operands (GY, GA) are multiplied by a power of two chosen from the upstream gradient's magnitude (a tiny
// range kernel) before they are split into fp16 halves, and the results are scaled back exactly: fp16 has 5 exponent bits
// and gradients come at any scale (loss scaling).
//
// Point queries (ImportanceRenderer.run_model under autograd; kPoint = true): the same kernel with the input rows indexed by
// point instead of by ray -- colours = the forward's rgb [T,32], g_rgb [T,32], GYc = g_rgb x 1.002 x s(1-s) (the render formula
// with ray = point and omega = 1/2), gsig = the upstream gradient of sigma (density_noise is additive).  With g_rgb == NULL
// (sigma-only queries) the LOAD warps read no colours and the GYc halves of the input tiles stay the zeros written at start.
//
// Roles (25 warps, one CTA per SM):  0-7 LOAD (features / colours / upstream gradient -> operand tiles)
//                                     8-15 SCATTER (the sample's 12 taps from its position, red.global.add.v4.f32 of GF x tap
//                                           weight; one texel = one 128-byte line = eight lanes.  kDet: four
//                                           red.global.add.u64 of the fixed-point value per lane and texel instead)
//                                     16-23 EPILOGUE (TMEM -> softplus / products -> operand tiles; GF -> shared memory): two
//                                           warps per TMEM lane quarter, 32 hidden units each
//                                     24 MMA issuer
// Citations relative to /root/reference/g_nerf/ (VR/ = training/volumetric_rendering/).
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <stdlib.h>
#include <stdio.h>
#include <cuda_fp16.h>
#include "triplane_b200.h"
#include "tpr_device.cuh"
#include "tpr_tc.cuh"

namespace tpr {
namespace bwdtc {
using namespace tc;

constexpr int kM = 128;                              // samples per tile
constexpr int kLoadWarps = 8, kScatWarps = 8, kEpiWarps = 8;
constexpr int kThreads = 32 * (kLoadWarps + kScatWarps + kEpiWarps + 1);      // 800
constexpr int kTile = kM * 128;                      // one operand tile: 128 rows x 128 bytes
// TMEM columns
constexpr uint32_t cD1 = 0, cGH = 64, cGF = 128, cW = 192;     // cW: 144 columns = [F lo | GYc lo | F hi | GYc hi | gsig hi, gsig lo, one, 0 ...]

struct __align__(1024) Smem {
  uint8_t w1k[64 * 128];            // G1 B: row n (hidden) = [W1t[.][n] hi, k = 0..31 | lo]
  uint8_t w2c[64 * 128];            // G2 B: row j (hidden) = [W2t[j][1 + c] hi, c = 0..31 | lo]
  uint8_t w1g[2][32 * 128];         // G3 B: [hi, lo] row k (channel) = W1t[k][j], j = 0..63
  // the inputs of a tile, double buffered: three 64-column swizzle atoms 16 KB apart.  Read K-major (rows = samples) by G1 / G2
  // and MN-major, as ONE B operand of N = 144 (lo, hi, sig) or N = 80 (hi, sig), by the weight-gradient MMAs
  struct In {
    uint8_t lo[kTile];              // [F lo | GYc lo]  (32 + 32 fp16 per sample; GYc scaled)
    uint8_t hi[kTile];              // [F hi | GYc hi]
    uint8_t sig[kTile];             // [gsig hi, gsig lo, one, 0 x 13 | unused]
  } in[2];
  uint8_t ga_hi[kTile], h_hi[kTile];   // stacked: MN-major A of WG, M = 128 = GA (64) then H (64); GA also the K-major A of G3
  uint8_t ga_lo[kTile], h_lo[kTile];
  float gf[2][kM * 32];             // d/d features of a tile, 16-byte chunks XOR-swizzled by (row & 7); double buffered
  float gsig[2][kM];                // scaled d/d sigma (the epilogue's rank-1 term)
  float b1[64], w2s[64];
  uint64_t in_full[2], in_free[2], g12_done, hga_ready, g3_done, gf_ready[2], gf_free[2], wg_done, all_done;
  uint32_t tmem_base;
};

struct Args {
  const float* planes; int H, W;        // packed [P,3,H,W,32]: image n samples plane set n % n_sets
  const float* dec;                     // packed decoder
  const float* pts;                     // [T,3]
  const float* colours;                 // [T,32], or (col_chunked != 0) [rays, 8, S, 4] as tpr_render_train keeps them
  int col_chunked;
  const float* features;                // [T,32] kept by the forward, or NULL: gather again
  const float* gsig; const float* omega;// [T] (point queries: omega unused)
  const float* g_rgb;                   // [rays,32]; point queries: [T,32] or NULL (sigma only)
  long long total, pts_per_img; int S;
  float box_scale;
  float* g_planes;                      // packed, zero-initialised; NULL: no scatter
  float* g_dec;                         // [kDecFloats], zero-initialised; NULL: no weight gradients
  const float* scale;                   // [2] device: power-of-two scale of the gradient-side operands and its inverse
  int lookahead;                        // G1 + G2 of tile i + 1 ahead of the weight-gradient MMAs of tile i
  long long* prof;                      // TPR_BWD_PROFILE: cycles CTA 0 spends per role and wait (NULL: off)
  // kDet (deterministic mode): the plane gradient goes to g_acc in fixed point (scale 2^e from det_hdr), the decoder gradient
  // to this CTA's row of dec_rows; g_planes / g_dec only say whether each is wanted
  unsigned long long* g_acc; float* dec_rows; int* det_hdr;
  int n_sets;                           // plane sets in planes / g_planes / g_acc
};

// ---- descriptors -------------------------------------------------------------------------------------------------
// addr16 / lbo16 / sbo16 in 16-byte units; layout 2 = SWIZZLE_128B, 0 = none
__device__ __forceinline__ uint64_t make_desc(uint32_t addr16, uint32_t lbo16, uint32_t sbo16, uint32_t layout) {
  return (uint64_t)(addr16 & 0x3fffu) | ((uint64_t)(lbo16 & 0x3fffu) << 16) | ((uint64_t)(sbo16 & 0x3fffu) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)layout << 61);
}
constexpr uint32_t kMajorMN = (1u << 15) | (1u << 16);       // instruction descriptor: A and B MN-major

__device__ __forceinline__ uint32_t pack_f16x2(float lo_elem, float hi_elem) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi_elem), "f"(lo_elem));
  return r;
}
__device__ __forceinline__ void unpack_f16x2(uint32_t v, float& lo_elem, float& hi_elem) {
  const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&v));
  lo_elem = f.x; hi_elem = f.y;
}
__device__ __forceinline__ void st_f16(uint8_t* tile, int row, int k, float v) {        // swizzled 128-byte rows of 64 fp16
  reinterpret_cast<__half*>(tile)[row * 64 + ((((k >> 3) ^ (row & 7)) << 3) | (k & 7))] = __float2half_rn(v);
}
// four fp32 values (columns 4 sub .. 4 sub + 3 of a 32-column block) -> 8 bytes of the hi tile's row and 8 bytes of the lo tile's,
// in the block that starts at 16-byte chunk `chunk0` (0: features, 4: colour-logit gradients)
__device__ __forceinline__ void st_hilo4(uint8_t* hi_tile, uint8_t* lo_tile, int row, int chunk0, int sub, float4 v) {
  const uint2 hi = make_uint2(pack_f16x2(v.x, v.y), pack_f16x2(v.z, v.w));
  float h0, h1, h2, h3;
  unpack_f16x2(hi.x, h0, h1); unpack_f16x2(hi.y, h2, h3);
  const uint2 lo = make_uint2(pack_f16x2(v.x - h0, v.y - h1), pack_f16x2(v.z - h2, v.w - h3));
  const int off = row * 128 + ((sub & 1) << 3) + (((chunk0 + (sub >> 1)) ^ (row & 7)) << 4);
  *reinterpret_cast<uint2*>(hi_tile + off) = hi;
  *reinterpret_cast<uint2*>(lo_tile + off) = lo;
}
// 16 fp32 values (hidden units [16 c, 16 c + 16) of row `row`) -> 32 bytes of a hi tile and of a lo tile (64 fp16 per row)
__device__ __forceinline__ void st_hilo16(uint8_t* hi_tile, uint8_t* lo_tile, int row, int c, const float (&v)[16]) {
  uint32_t hi[8], lo[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float a, b;
    hi[i] = pack_f16x2(v[2 * i], v[2 * i + 1]);
    unpack_f16x2(hi[i], a, b);
    lo[i] = pack_f16x2(v[2 * i] - a, v[2 * i + 1] - b);
  }
#pragma unroll
  for (int hh = 0; hh < 2; ++hh) {
    const int off = row * 128 + (((2 * c + hh) ^ (row & 7)) << 4);
    *reinterpret_cast<uint4*>(hi_tile + off) = make_uint4(hi[4 * hh], hi[4 * hh + 1], hi[4 * hh + 2], hi[4 * hh + 3]);
    *reinterpret_cast<uint4*>(lo_tile + off) = make_uint4(lo[4 * hh], lo[4 * hh + 1], lo[4 * hh + 2], lo[4 * hh + 3]);
  }
}

// ---- the range kernel: power-of-two scale for the gradient-side operands -----------------------------------------------
__global__ void scale_kernel(const float* __restrict__ g_rgb, long long n_rgb, const float* __restrict__ gsig, long long n_sig,
                             const float* __restrict__ dec, unsigned* __restrict__ acc /*[2], zeroed*/) {
  float mg = 0.f, ms = 0.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n_rgb; i += (long long)gridDim.x * blockDim.x) mg = fmaxf(mg, fabsf(g_rgb[i]));
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n_sig; i += (long long)gridDim.x * blockDim.x) ms = fmaxf(ms, fabsf(gsig[i]));
  mg = warp_max(mg); ms = warp_max(ms);
  if ((threadIdx.x & 31) == 0) { atomicMax(acc, __float_as_uint(mg)); atomicMax(acc + 1, __float_as_uint(ms)); }   // (non-negative floats order as uints)
  (void)dec;
}
__global__ void scale_finish_kernel(const unsigned* __restrict__ acc, const float* __restrict__ dec, float* __restrict__ scale) {
  // bound of |GYc| = |g_rgb| * 2 * 1.002 * omega * s(1-s) <= 0.501 |g_rgb| (point queries: 1.002 s(1-s) <= 0.2505); of |GH| = |GYc| . sum_c |W2c| + |gsig| |w2s|
  __shared__ float col[64];
  const int j = threadIdx.x;
  if (j < 64) {
    float sum = 0.f;
    for (int c = 0; c < 32; ++c) sum += fabsf(dec[kW2tOff + j * kOutPad + 1 + c]);
    col[j] = sum;
  }
  __syncthreads();
  if (j == 0) {
    const float mg = __uint_as_float(acc[0]) * 0.501f, ms = __uint_as_float(acc[1]);
    float wc = 0.f, wsig = 0.f;
    for (int i = 0; i < 64; ++i) { wc = fmaxf(wc, col[i]); wsig = fmaxf(wsig, fabsf(dec[kW2tOff + i * kOutPad])); }
    const float bound = fmaxf(fmaxf(mg, ms), mg * wc + ms * wsig);
    float sc = 1.0f;
    if (bound > 0.f && bound < 3.0e38f) {
      int e;
      frexpf(bound, &e);                       // bound = m * 2^e, m in [0.5, 1)
      int k = 13 - e;                          // scaled bound < 2^13: fp16 headroom of 8 for sums the bound does not cover
      k = max(-100, min(100, k));
      sc = ldexpf(1.0f, k);
    }
    scale[0] = sc; scale[1] = 1.0f / sc;
  }
}

// Deterministic mode: the fixed-point exponent e of the plane-gradient accumulator.  |GF_k| <= max|GA| . sum_j |W1t[k][j]|
// and |GA| <= |GH| (softplus' <= 1) <= mg wc + ms wsig (the bound of scale_finish_kernel); a texel takes at most K samples'
// contributions with tap weights of sum <= 1 per plane, so its sum is at most K . bound_GF and e = 62 - ceil(log2(K . bound_GF))
// cannot overflow.  K = the samples that share one plane set: total / n_sets (with several images per set, F images add into
// the same texels).  The bound scales exactly with the upstream gradient, so 2^k x the upstream gradient gives e - k and the
// same integers.  A non-finite bound (inf upstream) or one whose e would leave the fp32 range marks the result NaN.
__global__ void det_bound_kernel(const unsigned* __restrict__ acc, const float* __restrict__ dec, long long K, int* __restrict__ hdr) {
  __shared__ float col[64], row[32];
  const int j = threadIdx.x;
  if (j < 64) {
    float sum = 0.f;
    for (int c = 0; c < 32; ++c) sum += fabsf(dec[kW2tOff + j * kOutPad + 1 + c]);
    col[j] = sum;
  }
  if (j < 32) {
    float sum = 0.f;
    for (int i = 0; i < 64; ++i) sum += fabsf(dec[kW1tOff + j * kHid + i]);
    row[j] = sum;
  }
  __syncthreads();
  if (j == 0) {
    const float mg = __uint_as_float(acc[0]) * 0.501f, ms = __uint_as_float(acc[1]);
    float wc = 0.f, wsig = 0.f, w1 = 0.f;
    for (int i = 0; i < 64; ++i) { wc = fmaxf(wc, col[i]); wsig = fmaxf(wsig, fabsf(dec[kW2tOff + i * kOutPad])); }
    for (int k = 0; k < 32; ++k) w1 = fmaxf(w1, row[k]);
    const double bound = ((double)mg * wc + (double)ms * wsig) * (double)w1 * (double)K;
    int e = 0, bad = !isfinite(bound);
    if (!bad && bound > 0.0) {
      int x;
      const double m = frexp(bound, &x);       // bound = m 2^x, m in [0.5, 1): ceil(log2(bound)) = x, or x - 1 when m = 0.5
      e = 62 - (m == 0.5 ? x - 1 : x);
      if (e < -126) { bad = 1; e = 0; }
      e = min(e, 127);                         // a tiny bound: 2^127 keeps every contribution far below 2^62
    }
    hdr[0] = e; hdr[1] = bad; hdr[2] = __float_as_int(ldexpf(1.0f, e));
  }
}

// TPR_BWD_PROFILE=1: CTA 0 adds the cycles each role's first warp spends in every wait / work phase to prof[slot]
// (kProf instantiation only; accumulated in registers, written once at the end of the role)
#define PROF_DECL() long long prof_t = 0, prof_acc[17]; if (kProf) { for (int k_ = 0; k_ < 17; ++k_) prof_acc[k_] = 0; }
#define PROF_T0() do { if (kProf) prof_t = clock64(); } while (0)
#define PROF(slot) do { if (kProf) { const long long t1_ = clock64(); prof_acc[slot] += t1_ - prof_t; prof_t = t1_; } } while (0)
#define PROF_FLUSH(first, last, cond) do { if (kProf && blockIdx.x == 0 && lane == 0 && (cond)) { for (int k_ = first; k_ <= last; ++k_) a.prof[k_] = prof_acc[k_]; } } while (0)
// ---- the kernel ------------------------------------------------------------------------------------------------------------
// kDet: the deterministic mode (Args::g_acc); the launch then has kLoadWarps x 33 floats of dynamic shared memory past Smem
template <bool kProf, bool kPoint, bool kDet = false>
__global__ void __launch_bounds__(kThreads, 1) decode_backward_tc_kernel(const Args a) {
  extern __shared__ uint8_t smem_raw[];
  Smem& s = *reinterpret_cast<Smem*>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  const bool want_planes = a.g_planes != nullptr, want_dec = a.g_dec != nullptr;
  const float sc = __ldg(a.scale), inv_sc = __ldg(a.scale + 1);

  // ---- one-time setup: barriers, TMEM, decoder operands
  if (tid == 0) {
    for (int b = 0; b < 2; ++b) {
      mbar_init(&s.in_full[b], kLoadWarps); mbar_init(&s.in_free[b], 1);
    }
    mbar_init(&s.g12_done, 1); mbar_init(&s.hga_ready, kEpiWarps); mbar_init(&s.g3_done, 1);
    mbar_init(&s.gf_ready[0], kEpiWarps); mbar_init(&s.gf_ready[1], kEpiWarps); mbar_init(&s.gf_free[0], kScatWarps);
    mbar_init(&s.gf_free[1], kScatWarps); mbar_init(&s.wg_done, 1); mbar_init(&s.all_done, 1);
    fence_mbar_init();
  }
  if (warp == 0) { tmem_alloc(&s.tmem_base, 512); tmem_relinquish(); }
  for (int i = tid; i < 64 * 32; i += kThreads) {            // W1t[k][n]: G1's B (row n: K = k), G3's B (row k: K = n)
    const int n = i >> 5, k = i & 31;
    const float w = __ldg(a.dec + kW1tOff + k * kHid + n);
    const __half hi = __float2half_rn(w), lo = __float2half_rn(w - __half2float(hi));
    reinterpret_cast<__half*>(s.w1k)[n * 64 + ((((k >> 3) ^ (n & 7)) << 3) | (k & 7))] = hi;
    reinterpret_cast<__half*>(s.w1k)[n * 64 + (((((32 + k) >> 3) ^ (n & 7)) << 3) | (k & 7))] = lo;
    reinterpret_cast<__half*>(s.w1g[0])[k * 64 + ((((n >> 3) ^ (k & 7)) << 3) | (n & 7))] = hi;
    reinterpret_cast<__half*>(s.w1g[1])[k * 64 + ((((n >> 3) ^ (k & 7)) << 3) | (n & 7))] = lo;
  }
  for (int i = tid; i < 64 * 32; i += kThreads) {            // W2t[j][1 + c]: G2's B (row j: K = c)
    const int j = i >> 5, c = i & 31;
    const float w = __ldg(a.dec + kW2tOff + j * kOutPad + 1 + c);
    const __half hi = __float2half_rn(w), lo = __float2half_rn(w - __half2float(hi));
    reinterpret_cast<__half*>(s.w2c)[j * 64 + ((((c >> 3) ^ (j & 7)) << 3) | (c & 7))] = hi;
    reinterpret_cast<__half*>(s.w2c)[j * 64 + (((((32 + c) >> 3) ^ (j & 7)) << 3) | (c & 7))] = lo;
  }
  if (tid < 64) { s.b1[tid] = __ldg(a.dec + kB1Off + tid); s.w2s[tid] = __ldg(a.dec + kW2tOff + tid * kOutPad); }
  if (kPoint && a.g_rgb == nullptr) {                         // sigma-only: the GYc halves (chunks 4-7 of every row) stay zero
    for (int i = tid; i < 2 * 2 * kM * 4; i += kThreads) {
      const int row = (i >> 2) & (kM - 1), tile = i >> 9;      // tile: buffer b = tile >> 1, hi / lo = tile & 1
      uint8_t* t = (tile & 1) ? s.in[tile >> 1].lo : s.in[tile >> 1].hi;
      *reinterpret_cast<uint4*>(t + row * 128 + (((4 + (i & 3)) ^ (row & 7)) << 4)) = make_uint4(0u, 0u, 0u, 0u);
    }
  }
  fence_proxy_async_smem();
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = s.tmem_base;

  const long long n_tiles = (a.total + kM - 1) / kM;
  const int G = (int)((n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x);     // tiles of this CTA: blockIdx.x + i * gridDim.x
  const size_t img_stride = (size_t)3 * a.H * a.W * kC;

  if (warp < kLoadWarps) {
    // ================================================ LOAD ================================================
    // Eight lanes per sample, 16 samples per warp: two halves of two passes each, the global loads of a half issued together
    // (the first half's before the wait for the operand buffer).  Measured alternatives at config 2, same box: all four passes'
    // loads up front (needs the upstream gradient read at use to stay under the CTA's 72 registers per thread) 8.32 vs 7.92 ms
    // for the train step; prefetch.global.L2 of the next tile's rows: no change (7.86 vs 7.83); setmaxnreg.inc for these warps
    // without a matching .dec elsewhere never returns.
    // Colours use their own lane mapping: a thread owns ONE sample per half (slot cs of eight consecutive samples) and two
    // 4-channel chunks (cq, cq + 4), so that a load instruction reads 4 chunks x 8 consecutive samples x 16 B = four full lines
    // of the chunk-major layout tpr_render_train keeps the colours in (eight lanes per sample would touch eight lines for the
    // same bytes: +0.19 ms for the kernel).
    const int grp = lane >> 3, sub = lane & 7;       // features: eight lanes per sample row
    const int cs = lane & 7, cq = lane >> 3;          // colours: sample slot, first chunk
    float b2acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};   // (scaled) colour-logit gradient sums: channels 4 (cq + 4 j) + k
    float b2sig = 0.f;
    PROF_DECL();
    for (int i = 0; i < G; ++i) {
      const int b = i & 1;
      const long long gs0 = ((long long)blockIdx.x + (long long)i * gridDim.x) * kM;
      PROF_T0();
      // tile-uniform index arithmetic once (64-bit divisions), 32-bit per sample: a tile straddles at most two images when an
      // image has >= 128 points (the launcher checks that), and (rr0 + sr) / S is a 32-bit division
      const long long n0 = gs0 / a.pts_per_img, rem0 = gs0 - n0 * a.pts_per_img;
      long long ray0 = 0;
      unsigned rr0 = 0;
      if (!kPoint) { ray0 = gs0 / a.S; rr0 = (unsigned)(gs0 - ray0 * a.S); }
      const bool want_col = !kPoint || a.g_rgb != nullptr;    // (warp-uniform)
      float4 f[2], colq[2], Aq[2];
#pragma unroll 1
      for (int half = 0; half < 2; ++half) {
#pragma unroll
      for (int it = 0; it < 2; ++it) {
        const int sr = warp * 16 + (2 * half + it) * 4 + grp;
        const long long gs = gs0 + sr;
        f[it] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (gs < a.total) {
          if (a.features != nullptr) {
            f[it] = __ldg(reinterpret_cast<const float4*>(a.features + gs * 32) + sub);
          } else {                                 // not kept by the forward: gather again (VR/renderer.py:39-65)
            const float px = __fmul_rn(__ldg(a.pts + 3 * gs + 0), a.box_scale), py = __fmul_rn(__ldg(a.pts + 3 * gs + 1), a.box_scale),
                        pz = __fmul_rn(__ldg(a.pts + 3 * gs + 2), a.box_scale);
            int n = (int)n0 + (rem0 + sr >= a.pts_per_img ? 1 : 0);
            // plane set n % n_sets, reduced only past the first n_sets images: a set index held across the tile (as the
            // scatter does) costs these warps spill traffic at their 72-register budget
            if (!kPoint && n >= a.n_sets) n = (int)((unsigned)n % (unsigned)a.n_sets);
            f[it] = gather_point(a.planes + (size_t)n * img_stride, a.H, a.W, px, py, pz, sub);
          }
        }
      }
      const int src = warp * 16 + 8 * half + cs;            // this thread's sample of the half
      const long long gsc = gs0 + src;
      float omq = 0.f, gsq = 0.f;
      colq[0] = colq[1] = Aq[0] = Aq[1] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (gsc < a.total) {
        const long long ray = kPoint ? gsc : ray0 + (rr0 + (unsigned)src) / (unsigned)a.S;     // the row of g_rgb
        if (want_col) {
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const int chunk = cq + 4 * j;
            colq[j] = (!kPoint && a.col_chunked)
                ? __ldg(reinterpret_cast<const float4*>(a.colours + ray * a.S * 32) + chunk * a.S + (gsc - ray * a.S))
                : __ldg(reinterpret_cast<const float4*>(a.colours + gsc * 32) + chunk);
            Aq[j] = __ldg(reinterpret_cast<const float4*>(a.g_rgb + ray * 32) + chunk);
          }
        }
        if (!kPoint) omq = __ldg(a.omega + gsc);
        gsq = __ldg(a.gsig + gsc);
      }
      PROF(0);
      if (half == 0) mbar_wait_parked(&s.in_free[b], ((uint32_t)(i >> 1) & 1u) ^ 1u);   // the weight-gradient MMAs of tile i - 2 have read the tiles
      PROF(2);
#pragma unroll
      for (int it = 0; it < 2; ++it) st_hilo4(s.in[b].hi, s.in[b].lo, warp * 16 + (2 * half + it) * 4 + grp, 0, sub, f[it]);
      {
        // rgb*2-1 (VR/ray_marcher.py:55), sigmoid*1.002 (training/triplane.py:134); times the operand scale
        const float om = kPoint ? 1.002f * sc : omq * (2.0f * 1.002f) * sc;
        const float gsg = gsq * sc;
#pragma unroll
        for (int j = 0; j < 2 && want_col; ++j) {
          const float cc[4] = {colq[j].x, colq[j].y, colq[j].z, colq[j].w}, aa[4] = {Aq[j].x, Aq[j].y, Aq[j].z, Aq[j].w};
          float g4[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float sv = (cc[k] + 0.001f) * (1.0f / 1.002f);           // sigmoid(logit)
            g4[k] = aa[k] * om * sv * (1.0f - sv);
            b2acc[j][k] += g4[k];
          }
          st_hilo4(s.in[b].hi, s.in[b].lo, src, 4, cq + 4 * j, make_float4(g4[0], g4[1], g4[2], g4[3]));
        }
        if (cq == 0) {
          b2sig += gsg;
          s.gsig[b][src] = gsg;
          // the third atom: columns (gsig hi, gsig lo, one, 0 ...) of this sample's row, 16-byte chunks 0 and 1
          const __half hi = __float2half_rn(gsg), lo = __float2half_rn(gsg - __half2float(hi));
          const uint32_t w0 = (uint32_t)__half_as_ushort(hi) | ((uint32_t)__half_as_ushort(lo) << 16);
          const uint32_t w1 = gsc < a.total ? 0x3c00u : 0u;               // fp16 1.0
          uint8_t* rowp = s.in[b].sig + src * 128;
          *reinterpret_cast<uint4*>(rowp + ((0 ^ (src & 7)) << 4)) = make_uint4(w0, w1, 0u, 0u);
          *reinterpret_cast<uint4*>(rowp + ((1 ^ (src & 7)) << 4)) = make_uint4(0u, 0u, 0u, 0u);
        }
      }
      PROF(3);
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s.in_full[b]);
    }
    PROF_FLUSH(0, 3, warp == 0);
    // gb2 (the bias of layer 2): sums of the outputs' gradients
    if constexpr (!kDet) {
    if (want_dec) {
#pragma unroll
      for (int j = 0; j < 2; ++j) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          float v = b2acc[j][k];
          v += __shfl_xor_sync(kFull, v, 1); v += __shfl_xor_sync(kFull, v, 2); v += __shfl_xor_sync(kFull, v, 4);
          if (cs == 0) atomicAdd(a.g_dec + kB2Off + 1 + 4 * (cq + 4 * j) + k, v * inv_sc);
        }
      }
      b2sig = warp_sum(b2sig);
      if (lane == 0) atomicAdd(a.g_dec + kB2Off, b2sig * inv_sc);
    }
    } else if (want_dec) {
      // deterministic: the eight warps' partials meet in shared memory and warp 0 adds them in warp order
      float* part = reinterpret_cast<float*>(&s + 1);          // [kLoadWarps][33]
#pragma unroll
      for (int j = 0; j < 2; ++j) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          float v = b2acc[j][k];
          v += __shfl_xor_sync(kFull, v, 1); v += __shfl_xor_sync(kFull, v, 2); v += __shfl_xor_sync(kFull, v, 4);
          if (cs == 0) part[warp * 33 + 1 + 4 * (cq + 4 * j) + k] = v;
        }
      }
      b2sig = warp_sum(b2sig);
      if (lane == 0) part[warp * 33] = b2sig;
      asm volatile("bar.sync 1, %0;" ::"n"(kLoadWarps * 32) : "memory");
      if (warp == 0) {
        float* row = a.dec_rows + (size_t)blockIdx.x * kDecFloats;
        for (int l = lane; l < 33; l += 32) {
          float t = 0.f;
#pragma unroll
          for (int w = 0; w < kLoadWarps; ++w) t += part[w * 33 + l];
          row[kB2Off + l] = t * inv_sc;
        }
      }
    }
  } else if (warp < kLoadWarps + kScatWarps) {
    // ================================================ SCATTER ================================================
    // Eight lanes per sample add GF x tap weight to the twelve texels of the sample (one 128-byte line each).  The taps are
    // recomputed here from the sample's position, loaded before the wait for GF.
    // (Handing a quarter of the rows to the epilogue warps, which idle for half of a tile's time, was measured SLOWER: 7.9 vs
    // 7.27 ms fwd+bwd.  The reductions are bound by the SM's own REDG rate -- ~0.74 cycles per 16-byte lane operation -- not by
    // how many warps issue them, and the epilogue's share lengthened the MMA <-> epilogue chain.)
    const int sw = warp - kLoadWarps, grp = lane >> 3, sub = lane & 7;
    const int plane_stride = a.H * a.W * kC;
    PROF_DECL();
    for (int i = 0; i < G; ++i) {
      const int b = i & 1;
      const long long gs0 = ((long long)blockIdx.x + (long long)i * gridDim.x) * kM;
      const long long n0 = gs0 / a.pts_per_img, rem0 = gs0 - n0 * a.pts_per_img;
      PROF_T0();
      float px[4], py[4], pz[4];
#pragma unroll
      for (int it = 0; it < 4; ++it) {
        const long long gs = gs0 + sw * 16 + it * 4 + grp;
        px[it] = py[it] = pz[it] = 0.f;
        if (want_planes && gs < a.total) { px[it] = __ldg(a.pts + 3 * gs + 0); py[it] = __ldg(a.pts + 3 * gs + 1); pz[it] = __ldg(a.pts + 3 * gs + 2); }
      }
      PROF(4);
      mbar_wait_parked(&s.gf_ready[b], (uint32_t)(i >> 1) & 1u);
      PROF(5);
      if (want_planes) {
        const int set0 = kPoint ? (int)n0 : (int)n0 % a.n_sets;    // the plane set of the tile's first image (see LOAD)
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          const int sr = sw * 16 + it * 4 + grp;
          if (gs0 + sr < a.total) {
            if constexpr (kDet) {
              // deterministic: GF x 2^e, four fixed-point reductions per lane and texel
              const float fx = __int_as_float(__ldg(a.det_hdr + 2));
              float4 gf = *reinterpret_cast<const float4*>(s.gf[b] + row_chunk_off(sr, sub));
              gf = make_float4(gf.x * fx, gf.y * fx, gf.z * fx, gf.w * fx);
              if (!fixed_ok(gf)) a.det_hdr[1] = 1;
              int n = set0 + (rem0 + sr >= a.pts_per_img ? 1 : 0);
              if (!kPoint && n == a.n_sets) n = 0;
              unsigned long long* img = a.g_acc + (size_t)n * img_stride + sub * 4;
              const float x = __fmul_rn(px[it], a.box_scale), y = __fmul_rn(py[it], a.box_scale), z = __fmul_rn(pz[it], a.box_scale);
#pragma unroll
              for (int p = 0; p < 3; ++p) {
                Taps tp;
                plane_taps(p == 2 ? z : x, p == 0 ? y : (p == 1 ? z : x), a.H, a.W, tp);
#pragma unroll
                for (int k = 0; k < 4; ++k)
                  if (tp.w[k] != 0.0f) {
                    unsigned long long* t = img + (unsigned)(p * plane_stride + tp.off[k]);
                    red_add_fixed(t, tp.w[k] * gf.x); red_add_fixed(t + 1, tp.w[k] * gf.y);
                    red_add_fixed(t + 2, tp.w[k] * gf.z); red_add_fixed(t + 3, tp.w[k] * gf.w);
                  }
              }
              continue;
            }
            const float4 gf = *reinterpret_cast<const float4*>(s.gf[b] + row_chunk_off(sr, sub));
            int n = set0 + (rem0 + sr >= a.pts_per_img ? 1 : 0);
            if (!kPoint && n == a.n_sets) n = 0;
            float* img = a.g_planes + (size_t)n * img_stride + sub * 4;
            const float x = __fmul_rn(px[it], a.box_scale), y = __fmul_rn(py[it], a.box_scale), z = __fmul_rn(pz[it], a.box_scale);
#pragma unroll
            for (int p = 0; p < 3; ++p) {
              Taps tp;
              plane_taps(p == 2 ? z : x, p == 0 ? y : (p == 1 ? z : x), a.H, a.W, tp);      // (x,y) (x,z) (z,x)
#pragma unroll
              for (int k = 0; k < 4; ++k)
                if (tp.w[k] != 0.0f)
                  atomicAdd(reinterpret_cast<float4*>(img + (unsigned)(p * plane_stride + tp.off[k])),
                            make_float4(tp.w[k] * gf.x, tp.w[k] * gf.y, tp.w[k] * gf.z, tp.w[k] * gf.w));
            }
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&s.gf_free[b]);
      PROF(6);
    }
    PROF_FLUSH(4, 6, sw == 0);
  } else if (warp < kLoadWarps + kScatWarps + kEpiWarps) {
    // ================================================ EPILOGUE ================================================
    const int q = warp & 3, hh = (warp - kLoadWarps - kScatWarps) >> 2;      // TMEM lane quarter (warps 16..23 -> 0..3, 0..3); hidden half
    const int row = q * 32 + lane;                            // the sample of this thread
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    PROF_DECL();
    for (int i = 0; i < G; ++i) {
      const int b = i & 1;
      PROF_T0();
      mbar_wait_parked(&s.g12_done, (uint32_t)i & 1u);
      PROF(7);
      tcgen05_fence_after();
      const float gsg = s.gsig[b][row];
#pragma unroll 1
      for (int c = 2 * hh; c < 2 * hh + 2; ++c) {
        uint32_t d1[16], gh[16];
        tmem_ld16(tmem + cD1 + lane_base + 16 * c, d1);
        tmem_ld16(tmem + cGH + lane_base + 16 * c, gh);
        tmem_wait_ld();
        float h[16], ga[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          const int j = 16 * c + k;
          const float x = __uint_as_float(d1[k]) + s.b1[j];
          const float e = __expf(x), d = 1.0f + e;
          h[k] = x > 20.0f ? x : __logf(d);                               // Softplus(beta=1, threshold=20)
          const float sp = x > 20.0f ? 1.0f : __fdividef(e, d);           // its derivative
          ga[k] = (__uint_as_float(gh[k]) + gsg * s.w2s[j]) * sp;         // d/d(layer-1 pre-activation), scaled
        }
        // the H / GA tiles are single buffered: the weight-gradient MMAs of the previous tile must have read them.  Waiting here,
        // after this chunk's TMEM loads and arithmetic, lets that work overlap those MMAs (G1 + G2 of this tile were issued
        // ahead of them)
        if (c == 2 * hh && i > 0) { mbar_wait_parked(&s.wg_done, (uint32_t)(i - 1) & 1u); PROF(8); }
        st_hilo16(s.h_hi, s.h_lo, row, c, h);
        st_hilo16(s.ga_hi, s.ga_lo, row, c, ga);
      }
      fence_proxy_async_smem();
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s.hga_ready);
      PROF(9);
      // ---- GF -> shared memory (unscaled), for the scatter warps
      mbar_wait_parked(&s.g3_done, (uint32_t)i & 1u);
      PROF(10);
      if (i > 1) mbar_wait_parked(&s.gf_free[b], (uint32_t)((i - 2) >> 1) & 1u);     // the scatter of tile i - 2 has read this buffer
      PROF(11);
      tcgen05_fence_after();
      {
        const int c = hh;                                     // this warp's 16 of the 32 channels
        uint32_t v[16];
        tmem_ld16(tmem + cGF + lane_base + 16 * c, v);
        tmem_wait_ld();
#pragma unroll
        for (int k4 = 0; k4 < 4; ++k4)
          *reinterpret_cast<float4*>(s.gf[b] + row_chunk_off(row, 4 * c + k4)) =
              make_float4(__uint_as_float(v[4 * k4]) * inv_sc, __uint_as_float(v[4 * k4 + 1]) * inv_sc,
                          __uint_as_float(v[4 * k4 + 2]) * inv_sc, __uint_as_float(v[4 * k4 + 3]) * inv_sc);
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s.gf_ready[b]);
      PROF(12);
    }
    PROF_FLUSH(7, 12, q == 0 && hh == 0);
    // ---- flush the weight gradients accumulated in TMEM: rows 0..63 = GA rows (gW1t, gb1), rows 64..127 = H rows (gW2t)
    if (want_dec && G > 0) {
      mbar_wait_parked(&s.all_done, 0u);
      tcgen05_fence_after();
      if constexpr (kDet) {
      const int j = row & 63;
      uint32_t v[16], u[16];
      // every element has one owning thread per CTA: deterministic mode stores it into the CTA's row
      float* drow = a.dec_rows + (size_t)blockIdx.x * kDecFloats;
      auto put = [&](int idx, float val) { drow[idx] = val; };
      if (row < 64) {
#pragma unroll 1
        for (int c = hh; c < hh + 1; ++c) {     // x F hi + x F lo: channels k = 16 c ..
          tmem_ld16(tmem + cW + lane_base + 64 + 16 * c, v);
          tmem_ld16(tmem + cW + lane_base + 16 * c, u);
          tmem_wait_ld();
#pragma unroll
          for (int k = 0; k < 16; ++k)
            put(kW1tOff + (16 * c + k) * kHid + j, (__uint_as_float(v[k]) + __uint_as_float(u[k])) * inv_sc);
        }
        tmem_ld16(tmem + cW + lane_base + 128, v);
        tmem_wait_ld();
        if (hh == 0) put(kB1Off + j, __uint_as_float(v[2]) * inv_sc);        // x the ones column
      } else {
#pragma unroll 1
        for (int c = hh; c < hh + 1; ++c) {
          tmem_ld16(tmem + cW + lane_base + 96 + 16 * c, v);
          tmem_ld16(tmem + cW + lane_base + 32 + 16 * c, u);
          tmem_wait_ld();
#pragma unroll
          for (int k = 0; k < 16; ++k)
            put(kW2tOff + j * kOutPad + 1 + 16 * c + k, (__uint_as_float(v[k]) + __uint_as_float(u[k])) * inv_sc);
        }
        tmem_ld16(tmem + cW + lane_base + 128, v);
        tmem_wait_ld();
        if (hh == 0) put(kW2tOff + j * kOutPad, (__uint_as_float(v[0]) + __uint_as_float(v[1])) * inv_sc);   // x gsig hi + lo
      }
      } else {
      const int j = row & 63;
      uint32_t v[16], u[16];
      if (row < 64) {
#pragma unroll 1
        for (int c = hh; c < hh + 1; ++c) {     // x F hi + x F lo: channels k = 16 c ..
          tmem_ld16(tmem + cW + lane_base + 64 + 16 * c, v);
          tmem_ld16(tmem + cW + lane_base + 16 * c, u);
          tmem_wait_ld();
#pragma unroll
          for (int k = 0; k < 16; ++k)
            atomicAdd(a.g_dec + kW1tOff + (16 * c + k) * kHid + j, (__uint_as_float(v[k]) + __uint_as_float(u[k])) * inv_sc);
        }
        tmem_ld16(tmem + cW + lane_base + 128, v);
        tmem_wait_ld();
        if (hh == 0) atomicAdd(a.g_dec + kB1Off + j, __uint_as_float(v[2]) * inv_sc);        // x the ones column
      } else {
#pragma unroll 1
        for (int c = hh; c < hh + 1; ++c) {
          tmem_ld16(tmem + cW + lane_base + 96 + 16 * c, v);
          tmem_ld16(tmem + cW + lane_base + 32 + 16 * c, u);
          tmem_wait_ld();
#pragma unroll
          for (int k = 0; k < 16; ++k)
            atomicAdd(a.g_dec + kW2tOff + j * kOutPad + 1 + 16 * c + k, (__uint_as_float(v[k]) + __uint_as_float(u[k])) * inv_sc);
        }
        tmem_ld16(tmem + cW + lane_base + 128, v);
        tmem_wait_ld();
        if (hh == 0) atomicAdd(a.g_dec + kW2tOff + j * kOutPad, (__uint_as_float(v[0]) + __uint_as_float(v[1])) * inv_sc);   // x gsig hi + lo
      }
      }
      tcgen05_fence_before();
    }
  } else {
    // ================================================ MMA issuer ================================================
    const uint32_t base16 = (smem_u32(&s) >> 4);
#define OFF16(member) (base16 + (uint32_t)(offsetof(Smem, member) >> 4))
    const uint32_t iF16_64 = instr_desc(kFmtF16, 128, 64), iF16_32 = instr_desc(kFmtF16, 128, 32);
    // G1 + G2 of tile i (both only need the tile's inputs; D1 / GH are free: the epilogue of tile i - 1 has read them before it
    // published H / GA)
    auto issue_g12 = [&](int i, bool block) -> bool {
      const int b = i & 1;
      if (block) mbar_wait_parked(&s.in_full[b], (uint32_t)(i >> 1) & 1u);
      else if (!__shfl_sync(0xffffffffu, (int)mbar_try_wait(&s.in_full[b], (uint32_t)(i >> 1) & 1u), 0)) return false;
      tcgen05_fence_after();
      if (elect_one_sync()) {
        // K-major operands, k-step = 32 bytes = 2 units; features in chunks 0-3 of a row, colour-logit gradients in chunks 4-7; W1 / W2
        // rows are [hi | lo]: the lo halves start 4 units into the row
        const uint32_t lo = OFF16(in) + (uint32_t)b * (uint32_t)(sizeof(Smem::In) >> 4), hi = lo + (kTile >> 4);
        const uint32_t w1 = OFF16(w1k), w2 = OFF16(w2c);
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {       // G1: D1 = [F hi | F lo] . [W1 hi | W1 lo]
          mma_f16_ss(tmem + cD1, make_desc(hi + 2 * ks, 1, 64, 2), make_desc(w1 + 2 * ks, 1, 64, 2), iF16_64, ks > 0);
          mma_f16_ss(tmem + cD1, make_desc(lo + 2 * ks, 1, 64, 2), make_desc(w1 + 2 * ks, 1, 64, 2), iF16_64, true);
          mma_f16_ss(tmem + cD1, make_desc(hi + 2 * ks, 1, 64, 2), make_desc(w1 + 4 + 2 * ks, 1, 64, 2), iF16_64, true);
        }
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {       // G2: GH = [GYc hi | lo] . [W2c hi | lo]
          mma_f16_ss(tmem + cGH, make_desc(hi + 4 + 2 * ks, 1, 64, 2), make_desc(w2 + 2 * ks, 1, 64, 2), iF16_64, ks > 0);
          mma_f16_ss(tmem + cGH, make_desc(lo + 4 + 2 * ks, 1, 64, 2), make_desc(w2 + 2 * ks, 1, 64, 2), iF16_64, true);
          mma_f16_ss(tmem + cGH, make_desc(hi + 4 + 2 * ks, 1, 64, 2), make_desc(w2 + 4 + 2 * ks, 1, 64, 2), iF16_64, true);
        }
        mma_commit(&s.g12_done);
      }
      __syncwarp();
      return true;
    };
    PROF_DECL();
    if (G > 0) issue_g12(0, true);
    for (int i = 0; i < G; ++i) {
      const int b = i & 1;
      PROF_T0();
      mbar_wait_parked(&s.hga_ready, (uint32_t)i & 1u);                      // H and GA tiles are in shared memory
      PROF(13);
      if (i > 0) mbar_wait_parked(&s.gf_ready[b ^ 1], (uint32_t)((i - 1) >> 1) & 1u);      // the previous GF has left TMEM
      PROF(14);
      tcgen05_fence_after();
      const uint32_t gah = OFF16(ga_hi), gal = OFF16(ga_lo);
      if (elect_one_sync()) {
        // G3: GF = GA . W1g^T, K = 64 hidden = 4 k-steps; GA hi / lo tiles (K-major), W1g hi / lo tiles
        const uint32_t wh = OFF16(w1g), wl = OFF16(w1g) + ((32 * 128) >> 4);
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          mma_f16_ss(tmem + cGF, make_desc(gah + 2 * ks, 1, 64, 2), make_desc(wh + 2 * ks, 1, 64, 2), iF16_32, ks > 0);
          mma_f16_ss(tmem + cGF, make_desc(gal + 2 * ks, 1, 64, 2), make_desc(wh + 2 * ks, 1, 64, 2), iF16_32, true);
          mma_f16_ss(tmem + cGF, make_desc(gah + 2 * ks, 1, 64, 2), make_desc(wl + 2 * ks, 1, 64, 2), iF16_32, true);
        }
        mma_commit(&s.g3_done);
      }
      __syncwarp();
      // G1 + G2 of the NEXT tile go ahead of this tile's weight-gradient MMAs when its inputs are already there (not waited for:
      // the weight-gradient commit is what frees the loaders' other buffer): the next epilogue's TMEM loads and arithmetic then
      // overlap WG instead of waiting behind it.  (TPR_BWD_DEBUG bit 3 = always after WG, for A/B.)
      const bool early = a.lookahead && i + 1 < G && issue_g12(i + 1, false);
      if (elect_one_sync()) {
        // WG: the weight gradients, accumulated over every tile of this CTA.  A = [GA ; H] (M = 128: two 64-element atoms along
        // MN, 16 KB apart = LBO 1024 units), MN-major: K = samples = rows, 16 rows = 2048 bytes = 128 units per k-step, 8-row
        // groups 1024 bytes apart (SBO 64).  B = the tile's three input atoms, MN-major likewise: [lo | hi | sig] x A hi (N = 144)
        // and [hi | sig] x A lo (N = 80, onto columns 64..143) -- two MMAs per k-step; every MMA re-reads its 4 KB A slice from
        // shared memory (32 cycles), which is what the six narrower MMAs per k-step of the first version were bound by
        if (want_dec) {
          const uint32_t lo = OFF16(in) + (uint32_t)b * (uint32_t)(sizeof(Smem::In) >> 4), hi = lo + (kTile >> 4);
          const uint32_t mn144 = instr_desc(kFmtF16, 128, 144) | kMajorMN, mn80 = instr_desc(kFmtF16, 128, 80) | kMajorMN;
#pragma unroll
          for (int ks = 0; ks < 8; ++ks) {
            mma_f16_ss(tmem + cW, make_desc(gah + 128 * ks, 1024, 64, 2), make_desc(lo + 128 * ks, 1024, 64, 2), mn144, i > 0 || ks > 0);
            mma_f16_ss(tmem + cW + 64, make_desc(gal + 128 * ks, 1024, 64, 2), make_desc(hi + 128 * ks, 1024, 64, 2), mn80, true);
          }
        }
        mma_commit(&s.wg_done);
        mma_commit(&s.in_free[b]);
        if (i == G - 1) mma_commit(&s.all_done);
      }
      __syncwarp();
      PROF(15);
      if (i + 1 < G && !early) issue_g12(i + 1, true);
      PROF(16);
    }
    PROF_FLUSH(13, 16, true);
#undef OFF16
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 0) { tcgen05_fence_after(); tmem_dealloc(tmem, 512); }
}

}  // namespace bwdtc

// Launch; returns cudaError_t (0 = ok) or -1 when the device cannot run it (the caller keeps the mma.sync kernel).
// scale_buf: 4 floats of device scratch ([0..1] the power-of-two scale and its inverse, [2..3] the range accumulators).
// point != 0: point queries (rows of colours / g_rgb per point, no omega, S unused; g_rgb may be NULL).
// n_sets: planes / g_planes hold n_sets plane sets; image n (of total / pts_per_img) reads and scatters to set n % n_sets.
// det != NULL: the deterministic mode (tpr_device.cuh: DetScratch); the launch sets det->n_rows and zeroes those rows, the
// caller zeroes det->acc and converts both afterwards (launch_det_finish).
int launch_bwd_decode_tc(const float* planes, int H, int W, const float* dec, const float* pts, const float* colours, int col_chunked,
                         const float* features, const float* gsig, const float* omega, const float* g_rgb, long long total,
                         long long pts_per_img, int n_sets, int S, int point, float box_scale, float* g_planes, float* g_dec,
                         float* scale_buf, DetScratch* det, int sms, int smem_optin, cudaStream_t st) {
  using namespace bwdtc;
  const size_t smem = sizeof(Smem) + 1024 + (det ? kLoadWarps * 33 * sizeof(float) : 0);
  if ((int)smem > smem_optin) return -1;
  cudaError_t e = cudaMemsetAsync(scale_buf + 2, 0, 2 * sizeof(float), st);
  if (e != cudaSuccess) return (int)e;
  const long long n_rgb = point ? (g_rgb ? total * 32 : 0) : (total / S) * 32;
  scale_kernel<<<sms * 4, 256, 0, st>>>(g_rgb, n_rgb, gsig, total, dec, reinterpret_cast<unsigned*>(scale_buf + 2));
  scale_finish_kernel<<<1, 64, 0, st>>>(reinterpret_cast<const unsigned*>(scale_buf + 2), dec, scale_buf);
  if (det) det_bound_kernel<<<1, 64, 0, st>>>(reinterpret_cast<const unsigned*>(scale_buf + 2), dec, total / n_sets, det->hdr);
  Args a;
  a.planes = planes; a.H = H; a.W = W; a.n_sets = n_sets; a.dec = dec; a.pts = pts; a.colours = colours; a.col_chunked = col_chunked; a.features = features; a.gsig = gsig;
  a.omega = omega; a.g_rgb = g_rgb; a.total = total; a.pts_per_img = pts_per_img; a.S = S; a.box_scale = box_scale;
  a.g_planes = g_planes; a.g_dec = g_dec; a.scale = scale_buf; a.prof = nullptr;
  a.g_acc = det ? det->acc : nullptr; a.dec_rows = det ? det->rows : nullptr; a.det_hdr = det ? det->hdr : nullptr;
  { const char* dbg = getenv("TPR_BWD_DEBUG"); const int d = dbg ? atoi(dbg) : 0;      // profiling A/B: 1 = no scatter, 2 = no weight gradients
    if (d & 1) a.g_planes = nullptr;
    if (d & 2) a.g_dec = nullptr;
    a.lookahead = (d & 8) ? 0 : 1; }
  static const bool profile = getenv("TPR_BWD_PROFILE") != nullptr;
  void (*kern)(const Args) = det ? (point ? decode_backward_tc_kernel<false, true, true> : decode_backward_tc_kernel<false, false, true>)
                           : profile ? (point ? decode_backward_tc_kernel<true, true> : decode_backward_tc_kernel<true, false>)
                                     : (point ? decode_backward_tc_kernel<false, true> : decode_backward_tc_kernel<false, false>);
  e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  if (pts_per_img < kM) return -1;                 // (a tile may straddle at most two images)
  const long long n_tiles = (total + kM - 1) / kM;
  long long grid = n_tiles < sms ? n_tiles : sms;
  if (det) {
    if (grid > kDetMaxRows) grid = kDetMaxRows;
    det->n_rows = (int)grid;
    if (g_dec && (e = cudaMemsetAsync(det->rows, 0, (size_t)grid * kDecFloats * sizeof(float), st)) != cudaSuccess) return (int)e;
    kern<<<(unsigned)grid, kThreads, smem, st>>>(a);
    return (int)cudaGetLastError();
  }
  if (profile) {                                    // debugging aid: synchronous, prints CTA 0's cycles per role and phase
    static const char* names[17] = {"load: issue loads", "-", "load: wait in_free", "load: operands", "scatter: load points",
                                    "scatter: wait gf_ready", "scatter: red", "epi: wait g12_done", "epi: wait wg_done", "epi: H/GA",
                                    "epi: wait g3_done", "epi: wait gf_free", "epi: GF", "mma: wait hga_ready", "mma: wait gf_ready",
                                    "mma: issue G3+WG", "mma: wait in_full + issue G12"};
    long long* prof = nullptr; long long host[17];
    cudaMalloc(&prof, sizeof(host)); cudaMemsetAsync(prof, 0, sizeof(host), st);
    a.prof = prof;
    kern<<<(unsigned)grid, kThreads, smem, st>>>(a);
    cudaStreamSynchronize(st);
    cudaMemcpy(host, prof, sizeof(host), cudaMemcpyDeviceToHost); cudaFree(prof);
    const long long tiles0 = (n_tiles + grid - 1) / grid;
    for (int k = 0; k < 17; ++k) fprintf(stderr, "[bwd profile] %-32s %8.0f cycles / tile\n", names[k], (double)host[k] / (double)tiles0);
    return (int)cudaGetLastError();
  }
  kern<<<(unsigned)grid, kThreads, smem, st>>>(a);
  return (int)cudaGetLastError();
}

// Deterministic mode ahead of the mma.sync kernel: the upstream gradient's range and the fixed-point exponent into det->hdr
// (what launch_bwd_decode_tc computes on its way).  Arguments as there.
int launch_det_bound(const float* dec, const float* gsig, const float* g_rgb, long long total, int n_sets, int S, int point,
                     float* scale_buf, DetScratch* det, int sms, cudaStream_t st) {
  using namespace bwdtc;
  cudaError_t e = cudaMemsetAsync(scale_buf + 2, 0, 2 * sizeof(float), st);
  if (e != cudaSuccess) return (int)e;
  const long long n_rgb = point ? (g_rgb ? total * 32 : 0) : (total / S) * 32;
  scale_kernel<<<sms * 4, 256, 0, st>>>(g_rgb, n_rgb, gsig, total, dec, reinterpret_cast<unsigned*>(scale_buf + 2));
  det_bound_kernel<<<1, 64, 0, st>>>(reinterpret_cast<const unsigned*>(scale_buf + 2), dec, total / n_sets, det->hdr);
  return (int)cudaGetLastError();
}

}  // namespace tpr
