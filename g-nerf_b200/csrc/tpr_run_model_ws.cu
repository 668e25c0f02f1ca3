// Warp-specialised ImportanceRenderer.run_model (VR/renderer.py:142-148) for arbitrary points on sm_100a:
// plane gather (VR/renderer.py:55-65) + OSGDecoder (training/triplane.py:124-136) with the decoder on tcgen05,
// for the density-grid extraction of gen_videos.py:33-55,198-209 (256^3 points, sigma only) and
// TriPlaneGenerator.sample / sample_mixed (training/triplane.py:92-104).
//
// Same building blocks as the fused forward (tpr_ws.cuh), different pipeline: there are no rays, so a tile is simply
// 128 consecutive points of one image and the three roles are
//   warps  0-15  GATHER   xyz -> bilinear taps -> 12 x 128-byte texel reads per point -> A1 operand tile (3 deep)
//   warps 16-23  DECODE   warp 16 issues the tcgen05.mma; all eight run the softplus epilogue out of TMEM, add up
//                         sigma (the single sigma row of layer 2 is an fp32 dot product) and store it, coalesced
//   warps 24-31  COLOUR   (only when rgb is wanted) read the 32 colour logits of a tile out of its TMEM slot,
//                         sigmoid, store rgb [P,32]
// Layer 1 is double buffered in TMEM (two 128-column stages: D1 / activations), so the tensor core works on tile
// t+1 while the epilogue of tile t runs; layer 2 (colour rows only) writes into a ring of eight 32-column slots.
// Every CTA walks a CONTIGUOUS range of tiles: on a regular grid consecutive tiles (neighbouring y rows) hit the
// same texels of two of the three planes, so the L1 keeps them.
//
// Citations relative to /root/reference/g_nerf/ (VR/ = training/volumetric_rendering/).
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include "triplane_b200.h"
#include "tpr_ws.cuh"

namespace tpr {
namespace wsrm {
using namespace tc;
using namespace ws;

constexpr int kColourWarps = 8;
// Gather warps: 16 when a COLOUR role shares the SM (sigma + rgb); 24 for sigma-only queries, where the eight warps the COLOUR
// role does not need gather as well.  With 24 they work as three teams of eight warps, team k gathering the tiles i = k (mod 3)
// into A1 buffer k, sixteen rows per warp: three tiles are in flight instead of one, and the random-line gather -- latency
// bound, more lines in flight = more bandwidth (profiles/r02_gather_shapes.json: 24 warps x 4 lines 17.2 TB/s, 16 x 4 14.6) --
// is what this kernel waits for.
template <bool RGB> struct Roles {
  static constexpr int gather = RGB ? ws::kGatherWarps : 24;
  static constexpr int teams = RGB ? 1 : 3;
  static constexpr int team_warps = gather / teams;                 // 16 or 8
  static constexpr int passes = ws::kRows / (8 * team_warps);       // 8-row passes per warp and tile: 1 or 2
  static constexpr int threads = 32 * (gather + ws::kDecodeWarps + (RGB ? kColourWarps : 0));
};
static_assert(Roles<false>::teams == ws::kBufs, "team k owns A1 buffer k");
constexpr int kStages = 2;                         // TMEM: stage s = columns [128 s, 128 s + 128) (D1, and bf16's activations behind it)
constexpr uint32_t kRmStageCols = 128;
constexpr int kSlots = 8;                          // colour slots: columns [256 + 32 k, 256 + 32 k + 32)
constexpr uint32_t kRmSlotBase = kStages * kRmStageCols;

struct RmArgs {
  const float* planes; int H, W;
  long long plane_sets;            // image n reads plane set n % plane_sets
  const float* dec; const float* xyz;
  long long n_pts, tiles_per_img, n_tiles;
  float box_scale;
  float* rgb; float* sigma;
};

struct RmBarriers {
  uint64_t a1_full[kBufs];       // 16 gather-warp arrivals
  uint64_t a1_free[kBufs];       // tcgen05.commit: layer 1 has consumed the tile
  uint64_t d1_full[kStages];     // tcgen05.commit: layer 1 of a tile is in its stage
  uint64_t a2_full[kStages];     // 8 decode-warp arrivals: D1 has been read (and the activations written back)
  uint64_t slot_full[kSlots];    // tcgen05.commit: layer 2 of a tile is in its slot
  uint64_t slot_free[kSlots];    // 8 colour-warp arrivals: the slot has been read
};

// one tile of 128 points -> A1 buffer.  Warp w owns rows [8w, 8w+8); same two steps as the forward's gather_tile.
template <int MODE>
__device__ __forceinline__ void gather_tile_points(const RmArgs& a, float* a1_hi, const float* __restrict__ img,
                                                   const float* __restrict__ pts, int nvalid, Tap2* tw, int row0, int lane) {
  // row0: the first of this warp's eight rows
  const int grp = lane >> 3, sub = lane & 7;
  {
    const int s = lane / 3, p = lane - s * 3;
    const int row = row0 + s;
    if (lane < 24 && row < nvalid) {
      const float* c = pts + (size_t)row * 3;
      // (2/box_warp) * coordinates (VR/renderer.py:61)
      const float px = __fmul_rn(__ldg(c + 0), a.box_scale), py = __fmul_rn(__ldg(c + 1), a.box_scale),
                  pz = __fmul_rn(__ldg(c + 2), a.box_scale);
      Taps tp;
      plane_taps(p == 2 ? pz : px, p == 0 ? py : (p == 1 ? pz : px), a.H, a.W, tp);   // (x,y) (x,z) (z,x)
      const int po = p * a.H * a.W * kC;
      *reinterpret_cast<uint4*>(tw[lane].off) = make_uint4((unsigned)(tp.off[0] + po) >> 2, (unsigned)(tp.off[1] + po) >> 2,
                                                           (unsigned)(tp.off[2] + po) >> 2, (unsigned)(tp.off[3] + po) >> 2);
      *reinterpret_cast<float4*>(tw[lane].w2) = make_float4(tp.w[0], tp.w[0], tp.w[1], tp.w[1]);
      *reinterpret_cast<float4*>(tw[lane].w2 + 4) = make_float4(tp.w[2], tp.w[2], tp.w[3], tp.w[3]);
    }
  }
  __syncwarp();
  const ulonglong2* base = reinterpret_cast<const ulonglong2*>(img) + sub;
  asm volatile("" : "+l"(base));
#pragma unroll 1
  for (int rd = 0; rd < 2; ++rd) {
    const int s = rd * 4 + grp;
    const int row = row0 + s;
    if (row < nvalid) blend_sample<MODE>(a1_hi, base, tw + s * 3, row, sub);
  }
  __syncwarp();           // the tap table is rewritten by the next tile
}

template <int MODE, bool RGB>
__global__ void __launch_bounds__(Roles<RGB>::threads, 1)
run_model_ws_kernel(const RmArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  Tiles<MODE>& tl = *reinterpret_cast<Tiles<MODE>*>(base);
  Tap2* taps = reinterpret_cast<Tap2*>(base + sizeof(Tiles<MODE>));
  __shared__ RmBarriers bars;
  __shared__ uint32_t tmem_base_sm;
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  constexpr int kGW = Roles<RGB>::gather;

  if (tid == 0) {
    for (int b = 0; b < kBufs; ++b) { mbar_init(&bars.a1_full[b], Roles<RGB>::team_warps); mbar_init(&bars.a1_free[b], 1); }
    for (int s = 0; s < kStages; ++s) { mbar_init(&bars.d1_full[s], 1); mbar_init(&bars.a2_full[s], kDecodeWarps); }
    for (int k = 0; k < kSlots; ++k) { mbar_init(&bars.slot_full[k], 1); mbar_init(&bars.slot_free[k], kColourWarps); }
    fence_mbar_init();
  }
  if (warp == 0) { tmem_alloc(&tmem_base_sm, 512); tmem_relinquish(); }
  // rows of a partial last tile are never written: start from finite operands
  for (int i = tid; i < (int)(sizeof(tl.a1) / 16); i += blockDim.x) reinterpret_cast<float4*>(tl.a1)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  stage_weights<MODE>(a.dec, tl);
  fence_proxy_async_smem();
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = __shfl_sync(0xffffffffu, tmem_base_sm, 0);
  const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;

  // this CTA's contiguous tile range
  const long long per = (a.n_tiles + gridDim.x - 1) / gridDim.x;
  const long long t0 = blockIdx.x * per;
  const int G = (int)max(0ll, min(a.n_tiles, t0 + per) - t0);
  const size_t img_stride = (size_t)3 * a.H * a.W * kC;
  auto tile_of = [&](int i, long long& n, long long& p0, int& nvalid) {
    const long long T = t0 + i;
    n = T / a.tiles_per_img;
    p0 = (T - n * a.tiles_per_img) * kRows;
    nvalid = (int)min((long long)kRows, a.n_pts - p0);
  };

  if (warp < kGW) {
    // ====================================== GATHER ======================================
    Tap2* tw = taps + warp * 24;
    const int team = warp / Roles<RGB>::team_warps, wt = warp - team * Roles<RGB>::team_warps;
#pragma unroll 1
    for (int i = team; i < G; i += Roles<RGB>::teams) {
      const int b = i % kBufs;
      const uint32_t ph = (uint32_t)(i / kBufs) & 1u;         // the tile's turn of the ring
      long long n, p0; int nvalid;
      tile_of(i, n, p0, nvalid);
      mbar_wait_parked(&bars.a1_free[b], ph ^ 1u);          // passes immediately the first time round
#pragma unroll 1
      for (int ps = 0; ps < Roles<RGB>::passes; ++ps)
        gather_tile_points<MODE>(a, tl.a1[b][0], a.planes + (size_t)(n % a.plane_sets) * img_stride,
                                 a.xyz + (size_t)(n * a.n_pts + p0) * 3, nvalid, tw, (wt * Roles<RGB>::passes + ps) * 8, lane);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars.a1_full[b]);
    }
  } else if (warp < kGW + kDecodeWarps) {
    // ====================================== DECODE ======================================
    const int dw = warp - kGW, q = dw & 3, h = dw >> 2;
    const bool issuer = dw == 0;
    const uint32_t dbase = smem_desc_lo(smem_u32(&tl));
    int b = 0; uint32_t ph = 0;                         // A1 ring position of the NEXT layer-1 issue
    // layer 1 of tile j into stage j & 1: its A1 tile must be gathered, and tile j-2 must have left the stage (its
    // epilogue has read D1; its layer 2, issued earlier, reads the activations before this MMA overwrites them
    // because the tensor pipe executes in issue order)
    auto issue_l1 = [&](int j) {
      mbar_wait_parked(&bars.a1_full[b], ph);
      if (j >= 2) mbar_wait_parked(&bars.a2_full[j & 1], (uint32_t)((j - 2) >> 1) & 1u);
      tcgen05_fence_after();
      const int bu = __shfl_sync(0xffffffffu, b, 0);
      const uint32_t st = tmem + (uint32_t)(j & 1) * kRmStageCols;
      if (elect_one_sync()) {
        issue_layer1<MODE>(dbase, bu, st);
        mma_commit(&bars.a1_free[b]);
        mma_commit(&bars.d1_full[j & 1]);
      }
      __syncwarp();
      if (++b == kBufs) { b = 0; ph ^= 1u; }
    };
    if (issuer && G > 0) issue_l1(0);
#pragma unroll 1
    for (int i = 0; i < G; ++i) {
      long long n, p0; int nvalid;
      tile_of(i, n, p0, nvalid);
      const int s = i & 1;
      const uint32_t sph = (uint32_t)(i >> 1) & 1u;
      if (issuer && i + 1 < G) issue_l1(i + 1);         // the tensor core works on tile i+1 during this epilogue
      mbar_wait_parked(&bars.d1_full[s], sph);
      tcgen05_fence_after();
      const float sgp = epilogue1<MODE, RGB>(tl, tmem + (uint32_t)s * kRmStageCols, lane_base, h);
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars.a2_full[s]);
      if (RGB && issuer) {
        const int k = i & (kSlots - 1);
        mbar_wait_parked(&bars.a2_full[s], sph);
        mbar_wait_parked(&bars.slot_free[k], ((uint32_t)(i / kSlots) & 1u) ^ 1u);     // passes the first time round
        tcgen05_fence_after();
        if (elect_one_sync()) {
          issue_layer2<MODE>(dbase, tmem + (uint32_t)s * kRmStageCols, tmem + kRmSlotBase + (uint32_t)k * kSlotCols);
          mma_commit(&bars.slot_full[k]);
        }
        __syncwarp();
      }
      // sigma of this tile: the two warps of a lane quarter add their halves (training/triplane.py:135)
      if (h == 1) tl.psig[q * 32 + lane] = sgp;
      named_bar_sync(3 + q, 64);
      if (h == 0) {
        const int row = q * 32 + lane;
        if (row < nvalid) a.sigma[n * a.n_pts + p0 + row] = sgp + tl.psig[row] + tl.bias2[kNc];
      }
      named_bar_sync(3 + q, 64);                        // psig is rewritten by the next tile
    }
  } else if (RGB) {
    // ====================================== COLOUR ======================================
    const int cw = warp - kGW - kDecodeWarps, q = cw & 3, hc = cw >> 2;
#pragma unroll 1
    for (int i = 0; i < G; ++i) {
      long long n, p0; int nvalid;
      tile_of(i, n, p0, nvalid);
      const int k = i & (kSlots - 1);
      mbar_wait_parked(&bars.slot_full[k], (uint32_t)(i / kSlots) & 1u);
      tcgen05_fence_after();
      uint32_t v[16];
      tmem_ld16(tmem + kRmSlotBase + (uint32_t)k * kSlotCols + lane_base + 16 * hc, v);
      tmem_wait_ld();
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars.slot_free[k]);
      const int row = q * 32 + lane;
      if (row < nvalid) {
        float4* dst = reinterpret_cast<float4*>(a.rgb + (size_t)(n * a.n_pts + p0 + row) * kC + 16 * hc);
#pragma unroll
        for (int c4 = 0; c4 < 4; ++c4) {
          float o[4];
#pragma unroll
          for (int c = 0; c < 4; ++c)      // sigmoid(x) * 1.002 - 0.001 (training/triplane.py:134); the slot holds -x log2e
            o[c] = colour_act_neglog2(__uint_as_float(v[4 * c4 + c]) + tl.bias2[16 * hc + 4 * c4 + c]);
          dst[c4] = make_float4(o[0], o[1], o[2], o[3]);
        }
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 0) { tcgen05_fence_after(); tmem_dealloc(tmem, 512); }
}

template <int MODE>
static size_t smem_bytes() { return 1024 + sizeof(Tiles<MODE>) + sizeof(Tap2) * Roles<false>::gather * 24; }

}  // namespace wsrm

// Launch; returns cudaError_t (0 = ok) or -1 if the shape does not fit (the caller uses the FFMA kernel).
int launch_run_model_ws(const float* planes, long long n_img, long long plane_sets, int H, int W, const float* dec, const float* xyz,
                        long long n_pts, float box_scale, float* rgb, float* sigma, int mode, int sms, int smem_optin, cudaStream_t st) {
  using namespace wsrm;
  RmArgs a;
  a.planes = planes; a.H = H; a.W = W; a.plane_sets = plane_sets; a.dec = dec; a.xyz = xyz; a.n_pts = n_pts;
  a.tiles_per_img = (n_pts + ws::kRows - 1) / ws::kRows;
  a.n_tiles = a.tiles_per_img * n_img;
  a.box_scale = box_scale; a.rgb = rgb; a.sigma = sigma;
  if (a.n_tiles >= (1ll << 31) * (long long)sms) return -1;          // the per-CTA tile count is an int
  typedef void (*Kernel)(const RmArgs);
  const bool want_rgb = rgb != nullptr;
  Kernel k = mode == 1 ? (want_rgb ? run_model_ws_kernel<1, true> : run_model_ws_kernel<1, false>)
                       : (want_rgb ? run_model_ws_kernel<2, true> : run_model_ws_kernel<2, false>);
  const size_t smem = mode == 1 ? smem_bytes<1>() : smem_bytes<2>();
  cudaFuncAttributes fa;
  cudaError_t e = cudaFuncGetAttributes(&fa, k);
  if (e != cudaSuccess) return (int)e;
  if ((int)smem > smem_optin - (int)fa.sharedSizeBytes) return -1;
  e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  const long long grid = a.n_tiles < sms ? a.n_tiles : sms;            // one CTA per SM: each owns all 512 TMEM columns
  const int threads = want_rgb ? Roles<true>::threads : Roles<false>::threads;
  k<<<(unsigned)grid, threads, smem, st>>>(a);
  return (int)cudaGetLastError();
}

}  // namespace tpr
