/*
 * triplane_b200.h -- C ABI of libtriplane_b200.so, the sm_100a tri-plane volume renderer.
 *
 * This is the drop-in boundary for ONE hot path of llrtt/G-NeRF: everything
 * ImportanceRenderer.forward does between receiving (planes, decoder, rays, options)
 * and returning (rgb, depth, weight_sum).  Citations are relative to
 * /root/reference/g_nerf/ ; VR/ = training/volumetric_rendering/.
 *
 * Conventions (mirroring the reference's plugin convention, torch_utils/ops/bias_act.cpp:39-92,
 * behind a C ABI instead of torch::Tensor):
 *   - every pointer is a DEVICE pointer on the current CUDA device unless the name ends in _host;
 *     all tensors are dense, contiguous, float32 (int32/int64 where stated);
 *   - the caller owns all memory (inputs, outputs, scratch); the library never allocates, frees
 *     or keeps a device pointer after the call returns (one exception with explicit create /
 *     destroy calls: the peer-mapped gather buffers of the multi-GPU section, tpr_peer_*);
 *   - every entry point is asynchronous on `stream` (a cudaStream_t passed as void*), never
 *     synchronises the device, and is re-entrant across host threads and streams;
 *   - return value: 0 = success, < 0 = argument error (TPR_E_*), > 0 = a cudaError_t from the
 *     launch; tpr_last_error() returns a thread-local message for the last non-zero return.
 *   - forward AND backward: tpr_render / tpr_render_train are the forward, tpr_render_backward the gradient with respect
 *     to the planes and the decoder (SURVEY.md section 8(f), row 3; the reference gets it from autograd).
 */
#ifndef TRIPLANE_B200_H_
#define TRIPLANE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TPR_ABI_VERSION 8

/* fixed by the reference model: OSGDecoder(32 -> 64 -> 1+32), three planes
 * (training/triplane.py:42,113-122; VR/renderer.py:29-37) */
#define TPR_CHANNELS 32
#define TPR_HIDDEN 64
#define TPR_OUT 33
#define TPR_PLANES 3
#define TPR_MAX_SAMPLES 256 /* depth_resolution + depth_resolution_importance */

enum {
  TPR_E_NULL = -1,      /* a required pointer is NULL */
  TPR_E_SHAPE = -2,     /* a size is out of the supported range */
  TPR_E_OPTION = -3,    /* an option value the reference would also reject (e.g. clamp_mode) */
  TPR_E_SCRATCH = -4,   /* scratch buffer too small */
  TPR_E_DEVICE = -5     /* not an sm_100 device / kernel image missing */
};

/* flags */
enum {
  TPR_MLP_FP32 = 0,     /* fp32-grade decoder, the 1e-4 max-abs parity mode: tcgen05 with fp16 hi + lo operand pairs
                           (three products per contraction, fp32 accumulation) when the sample counts fit the TMEM
                           slots, the FFMA kernel otherwise */
  TPR_MLP_BF16 = 1,     /* decoder on tensor cores with bf16 operands: the >= 50 dB PSNR mode */
  TPR_MLP_FFMA = 2      /* force the fp32 FFMA kernel (A/B comparisons) */
};
/* A bit OR-ed into the flags of tpr_render_backward (opt->flags) and tpr_run_model_backward (flags): the deterministic
 * backward.  Two calls with equal inputs on the same device give bit-identical gradients, and the plane gradient does not
 * depend on the order of the samples: it is accumulated in 64-bit fixed point (every contribution scaled by a power of two
 * chosen from a bound on any texel's sum, so nothing overflows).  The decoder gradient is summed per CTA and the partial
 * rows are added in a fixed order in fp64: bit-identical for the same GPU model and shape, not across GPUs with different
 * SM counts.  Needs tpr_backward_deterministic_scratch_bytes more scratch.  The forward is deterministic without it. */
#define TPR_BWD_DETERMINISTIC 0x100

/* The subset of `rendering_options` the hot path reads (SURVEY.md section 5, option table;
 * VR/renderer.py:91-100,116,143-146; VR/ray_marcher.py:32,52). */
typedef struct TprOptions {
  /* Python floats in the reference, so doubles here: the kernels reproduce the exact float32
   * constants torch derives from them ((end-start)/(D-1), 1/start, 2/box_warp ...). */
  double ray_start;              /* scalar limits (VR/renderer.py:100); ignored if per-ray limits given */
  double ray_end;
  double box_warp;               /* VR/renderer.py:61 */
  int32_t depth_resolution;      /* Dc >= 2 */
  int32_t depth_resolution_importance; /* Df >= 0; 0 = coarse pass only (VR/renderer.py:116,136-137) */
  int32_t disparity_space_sampling;    /* VR/renderer.py:174-181 */
  int32_t white_back;            /* VR/ray_marcher.py:52-53 */
  int32_t flags;                 /* TPR_MLP_* */
  int32_t tile_width;            /* perf hint only, never changes results: rays form a square image this many pixels
                                    wide with x fastest (0 = infer from a perfect-square ray count, < 0 = no image) */
  int32_t plane_sets;            /* 0 (= n_img): image n samples plane set n, the reference's one-to-one batch.  P > 0:
                                    planes_packed holds P plane sets and image (camera) n samples set n % P -- several
                                    frames of the gen_videos.py:153-171 orbit, each a batch of P identities, rendered as ONE
                                    call against planes packed once.  n_img must be a multiple of P */
  int32_t output_layout;         /* TPR_LAYOUT_*: how rgb is written */
  int32_t depth_clamp_group;     /* 0: the depth clamp (VR/ray_marcher.py:50) uses the range of ALL sample depths of the call,
                                    like one reference forward.  k > 0: every k consecutive images clamp against their own
                                    range (k = the batch of one reference forward when several forwards are batched) */
  int32_t reserved;
  /* options.get('density_noise', 0) (VR/renderer.py:146): sigma += randn_like(sigma) * density_noise after each of the two
   * point queries.  The draws are the caller's, like jitter and u: density_noise_coarse [N,M*Dc] then density_noise_fine
   * [N,M*Df] (device pointers, standard normal; the host shim draws them with the reference's torch.randn_like calls in the
   * reference's order: jitter, coarse noise, u, fine noise).  Both ignored (may be NULL) when density_noise == 0. */
  double density_noise;
  const float* density_noise_coarse;
  const float* density_noise_fine;
} TprOptions;

/* output_layout */
enum {
  TPR_LAYOUT_CHANNELS_LAST = 0,  /* rgb [N,M,32], what ImportanceRenderer.forward returns (VR/renderer.py:140) */
  TPR_LAYOUT_CHANNELS_FIRST = 1  /* rgb [N,32,M] = the [N,32,H,W] feature image TriPlaneGenerator.synthesis builds from it with
                                    permute + contiguous (training/triplane.py:81): the transpose is folded into the store */
};

int tpr_abi_version(void);
const char* tpr_last_error(void);

/* ---- layout preparation --------------------------------------------------------------- */

/* Planes arrive as [N,3,32,H,W] (training/triplane.py:74).  The renderer wants channels-last
 * [N,3,H,W,32] so that one texel is one 128-byte line.  tpr_pack_planes does that transpose. */
size_t tpr_packed_planes_bytes(int64_t n_img, int32_t height, int32_t width);
int tpr_pack_planes(const float* planes_nchw, int64_t n_img, int32_t height, int32_t width,
                    float* planes_packed, void* stream);
/* The inverse transpose, [N,3,H,W,32] -> [N,3,32,H,W]: the plane gradient of tpr_render_backward in the layout autograd hands to
 * the backbone (the adjoint of the pack above; training/triplane.py:74). */
int tpr_unpack_planes(const float* planes_packed, int64_t n_img, int32_t height, int32_t width, float* planes_nchw,
                      void* stream);

/* Decoder parameters as stored by OSGDecoder.net[0]/net[2] (training/triplane.py:118-122) plus
 * the runtime gains FullyConnectedLayer applies on every call (training/networks_stylegan2.py:
 * 118-119,122-127).  Packs them (gains and the 1/3 plane mean folded in) for the kernels. */
size_t tpr_packed_decoder_bytes(void);
int tpr_pack_decoder(const float* w1 /*[64,32]*/, const float* b1 /*[64]*/,
                     const float* w2 /*[33,64]*/, const float* b2 /*[33]*/,
                     float w1_gain, float b1_gain, float w2_gain, float b2_gain,
                     float* decoder_packed, void* stream);

/* ---- a1: RaySampler.forward (VR/ray_sampler.py:24-63) ---------------------------------- */
int tpr_ray_sample(const float* cam2world /*[N,4,4]*/, const float* intrinsics /*[N,3,3]*/,
                   int64_t n_img, int32_t resolution,
                   float* origins /*[N,res*res,3]*/, float* dirs /*[N,res*res,3]*/, void* stream);

/* ---- a8: ImportanceRenderer.run_model (VR/renderer.py:142-148) ------------------------- */
/* plane gather + decoder for arbitrary points; rgb may be NULL (density grids read sigma only,
 * gen_videos.py:206). */
int tpr_run_model(const float* planes_packed, int64_t n_img, int32_t height, int32_t width,
                  const float* decoder_packed, const float* xyz /*[N,P,3]*/, int64_t n_pts,
                  double box_warp, float* rgb /*[N,P,32] or NULL*/, float* sigma /*[N,P,1]*/,
                  int32_t flags, void* stream);

/* ---- a5: OSGDecoder.forward on already gathered features (training/triplane.py:124-136) - */
int tpr_decode(const float* features /*[N,3,P,32]*/, int64_t n_img, int64_t n_pts,
               const float* decoder_packed, float* rgb /*[N,P,32]*/, float* sigma /*[N,P,1]*/,
               int32_t flags, void* stream);

/* ---- a13: ImportanceRenderer.forward (VR/renderer.py:88-140), fused ---------------------- */
/* jitter [N,M,Dc] stands for torch.rand_like at VR/renderer.py:190, u [N*M,Df] for torch.rand at
 * :237 (the host shim draws both with the same torch calls, so the global RNG stream is consumed
 * exactly as the reference consumes it).  ray_start_per_ray/ray_end_per_ray [N*M] are optional
 * (the 'auto' limits branch, VR/renderer.py:91-97,183-186); pass NULL for scalar limits.
 * Outputs: rgb [N,M,32], depth [N,M,1], weight_sum [N,M,1].  Optional debug outputs (NULL to
 * skip): fine_depths [N*M,Df], fine_inds [N*M,Df] int32 (the searchsorted result, :240).
 * scratch: tpr_render_scratch_bytes() bytes.  depth_range_io [2] (device) receives the global
 * (min,max) of all sample depths that VR/ray_marcher.py:50 clamps against; if
 * clamp_depth != 0 the clamp is applied by a trailing kernel, otherwise the caller applies it
 * (after an all-reduce when rays are sharded over GPUs) with tpr_clamp_depth. */
size_t tpr_render_scratch_bytes(int64_t n_img, int64_t n_rays, const TprOptions* opt);
int tpr_render(const float* planes_packed, int64_t n_img, int32_t height, int32_t width,
               const float* decoder_packed,
               const float* origins /*[N,M,3]*/, const float* dirs /*[N,M,3]*/, int64_t n_rays,
               const float* jitter, const float* u,
               const float* ray_start_per_ray, const float* ray_end_per_ray,
               const TprOptions* opt,
               float* rgb, float* depth, float* weight_sum,
               float* fine_depths, int32_t* fine_inds,
               float* depth_range_io, int32_t clamp_depth,
               void* scratch, size_t scratch_bytes, void* stream);
int tpr_clamp_depth(float* depth, int64_t n, const float* depth_range /*[2] device*/, void* stream);

/* ---- a13 on several GPUs: render + gather in one kernel (SURVEY.md section 8(e)) ------------------------------ */
/* One process per GPU renders its share of the images; every GPU needs all rendered features / depths / weight
 * sums (136 bytes per ray).  Instead of an all-gather AFTER the render, the render kernel's epilogue stores each
 * ray's outputs into this GPU's slice of its own gather buffers AND into the same slice of every peer's gather
 * buffers through peer-mapped NVLink pointers, so the exchange rides along with the render, ray group by ray group.
 * The caller completes the exchange with any cross-GPU barrier that orders "my render kernel finished" before
 * "peers read" -- the all-reduce of the depth range (VR/ray_marcher.py:50 clamps against the range of the WHOLE
 * batch) is that barrier -- and then clamps the gathered depths with tpr_clamp_depth.
 *
 * Peer buffers: tpr_peer_alloc makes a device allocation that other processes on the same node can map
 * (cudaMalloc + cudaIpcGetMemHandle; `handle_out` is the 64-byte cudaIpcMemHandle_t to send to the peers by any
 * means, e.g. torch.distributed.all_gather_object); tpr_peer_open maps a peer's allocation into this process
 * (cudaIpcOpenMemHandle, enabling peer access); tpr_peer_close / tpr_peer_free undo them. */
#define TPR_MAX_PEERS 15
#define TPR_PEER_HANDLE_BYTES 64
typedef struct TprPeerSinks {
  int32_t n_peers;                    /* 0 .. TPR_MAX_PEERS */
  int32_t reserved;
  float* rgb[TPR_MAX_PEERS];          /* peer-mapped pointers shaped and laid out exactly like rgb / depth / weight_sum */
  float* depth[TPR_MAX_PEERS];
  float* weight_sum[TPR_MAX_PEERS];
} TprPeerSinks;
int tpr_peer_alloc(size_t bytes, void** dev_ptr, unsigned char* handle_out /*[64]*/);
int tpr_peer_open(const unsigned char* handle /*[64]*/, void** dev_ptr);
int tpr_peer_close(void* dev_ptr);
int tpr_peer_free(void* dev_ptr);
/* tpr_render with peer sinks.  clamp_depth must be 0 (the clamp needs the all-reduced range). */
int tpr_render_peers(const float* planes_packed, int64_t n_img, int32_t height, int32_t width,
                     const float* decoder_packed,
                     const float* origins, const float* dirs, int64_t n_rays,
                     const float* jitter, const float* u,
                     const float* ray_start_per_ray, const float* ray_end_per_ray,
                     const TprOptions* opt,
                     float* rgb, float* depth, float* weight_sum,
                     float* depth_range_io,
                     void* scratch, size_t scratch_bytes,
                     const TprPeerSinks* peers, void* stream);

/* ---- a13 with HOST buffers: the call a CPU-side caller makes (and the one bench.py times end to end) ---------- */
/* Same result as tpr_render for scalar ray limits, but planes [N,3,32,H,W] (the backbone's layout, NOT repacked),
 * origins and dirs are HOST pointers (pinned memory for the copies to be asynchronous) and rgb / depth /
 * weight_sum are written to HOST memory.  decoder_packed, jitter and u stay DEVICE pointers (the two uniform draws
 * are made on the device, exactly like the reference's torch.rand calls).  One image's planes take longer to cross
 * PCIe than to render, so the library pipelines image by image over two internal copy streams (created once per
 * device, the only state the library keeps) and `stream`: H2D of image i+1, repack + render of image i and D2H of
 * image i-1 overlap.  `workspace` is a DEVICE buffer of tpr_render_host_workspace_bytes() bytes.
 * Asynchronous like every other entry: the outputs are complete when `stream` has drained.
 * depth_range_io: DEVICE [2], receives the global depth range (may be NULL unless depth_host is NULL, see
 * tpr_render_host_depth).  opt->plane_sets must be 0 (or n_img) and opt->depth_clamp_group 0:
 * every image brings its own planes across PCIe and the call clamps against one range, like one reference forward.
 * Calls on one device are serialised inside the library while they ENQUEUE (they share the two copy streams); the enqueued
 * work of different callers' streams still overlaps. */
size_t tpr_render_host_workspace_bytes(int64_t n_img, int32_t height, int32_t width, int64_t n_rays);
int tpr_render_host(const float* planes_host, int64_t n_img, int32_t height, int32_t width,
                    const float* decoder_packed,
                    const float* origins_host /*[N,M,3]*/, const float* dirs_host /*[N,M,3]*/, int64_t n_rays,
                    const float* jitter, const float* u, const TprOptions* opt,
                    float* rgb_host, float* depth_host, float* weight_sum_host, float* depth_range_io,
                    void* workspace, size_t workspace_bytes, void* stream);

/* Rays sharded over several GPUs (SURVEY.md section 8(e)): the clamp of VR/ray_marcher.py:50 needs the range of ALL ranks'
 * depths.  Call tpr_render_host with depth_host = NULL (depth stays, unclamped, in the workspace; depth_range_io receives
 * this GPU's range), all-reduce the two floats (MIN, MAX), then this: clamp with the global range and copy depth
 * [N,M] to the host.  Same workspace and shape as the tpr_render_host call before it. */
int tpr_render_host_depth(void* workspace, size_t workspace_bytes, int64_t n_img, int32_t height, int32_t width,
                          int64_t n_rays, const float* depth_range /*[2] device*/, float* depth_host, void* stream);

/* ---- a9: MipRayMarcher2.forward (VR/ray_marcher.py:25-57), stand-alone ------------------ */
/* colors [R,S,C], densities [R,S], depths [R,S] in the given (not re-sorted) order ->
 * rgb [R,C], depth [R], weights [R,S-1].  depth_range is FOUR floats: [0..1] receive
 * min/max(depths), [2..3] are scratch; the clamp is applied when clamp_depth != 0. */
int tpr_ray_march(const float* colors, const float* densities, const float* depths,
                  int64_t n_rays, int32_t n_samples, int32_t n_channels, int32_t white_back,
                  float* rgb, float* depth, float* weights, float* depth_range, int32_t clamp_depth,
                  void* stream);

/* ---- a10/a11: sample_importance / sample_pdf (VR/renderer.py:194-253), stand-alone ------- */
/* z_vals [R,S], weights [R,S-1] (coarse march weights), u [R,K] -> samples [R,K], inds [R,K]. */
int tpr_sample_importance(const float* z_vals, const float* weights, const float* u,
                          int64_t n_rays, int32_t n_samples, int32_t n_importance,
                          float* samples, int32_t* inds, void* stream);
/* bins [R,B+2] (only the first B+1 entries of each row are read, like the reference's call at
 * :209-210), weights [R,B], u [R,K] -> samples [R,K], inds [R,K]. */
int tpr_sample_pdf(const float* bins, int32_t bins_stride, const float* weights, const float* u,
                   int64_t n_rays, int32_t n_weights, int32_t n_importance,
                   float* samples, int32_t* inds, void* stream);

/* ---- a7: sample_stratified (VR/renderer.py:169-192), stand-alone ------------------------------ */
/* jitter [R,D] stands for the torch.rand_like draw (:177,185,190).  Scalar limits from opt (ray_start, ray_end,
 * depth_resolution, disparity_space_sampling); ray_start_per_ray / ray_end_per_ray [R] (both or neither) select the
 * per-ray branch (:183-186).  depths [R,D]. */
int tpr_sample_stratified(const float* jitter, int64_t n_rays, const float* ray_start_per_ray,
                          const float* ray_end_per_ray, const TprOptions* opt, float* depths, void* stream);

/* ---- a14: math_utils.get_ray_limits_box (VR/math_utils.py:46-98) ------------------------ */
int tpr_ray_limits_box(const float* origins, const float* dirs, int64_t n_rays,
                       float box_side_length, float* t_min, float* t_max, void* stream);

/* ---- a4 stand-alone: sample_from_planes (VR/renderer.py:55-65) ------------------------------------------------ */
/* xyz [N,P,3] -> features [N,3,P,32]: the three bilinear plane lookups of every point, NOT summed (what the reference hands
 * to OSGDecoder.forward; tpr_decode takes exactly this tensor).  grid_sample(bilinear, zeros, align_corners=False). */
int tpr_sample_planes(const float* planes_packed, int64_t n_img, int32_t height, int32_t width, const float* xyz,
                      int64_t n_pts, double box_warp, float* features, void* stream);

/* ---- a8: the density_noise term of run_model (VR/renderer.py:146): sigma[i] += noise[i] * density_noise ---------------- */
int tpr_add_density_noise(float* sigma, const float* noise, int64_t n, double density_noise, void* stream);

/* ---- a12 / a15 stand-alone: unify_samples / sort_samples (VR/renderer.py:150-167) ---------------------------------- */
/* Sort every ray's samples by depth and carry colours and densities along: depths [R,S], colours [R,S,C], densities [R,S]
 * -> *_sorted of the same shapes (ties keep their input order).  S <= TPR_MAX_SAMPLES. */
int tpr_sort_samples(const float* depths, const float* colours, const float* densities, int64_t n_rays, int32_t n_samples,
                     int32_t n_channels, float* depths_sorted, float* colours_sorted, float* densities_sorted, void* stream);

/* ---- a15: sample_from_3dgrid (VR/renderer.py:67-80; no caller in the reference) ------------------------------------ */
/* grid [G,C,D,H,W] with G == 1 (shared by the whole batch) or G == N; coords [N,P,3] as (x, y, z) in [-1,1], x walking W,
 * y walking H, z walking D -> features [N,P,C]: trilinear, zero padding, align_corners=False. */
int tpr_sample_3dgrid(const float* grid, int64_t n_grids, int32_t channels, int32_t depth, int32_t height, int32_t width,
                      const float* coords, int64_t n_batch, int64_t n_pts, float* features, void* stream);

/* ---- backward of a13 (SURVEY.md section 8(f) row 3; the reference gets it from autograd, used by
 *      training/training_loop.py:335,377) ------------------------------------------------------------------------- */
/* Gradients of L with respect to the tri-planes and the decoder, given g_rgb = dL/d(rgb) [N,M,32] (channels last, whatever
 * opt->output_layout the forward wrote), g_depth = dL/d(depth) [N,M], g_weight_sum = dL/d(weight_sum) [N,M] of one
 * tpr_render call.  N = n_img cameras.
 * depths_coarse [N*M,Dc] (tpr_sample_stratified of the forward's jitter) and depths_fine [N*M,Df] (the forward's
 * fine_depths output; NULL when Df = 0) are the sample depths of the forward, constants of the graph exactly as in the
 * reference (VR/renderer.py:198,210: torch.no_grad + detach).  From opt: box_warp, depth_resolution,
 * depth_resolution_importance, white_back, flags (decoder precision of the colour/density recomputation), and the forward's
 * frame batching:
 *   plane_sets = P > 0 (P divides n_img): camera n sampled plane set n % P; planes_packed and g_planes_packed are then
 *     [P,3,H,W,32] and the gradient of a set is the sum over its cameras.  0: one set per camera (P = N).
 *   depth_clamp_group = k: 0 = depth_range [2] (device) is the call's (min, max); k > 0 = depth_range holds
 *     2 * ceil(N / k) floats, the (min, max) of the depths of cameras [j k, j k + k) (the last group may be shorter).  The
 *     clamp of VR/ray_marcher.py:50 passes gradient only inside the camera's range.  The forward keeps per-group ranges
 *     in its scratch only; each is the min and max of the group's coarse and importance depths, so a caller reduces those.
 * Either output may be NULL when the caller does not need that gradient (its phase of the kernel is skipped).
 * g_planes_packed [P,3,H,W,32] (the layout of tpr_pack_planes; OVERWRITTEN) and g_decoder_packed
 * [tpr_packed_decoder_bytes()] (the layout of tpr_pack_decoder; OVERWRITTEN; convert with tpr_unpack_decoder_grad).
 * scratch: tpr_render_backward_scratch_bytes(n_img, n_rays, Dc + Df) bytes, plus
 * tpr_backward_deterministic_scratch_bytes(P, height, width) with TPR_BWD_DETERMINISTIC.
 * sample_colours / sample_sigma [N*M,S]: the per-sample decoder outputs kept by tpr_render_train, in ITS layout (both or
 * neither); NULL = re-evaluate them here with the point-query kernel (tpr_run_model), 3 ms more at config 2.
 * sample_features [N*M,S,32]: the summed plane features of every sample, also kept by tpr_render_train; NULL = gather
 * them again. */
size_t tpr_render_backward_scratch_bytes(int64_t n_img, int64_t n_rays, int32_t n_samples);
int tpr_render_backward(const float* planes_packed, int64_t n_img, int32_t height, int32_t width,
                        const float* decoder_packed, const float* origins, const float* dirs, int64_t n_rays,
                        const float* depths_coarse, const float* depths_fine, const float* depth_range,
                        const TprOptions* opt, const float* g_rgb, const float* g_depth, const float* g_weight_sum,
                        const float* sample_colours, const float* sample_sigma, const float* sample_features,
                        float* g_planes_packed, float* g_decoder_packed, void* scratch, size_t scratch_bytes,
                        void* stream);
/* tpr_render for a caller that will ask for gradients: additionally keeps every sample's colours (N*M*S*32 floats, an opaque
 * hand-over to tpr_render_backward: [ray][8 chunks of 4 channels][S][4], which is what the kernel's warps store as 256-byte
 * runs) and sigma [N*M,S] (the forward's sample order: ray-major, coarse then importance samples) and the importance depths
 * fine_depths [N*M,Df].  *samples_saved (host) = 1 if the kernel that ran kept them (the warp-specialised kernel), 0 if the sample
 * counts forced another kernel -- then pass NULL for them to tpr_render_backward.  The depth clamp is applied. */
int tpr_render_train(const float* planes_packed, int64_t n_img, int32_t height, int32_t width,
                     const float* decoder_packed, const float* origins, const float* dirs, int64_t n_rays,
                     const float* jitter, const float* u, const float* ray_start_per_ray, const float* ray_end_per_ray,
                     const TprOptions* opt, float* rgb, float* depth, float* weight_sum, float* fine_depths,
                     float* depth_range_io, float* sample_colours, float* sample_sigma,
                     float* sample_features /* [N*M,S,32] or NULL */, int32_t* samples_saved,
                     void* scratch, size_t scratch_bytes, void* stream);
/* packed decoder gradient -> gradients of net.0.weight [64,32], net.0.bias [64], net.2.weight [33,64], net.2.bias [33]
 * (the chain rule through the runtime gains, training/networks_stylegan2.py:118-127, and the plane mean's 1/3). */
int tpr_unpack_decoder_grad(const float* g_decoder_packed, float w1_gain, float b1_gain, float w2_gain, float b2_gain,
                            float* g_w1, float* g_b1, float* g_w2, float* g_b2, void* stream);
/* ---- backward of a8: ImportanceRenderer.run_model under autograd (TriPlaneGenerator.sample / sample_mixed,
 *      training/triplane.py:92-104; e.g. EG3D's density regulariser) -------------------------------------------- */
/* Gradients of L with respect to the tri-planes and the decoder, given g_rgb = dL/d(rgb) [N,P,32] and g_sigma = dL/d(sigma)
 * [N,P] of one tpr_run_model call on the same planes, decoder, xyz, box_warp and flags.  rgb [N,P,32] is that call's rgb output
 * (required with g_rgb).  Either upstream gradient may be NULL (= zero; not both): g_rgb = NULL is the sigma-only query and
 * reads no colours.  density_noise is additive, so g_sigma is the gradient of the noise-free sigma too.  The features are
 * gathered again (nothing per point is kept by the forward).  Either output may be NULL (not both); g_planes_packed
 * [N,3,H,W,32] and g_decoder_packed are OVERWRITTEN, in the layouts of tpr_render_backward (convert with tpr_unpack_planes /
 * tpr_unpack_decoder_grad).  flags: the forward's TPR_MLP_* (TPR_MLP_BF16 selects reduced-precision products where the
 * mma.sync fall-back runs).  scratch: tpr_run_model_backward_scratch_bytes(n_img, n_pts) bytes. */
size_t tpr_run_model_backward_scratch_bytes(int64_t n_img, int64_t n_pts);
int tpr_run_model_backward(const float* planes_packed, int64_t n_img, int32_t height, int32_t width,
                           const float* decoder_packed, const float* xyz /*[N,P,3]*/, int64_t n_pts, double box_warp,
                           const float* rgb /*[N,P,32] or NULL*/, const float* g_rgb /*[N,P,32] or NULL*/,
                           const float* g_sigma /*[N,P] or NULL*/, int32_t flags,
                           float* g_planes_packed /*or NULL*/, float* g_decoder_packed /*or NULL*/,
                           void* scratch, size_t scratch_bytes, void* stream);
/* Extra scratch of the deterministic backward (TPR_BWD_DETERMINISTIC), on top of tpr_render_backward_scratch_bytes /
 * tpr_run_model_backward_scratch_bytes: the int64 plane-gradient accumulator [N,3,H,W,32] plus 512 per-CTA rows of the
 * packed decoder gradient (a launch in this mode uses at most 512 CTAs) and 256 bytes.  0 for a bad shape.  For
 * tpr_render_backward with plane_sets = P > 0 pass P as n_img: the accumulator holds one entry per plane set. */
size_t tpr_backward_deterministic_scratch_bytes(int64_t n_img, int32_t height, int32_t width);
/* the two stages of tpr_render_backward, stand-alone (tests): the march's backward -- sigma [R,S], colours [R,S,32] of
 * the samples in forward order -> g_sigma [R,S] and the composite weight omega [R,S] of each sample's colour
 * (dL/d(colour_c) = 2 * g_rgb_c * omega) */
int tpr_march_backward(const float* depths_coarse, const float* depths_fine, int32_t dc, int32_t df, const float* sigma,
                       const float* colours, const float* g_rgb, const float* g_depth, const float* g_weight_sum,
                       const float* depth_range, int32_t white_back, int64_t n_rays_total, float* g_sigma, float* omega,
                       void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TRIPLANE_B200_H_ */
