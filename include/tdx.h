/*
 * tdx.h -- C ABI of the B200-native InfiniteDiffusion sampling hot path (libtdx.so).
 *
 * Plain C: pointers, sizes, POD structs.  No torch / C++ types cross this boundary.  Every device pointer is owned
 * by the caller unless a handle says otherwise; every launch goes to the `stream` argument (a CUstream/cudaStream_t
 * passed as void*).  All functions return 0 on success or a negative TDX_E_* code; tdx_last_error() returns a
 * human-readable message for the calling thread.  There is no CPU fallback anywhere behind this header.
 *
 * Devices and streams: the library launches on the CURRENT device (it never calls cudaSetDevice) -- make the device
 * that owns the pointers current before a call.  Per-device state (split-K scratch, opted-in kernel attributes, SM
 * count) is created the first time a device is used and must not be created inside a stream capture: call
 * tdx_program_add_* / tdx_igemm_run once outside a capture first.  The split-K scratch is ONE buffer per device:
 * launches on the same device must be stream-ordered with respect to each other (the reference drives its models from
 * one thread and one stream, world_pipeline.py; so does the Python host here).  Not thread-safe per handle.
 *
 * Each entry point cites the reference interface (xandergos/terrain-diffusion @ 82a0431) it replaces.
 * The reference has no FFI of its own (pure Python); INTEGRATION.md shows the ctypes stub a maintainer would add.
 *
 * Activation layout ("NC8HW8"): a [N, C, H, W] activation is stored as bf16 [N][C/8][H][W][8] -- channel groups of 8
 * (16 bytes) are the innermost unit, so a TMA box of (W-run x rows x groups) lands in shared memory exactly in the
 * tcgen05 K-major no-swizzle core-matrix order, and one thread's 8-channel store is a 16-byte vector.
 */
#ifndef TDX_H_
#define TDX_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TDX_OK 0
#define TDX_E_INVALID -1   /* bad argument / unsupported shape */
#define TDX_E_CUDA -2      /* CUDA runtime / driver error */
#define TDX_E_UNSUPPORTED -3

const char* tdx_last_error(void);
/* Library + device probe: fills sm count, compute capability; fails if the device is not sm_100. */
int tdx_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* sizeof() of the public structs (0: TdxOutSpec, 1: TdxIgemmDesc, 2: TdxConvInDesc, 3: TdxConvOutDesc, 4: TdxEmbedBlock, 5: TdxEmbedDesc, 6: TdxAttnDesc, 7: TdxIm2colDesc, 8: TdxConvOutGuidedDesc) so bindings can verify their layout. */
int tdx_abi_sizeof(int which);

/* ------------------------------------------------------------------------------------------------------------------
 * Implicit-GEMM convolution on tcgen05 (the operator under MPConv.forward, models/mp_layers.py:201-221, with the
 * surrounding UNetBlock elementwise math, models/unet_block.py:116-156, fused into its epilogue).
 *
 * out[m, n] = sum over segments s, taps (r,c), channels k of  A_s[pixel(m)+(r-1,c-1), k] * B[n, s, k, r, c]
 *   m: output pixel inside a 16x8 tile (M = 128), n: output channel (64 per work item), K = sum_s taps_s * C_s.
 * Up to 3 K-segments (e.g. the two halves of an mp_concat, or a 3x3 residual conv + a 1x1 skip conv fused as extra K).
 * ------------------------------------------------------------------------------------------------------------------ */
enum { TDX_OUT_NONE = 0, TDX_OUT_RAW = 1, TDX_OUT_SILU = 2, TDX_OUT_PNORM_SILU = 3 };
enum { TDX_SP_SAME = 0, TDX_SP_DOWN2 = 1, TDX_SP_UP2 = 2 };
enum { TDX_EPI_EMB_SILU = 1, TDX_EPI_RESID = 2, TDX_EPI_PNORM = 4 };

typedef struct TdxOutSpec {
  void* ptr;      /* bf16 NC8HW8, Cout channels; spatial size per `spatial` */
  int32_t kind;   /* TDX_OUT_*: raw v | mp_silu(scale*v) | mp_silu(pixelnorm(v)) */
  int32_t spatial;/* TDX_SP_*: same HxW | every 2nd pixel into H/2 x W/2 | nearest x2 into 2H x 2W */
  float scale;
  int32_t _pad;
} TdxOutSpec;

typedef struct TdxIgemmDesc {
  /* A operand: up to 3 activation tensors (bf16 NC8HW8, all n_img x C_s x H x W) */
  const void* a_ptr[3];
  int32_t a_channels[3];   /* multiple of 64 */
  int32_t a_taps[3];       /* 9 (3x3, pad 1) or 1 (1x1) */
  int32_t n_seg;
  /* B operand: packed bf16 weights [c_out/n_per_item slices][stage = (segment, 64-ch chunk, tap)][8][n_per_item][8] */
  const void* b_packed;
  int32_t c_out;           /* multiple of 64, <= 256 */
  int32_t n_per_item;      /* output channels per work item = MMA N the weights were packed for (tdx_igemm_choose_n) */
  int32_t n_img, height, width;   /* output == input spatial size; multiples of 8 */
  /* epilogue */
  int32_t epi_flags;       /* TDX_EPI_* */
  const float* cvec;       /* [n_img][c_out] fp32 embedding scale (TDX_EPI_EMB_SILU): v = mp_silu(v * c)          */
  const void* resid;       /* bf16 NC8HW8 residual (TDX_EPI_RESID): v = v + resid_scale * r'                      */
  int32_t resid_spatial;   /* TDX_SP_SAME | TDX_SP_UP2 (r is H/2 x W/2) | TDX_SP_DOWN2 (r is 2H x 2W)            */
  int32_t resid_pnorm;     /* r' = pixelnorm(r) over channels (unet_block.py:121) when non-zero                  */
  float resid_scale;
  float clip;              /* > 0: v = clamp(v, -clip, +clip) after the residual (unet_block.py:153-154); 0: off  */
  TdxOutSpec out[3];
  /* Pixel-norm side channel (fp32 [n_img][H][W] planes).  A launch that computes the pixel-norm of its result (a
   * TDX_OUT_PNORM_SILU output or TDX_EPI_PNORM) can also store the per-pixel factor 1 / (1e-4 + rms over c_out) in
   * rms_out; the launch that later adds pixelnorm(that tensor) as its residual passes the plane as resid_inv (with
   * resid_pnorm = 0: r' = r * resid_inv[pixel], at the residual's resolution) instead of re-reading every channel of
   * the residual to recompute it.  Both may be NULL. */
  float* rms_out;
  const float* resid_inv;
  /* Split-K factor: 0 = the library's cost model picks it (together with the residency of the weights); > 0 forces it
   * (the launch fails with TDX_E_INVALID when that split is impossible for the shape).  Used with n_per_item by the
   * measured per-shape table terrain_diffusion_b200/tuned_shapes.json (tools/tune_igemm.py). */
  int32_t k_split;
  int32_t _reserved;
} TdxIgemmDesc;

/* Output channels per work item (64/128/192/256) the library prefers for this launch shape: balances the MMA issue
 * pipe time (max(48, N/2) cycles per K=16 step), L2->SM traffic and CTA count.  Pack the weights for this value. */
int tdx_igemm_choose_n(int32_t c_out, int32_t n_img, int32_t height, int32_t width, const int32_t* a_channels,
                       const int32_t* a_taps, int32_t n_seg);
/* Elements of packed B for a descriptor's segments. */
int64_t tdx_igemm_packed_weight_elems(const int32_t* a_channels, const int32_t* a_taps, int32_t n_seg, int32_t c_out);
/* One launch of the persistent tcgen05 kernel. */
int tdx_igemm_run(const TdxIgemmDesc* desc, void* stream);


/* ------------------------------------------------------------------------------------------------------------------
 * First convolution (EDMUnet2D.forward, models/edm_unet.py:168-172: cat([x, ones]) -> enc['..._conv'] = MPConv 3x3).
 * Reads the caller's planar NCHW input directly (up to two sources, e.g. the scaled noisy sample and the conditioning
 * image of sample_decoder_diffusion_tiled, training/evaluation/sample_diffusion_decoder.py:108-110), appends the
 * ones channel (zero-padded at the border like the reference's conv), and writes bf16 NC8HW8 outputs.
 * ------------------------------------------------------------------------------------------------------------------ */
typedef struct TdxConvInDesc {
  const void* src[2];        /* NCHW planar, n_img x src_channels[i] x H x W */
  int32_t src_channels[2];   /* channels of each source (second may be 0) */
  int32_t src_dtype[2];      /* 0 = fp32, 1 = bf16 */
  const float* src_scale[2]; /* optional DEVICE scalar multiplied into source i (precondition_inputs), or NULL */
  const float* weight;       /* fp32 effective weights, tap-major [3*3][sum(src_channels)+1][c_out] (ones channel last) */
  int32_t c_out;             /* multiple of 64, <= 256; sum(src_channels) <= 15 */
  int32_t n_img, height, width;
  TdxOutSpec out[3];         /* same semantics as TdxIgemmDesc.out (TDX_SP_SAME only) */
} TdxConvInDesc;
int tdx_conv_in_run(const TdxConvInDesc* desc, void* stream);

/* The same first convolution on the tensor cores: this launch only gathers the 3x3 neighbourhood of every pixel into
 * a bf16 NC8HW8 tensor of k_pad "channels" -- channel k = tap * ci + c for tap = 3*dy+dx in 0..8 and c in
 * 0..ci-1 (ci = sum(src_channels) + 1, the ones channel last; zero outside the image, like the reference's padded
 * conv), zero for k >= 9*ci -- and the convolution itself becomes a 1x1 tdx_igemm_run over that tensor with the
 * weight matrix [c_out][k_pad] (so it gets the igemm epilogue: pixel-norm, silu, three outputs).  The inputs and
 * weights are rounded to bf16, as in the reference's bf16 autocast of models/edm_unet.py:168-172. */
typedef struct TdxIm2colDesc {
  const void* src[2];        /* NCHW planar, n_img x src_channels[i] x H x W */
  int32_t src_channels[2];   /* channels of each source (second may be 0) */
  int32_t src_dtype[2];      /* 0 = fp32, 1 = bf16 */
  const float* src_scale[2]; /* optional DEVICE scalar multiplied into source i, or NULL */
  void* out;                 /* bf16 NC8HW8 [n_img][k_pad/8][H][W][8] */
  int32_t k_pad;             /* 9 * (sum(src_channels) + 1) rounded up to a multiple of 64; sum = 5 or 11 */
  int32_t n_img, height, width;
} TdxIm2colDesc;
int tdx_im2col_run(const TdxIm2colDesc* desc, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Last convolution (out_conv with out_gain folded, models/edm_unet.py:179) + optionally the whole scheduler update
 * (EDMDPMSolverMultistepScheduler.step, scheduler/dpmsolver.py:650-726, closed form of SURVEY.md Appendix B):
 *     F  = conv3x3(x_raw)                          -> model_out (fp32 NCHW, optional)
 *     x0 = c_skip*sample + c_out*F ; sample' = r*sample + (1-r)*x0 + k*(x0 - x0_prev) ; x0_prev = x0
 * coef points at DEVICE floats {c_skip, c_out, r, k}.
 * ------------------------------------------------------------------------------------------------------------------ */
typedef struct TdxConvOutDesc {
  const void* x;           /* bf16 NC8HW8, n_img x c_in x H x W */
  int32_t c_in;            /* multiple of 8 */
  const float* weight;     /* fp32 effective weights, tap-major [3*3][c_in][c_out == 1 ? 1 : 8] (zero padded) */
  int32_t c_out;           /* 1..8 */
  int32_t n_img, height, width;
  float* model_out;        /* fp32 NCHW [n_img][c_out][H][W] or NULL */
  const float* sched_coef; /* DEVICE {c_skip, c_out, r, k} or NULL (no scheduler fusion) */
  float* sample;           /* fp32 NCHW, updated in place (requires sched_coef) */
  float* x0_prev;          /* fp32 NCHW solver history, read+written (requires sched_coef) */
} TdxConvOutDesc;
int tdx_conv_out_run(const TdxConvOutDesc* desc, void* stream);
/* The same launch with two-model autoguidance (EDM2 autoguidance; sample_diffusion_base.py:105-110,
 * sample_diffusion_decoder.py:112-117) applied to the convolution's result before the update:
 *     F_m = conv3x3(x_raw) ;  F = F_g + s*(F_m - F_g)   (separately rounded sub, mul, add)
 *     x0  = c_skip*sample + c_out*F ; sample' = r*sample + (1-r)*x0 + k*(x0 - x0_prev) ; x0_prev = x0
 * F_g (guide_out) is the guide model's output, fp32 NCHW [n_img][c_out][H][W], e.g. written earlier in the same program
 * by the guide's own last convolution in plain model_out mode.  base.sched_coef is required and points at FIVE device
 * floats {c_skip, c_out, r, k, s}: the guidance scale lives in the table, so a recorded program can change it without
 * being rebuilt.  base.model_out (optional) receives the combined F. */
typedef struct TdxConvOutGuidedDesc {
  TdxConvOutDesc base;
  const float* guide_out;
} TdxConvOutGuidedDesc;
int tdx_conv_out_guided_run(const TdxConvOutGuidedDesc* desc, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Embedding path (EDMUnet2D.compute_embeddings, models/edm_unet.py:145-159, + the per-block modulation vector of
 * UNetBlock.forward, models/unet_block.py:129-131):
 *     emb  = mp_silu(noise_linear(MPPositionalEmbedding(t)))        (or a caller-computed emb for conditional models)
 *     c_b  = emb_linear_b(emb)*gain_b + 1 ;  c_b /= sqrt(mean(c_b^2) + 1e-8)          for every block b
 * ------------------------------------------------------------------------------------------------------------------ */
typedef struct TdxEmbedBlock {
  const float* weight;   /* fp32 effective, TRANSPOSED [emb_channels][c_out], emb_gain folded */
  float* cvec;           /* fp32 [n_img][c_out] */
  int32_t c_out;
  int32_t _pad;
} TdxEmbedBlock;
typedef struct TdxEmbedDesc {
  const float* noise_labels;   /* DEVICE fp32 [n_img] (trigflow t); used when emb_in is NULL */
  const float* emb_in;         /* DEVICE fp32 [n_img][emb_channels] precomputed embedding, or NULL */
  const float* noise_weight;   /* fp32 effective, TRANSPOSED [noise_dims][emb_channels] */
  const float* noise_freqs;    /* DEVICE fp32 [noise_dims/2]: the model's MPPositionalEmbedding.freqs buffer */
  int32_t noise_dims;          /* even, <= 256 */
  int32_t emb_channels;        /* <= 1024 */
  int32_t n_img;
  int32_t n_blocks;
  const TdxEmbedBlock* blocks; /* HOST array of n_blocks entries (copied by the call) */
} TdxEmbedDesc;
int tdx_embed_run(const TdxEmbedDesc* desc, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Cosine self-attention core of UNetBlock.attn (models/unet_block.py:102-108) between the qkv and proj 1x1 convs
 * (which run as tdx_igemm launches): per-head pixel-norm of q, k, v; softmax(q^T k / sqrt(d)); weighted sum of v.
 * q, k, v, out: bf16 NC8HW8 with channel = head*64 + d, spatial size tokens = H*W.
 * ------------------------------------------------------------------------------------------------------------------ */
typedef struct TdxAttnDesc {
  const void* q;
  const void* k;
  const void* v;
  void* out;
  int32_t n_img, heads, head_dim, tokens;
} TdxAttnDesc;
int tdx_attn_run(const TdxAttnDesc* desc, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Scheduler / consistency / blend elementwise kernels (fp32, vectorised).
 * ------------------------------------------------------------------------------------------------------------------ */
/* scheduler.step closed form on a standalone model output (dpmsolver.py:650-726); coef = host floats. */
int tdx_sched_step(float* sample, const float* model_out, float* x0_prev, int64_t numel, float c_skip, float c_out,
                   float r, float k, void* stream);
/* canvas_val[c, y0+y, x0+x] += tile[c,y,x]*w[y,x] ; canvas_w[y0+y, x0+x] += w[y,x]   (sample_diffusion_decoder.py
 * :122-123; infinite_tensor's window sum).  Separate rounding of the product and the sum (no FMA contraction), so
 * applying tiles in the reference's row-major order reproduces its fp32 result bit for bit. */
int tdx_blend_accumulate(float* canvas_val, float* canvas_w, int32_t channels, int32_t canvas_h, int32_t canvas_w_px,
                         const float* tile, const float* window, int32_t tile_h, int32_t tile_w, int32_t y0,
                         int32_t x0, void* stream);
/* dst[c, y0+y, x0+x] += tile[c, y, x] (fp32, clipped to dst): the window-sum of the reference's canvas engine
 * (infinite_tensor: "sums overlapping window outputs", annotated_infinite_panorama.py:141-146) for tiles that are
 * already packed as (x*w, w). */
int tdx_canvas_add(float* dst, int32_t channels, int32_t dst_h, int32_t dst_w, const float* tile, int32_t tile_h,
                   int32_t tile_w, int32_t y0, int32_t x0, void* stream);
/* out = canvas_val / canvas_w [/ divisor]   (normalise-on-read, world_pipeline.py:1223,1301; the bounded samplers
 * divide by sigma_data afterwards, sample_diffusion_decoder.py:211).  divisor == 1 skips the second division. */
int tdx_blend_normalize(float* out, const float* canvas_val, const float* canvas_w, int32_t channels, int64_t plane,
                        float divisor, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Elementwise glue of the consistency stages (WorldPipeline._latent_inference / _decoder_inference,
 * inference/world_pipeline.py:1052-1131,1209-1242); the U-Net and the TrigFlow update s' = cos t*x_t - sin t*sigma_d*pred
 * run as a one-step program whose last convolution applies the update (tdx_conv_out_run coefficients
 * {cos t, sin t*sigma_d, 0, 0}).
 * ------------------------------------------------------------------------------------------------------------------ */
/* x_t = a*sample + b*noise (world_pipeline.py:1097-1098,1235: a = cos t, b = sin t*sigma_data); sample may be NULL (0). */
int tdx_trig_mix(float* out, const float* sample, const float* noise, int64_t numel, float a, float b, void* stream);
/* out[n][c] = x[n][c]*scale*w, out[n][C] = w: the packed window output cat([x*w, w]) (world_pipeline.py:1130,1242). */
int tdx_pack_weighted(float* out, const float* x, const float* w, int32_t n_img, int32_t channels, int64_t plane,
                      float scale, void* stream);
/* cond[n][c] = nearest_upsample(packed[n][c] / packed[n][last], factor) for c < keep: normalise-on-read of a packed
 * window + F.interpolate(mode='nearest') (world_pipeline.py:1223-1226). */
int tdx_window_to_cond(float* out, const float* packed, int32_t n_img, int32_t packed_channels, int32_t keep, int32_t h,
                       int32_t w, int32_t factor, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Elevation read-out (WorldPipeline._compute_elev, inference/world_pipeline.py:1277-1313): the reference normalises
 * the canvases on read and runs data/laplacian_encoder.py (torchvision resize + gaussian_blur) on the CPU for every
 * get().  These five fp32 primitives keep it on the device; terrain_diffusion_b200/inference/postproc.py composes them
 * exactly like laplacian_decode / laplacian_encode / laplacian_denoise.  All tensors are contiguous [h][w] fp32 unless a
 * pitch (in elements) is given.
 * ------------------------------------------------------------------------------------------------------------------ */
/* out = num / den * scale + offset   (world_pipeline.py:1301-1304: (sum x*w)/(sum w) * STD + MEAN) */
int tdx_post_normalize(const float* num, const float* den, int64_t pitch, float* out, int32_t h, int32_t w, float scale,
                       float offset, void* stream);
/* pad_linear_extrapolation (laplacian_encoder.py:6-40): out is (h+2) x (w+2) */
int tdx_post_pad_extrapolate(const float* x, int32_t h, int32_t w, float* out, void* stream);
/* One axis of TF.resize(..., BILINEAR) = torch interpolate(bilinear, align_corners=False, antialias=True): axis 1
 * resizes the width to out_size ([h][w] -> [h][out_size]), axis 0 the height.  torch resizes the width first. */
int tdx_resize_aa_axis(const float* x, int32_t h, int32_t w, float* out, int32_t out_size, int32_t axis, void* stream);
/* TF.gaussian_blur(x, kernel_size, sigma): reflect padding, outer product of two normalised 1-D Gaussians. */
int tdx_gaussian_blur(const float* x, int32_t h, int32_t w, float* out, int32_t ksize, float sigma, void* stream);
/* out[y][x] = f(a[y][x] + b[y][x]) over an h x w window of two pitched tensors (pass the pointers of the window's
 * first element): f = identity (laplacian_decode, laplacian_encoder.py:131) or sign(v) v^2 (world_pipeline.py:1312);
 * out_i16 (optional) additionally receives clip(floor(v), -32768, 32767) (api.py:73-77).  out or out_i16 may be NULL. */
int tdx_post_combine(const float* a, int64_t a_pitch, const float* b, int64_t b_pitch, float* out, int16_t* out_i16,
                     int32_t h, int32_t w, int32_t signed_square, void* stream);

/* Climate read-out (WorldPipeline._compute_climate, inference/world_pipeline.py:1314-1365).
 * tdx_lapse_rate = local_baseline_temperature_torch (inference/postprocessing.py:262-326) on the normalised coarse
 * planes: `coarse_elev_sqrt` is coarse channel 0 (signed square root of metres; e = max(0, c)^2 inside), `temp` channel
 * 2; outputs are the (h-win+1) x (w-win+1) valid-window maps of sea-level temperature and lapse rate. */
int tdx_lapse_rate(const float* temp, const float* coarse_elev_sqrt, int32_t h, int32_t w, int32_t win, float beta_lo,
                   float beta_hi, float fallback_beta, float eps, float fallback_threshold, float* t_sea, float* beta,
                   void* stream);
/* Bilinear, border-clamped grid_sample (align_corners=False) of [t_sea, beta, coarse channels 3..5] at the centres of
 * pixels [i1, i1+h) x [j1, j1+w) (one coarse cell = coarse_stride pixels, window origin cell (ci1, cj1); the sampled
 * part of `coarse` [n_ch][hc][wc] starts at (crop, crop) and has the size of t_sea) and the lapse-rate correction:
 * out[5][h][w] = {t_sea + beta*max(elev, 0), coarse 3, coarse 4, coarse 5, beta}. */
int tdx_climate_sample(const float* t_sea, const float* beta, const float* coarse, int32_t n_ch, int32_t hc, int32_t wc,
                       int32_t crop, const float* elev, int32_t i1, int32_t j1, int32_t h, int32_t w,
                       int32_t coarse_stride, int32_t ci1, int32_t cj1, float* out, void* stream);

/* Tile-seeded N(0,1) field, bit-exact with inference/portable_rng.py + world_pipeline.py:66-115 */
int tdx_noise_patch(uint64_t base_seed, int64_t y0, int64_t x0, int32_t h, int32_t w, int32_t channels,
                    int32_t tile_h, int32_t tile_w, float* out, void* workspace, int64_t workspace_bytes,
                    void* stream);
int64_t tdx_noise_patch_workspace_bytes(int32_t channels, int32_t tile_h, int32_t tile_w);
/* Batched form (one call for all windows of a stage batch, world_pipeline.py:1085-1092 runs this per tile in a Python
 * loop): n_patches patches of one shape, origins in HOST arrays, out = [n][C][h][w]; bit-identical to n single calls. */
int tdx_noise_patches(uint64_t base_seed, int32_t n_patches, const int64_t* y0s, const int64_t* x0s, int32_t h, int32_t w,
                      int32_t channels, int32_t tile_h, int32_t tile_w, float* out, void* workspace,
                      int64_t workspace_bytes, void* stream);
int64_t tdx_noise_patches_workspace_bytes(int32_t channels, int32_t tile_h, int32_t tile_w);
/* portable_rng.standard_normal(seed, n) (inference/portable_rng.py:77-82): one raw stream, bit-exact;
 * workspace >= tdx_noise_patch_workspace_bytes(1, 1, n). */
int tdx_standard_normal(uint64_t seed, int64_t n, float* out, void* workspace, int64_t workspace_bytes, void* stream);
/* Synchronises `stream` and reports whether the last tdx_noise_patch on `workspace` completed its streams. */
int tdx_noise_patch_status(void* workspace, void* stream);
/* _tile_seed (world_pipeline.py:58-63): 64-bit seed of tile (ty, tx); host-side integer hash. */
uint64_t tdx_tile_seed(uint64_t base_seed, int64_t ty, int64_t tx);

/* ------------------------------------------------------------------------------------------------------------------
 * Program: a recorded sequence of the launches above with pre-built TMA descriptors, replayed as one CUDA graph.
 * This is what EDMUnet2D.forward / the N-step tile sampler become: the Python host plans the launch list once per
 * (model, batch, H, W) and then issues ONE call per forward (or per whole N-step solve).
 * ------------------------------------------------------------------------------------------------------------------ */
typedef struct TdxProgram TdxProgram;
int tdx_program_create(TdxProgram** out);
int tdx_program_add_conv_in(TdxProgram* p, const TdxConvInDesc* d);
int tdx_program_add_im2col(TdxProgram* p, const TdxIm2colDesc* d);
int tdx_program_add_igemm(TdxProgram* p, const TdxIgemmDesc* d);
int tdx_program_add_conv_out(TdxProgram* p, const TdxConvOutDesc* d);
int tdx_program_add_conv_out_guided(TdxProgram* p, const TdxConvOutGuidedDesc* d);
int tdx_program_add_embed(TdxProgram* p, const TdxEmbedDesc* d);
int tdx_program_add_attn(TdxProgram* p, const TdxAttnDesc* d);
int tdx_program_num_launches(const TdxProgram* p);
/* use_graph != 0: capture on first run, replay afterwards. */
int tdx_program_run(TdxProgram* p, int use_graph, void* stream);
/* Capture + instantiate + upload the graph without running it (keeps one-time costs out of timed regions). */
int tdx_program_instantiate(TdxProgram* p, void* stream);
/* Eager run with a CUDA event pair around every launch: ms_per_launch[i] = device time of launch i (in program
 * order, tdx_program_num_launches entries); kinds[i] = 0 conv_in, 1 igemm, 2 conv_out (guided or not), 3 embed, 4 attn, 5 im2col.  Synchronises. */
int tdx_program_profile(TdxProgram* p, float* ms_per_launch, int32_t* kinds, void* stream);
int tdx_program_destroy(TdxProgram* p);

#ifdef __cplusplus
}
#endif
#endif /* TDX_H_ */
