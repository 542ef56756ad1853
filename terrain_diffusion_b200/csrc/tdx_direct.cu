// CUDA-core kernels around the tensor-core path: first / last convolution (tiny K or tiny N), the embedding /
// modulation vectors, and the fp32 elementwise scheduler + blend kernels.  All HBM-bound or launch-bound; the design
// rules that matter are coalescing (threads walk x), 16-byte vectors on the NC8HW8 side and broadcast smem weights.
#include "tdx_common.h"
#include "tdx_ptx.cuh"

namespace tdx {

__device__ __forceinline__ float mp_silu_precise(float x) { return x / (1.0f + expf(-x)) / 0.596f; }

// ------------------------------------------------------------------------------------------------ first conv
constexpr int kConvInGroups = 4;   // 32-pixel groups per block (amortises the weight staging)
constexpr int kConvOutGroups = 1;  // conv_out stages only 9*C*COUT weights: more, smaller blocks keep every SM busy

struct ConvInParams {
  const void* src[2];
  int src_ch[2];
  int src_dtype[2];
  const float* src_scale[2];
  const float* weight;
  int ci;  // total input channels incl. the ones channel
  int cout;
  int H, W;
  TdxOutSpec out[3];
};

__device__ __forceinline__ float load_in(const void* base, int dtype, size_t idx) {
  if (dtype == 0) return __ldg(reinterpret_cast<const float*>(base) + idx);
  return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(base)[idx]);
}

// Block = 128 threads = 32 consecutive pixels x 4 warps; warp w computes output channels [oc0 + 16w, oc0 + 16w + 16)
// of each 64-channel group, so weights are warp-broadcast shared-memory reads and every store is a 512-byte row of
// 16-byte pixel vectors.
template <int CI>
__global__ void __launch_bounds__(128) conv_in_kernel(const ConvInParams p) {
  extern __shared__ float ws[];  // [tap][ci][cout]
  __shared__ float ssq[4][32];
  const int CO = p.cout;
  for (int i = threadIdx.x; i < (9 * CI * CO) / 4; i += blockDim.x)
    reinterpret_cast<float4*>(ws)[i] = __ldg(reinterpret_cast<const float4*>(p.weight) + i);
  pdl_launch_dependents();
  pdl_wait();  // the sources / scale come from earlier kernels; weights above are constants
  __syncthreads();
  const int img = blockIdx.y;
  const int lane = threadIdx.x & 31, wq = threadIdx.x >> 5;
  for (int grp = 0; grp < kConvInGroups; ++grp) {
  const int pix = (blockIdx.x * kConvInGroups + grp) * 32 + lane;
  const bool inb = pix < p.H * p.W;
  const int y = inb ? pix / p.W : 0, x = inb ? pix % p.W : 0;
  const size_t plane = (size_t)p.H * p.W;
  const float s0 = p.src_scale[0] ? __ldg(p.src_scale[0]) : 1.0f;
  const float s1 = p.src_scale[1] ? __ldg(p.src_scale[1]) : 1.0f;
  const int c0n = p.src_ch[0], c1n = p.src_ch[1];
  const int C8 = CO >> 3;

  float sumsq = 0.f;
  for (int oc0 = 0; oc0 < CO; oc0 += 64) {
    const int oc = oc0 + wq * 16;
    float acc[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) acc[j] = 0.f;
#pragma unroll 1
    for (int tap = 0; tap < 9; ++tap) {
      // the CI input values of this tap (zero padded at the border, ones channel included), loaded as one batch
      const int yy = y + tap / 3 - 1, xx = x + tap % 3 - 1;
      const bool ok = inb && yy >= 0 && yy < p.H && xx >= 0 && xx < p.W;
      const size_t off = (size_t)yy * p.W + xx;
      float in[CI];
#pragma unroll
      for (int ci = 0; ci < CI; ++ci) {
        float v = 0.f;
        if (ok) {
          if (ci < c0n) v = load_in(p.src[0], p.src_dtype[0], ((size_t)img * c0n + ci) * plane + off) * s0;
          else if (ci < c0n + c1n) v = load_in(p.src[1], p.src_dtype[1], ((size_t)img * c1n + (ci - c0n)) * plane + off) * s1;
          else v = 1.0f;
        }
        in[ci] = v;
      }
#pragma unroll
      for (int ci = 0; ci < CI; ++ci) {
        {
          const float v = in[ci];
          const float4* w4 = reinterpret_cast<const float4*>(ws + (tap * CI + ci) * CO + oc);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 w = w4[j];
            acc[4 * j + 0] = fmaf(w.x, v, acc[4 * j + 0]);
            acc[4 * j + 1] = fmaf(w.y, v, acc[4 * j + 1]);
            acc[4 * j + 2] = fmaf(w.z, v, acc[4 * j + 2]);
            acc[4 * j + 3] = fmaf(w.w, v, acc[4 * j + 3]);
          }
        }
      }
    }
#pragma unroll
    for (int j = 0; j < 16; ++j) sumsq = fmaf(acc[j], acc[j], sumsq);
    if (inb) {
#pragma unroll
      for (int o = 0; o < 3; ++o) {
        const TdxOutSpec& os = p.out[o];
        if (os.kind != TDX_OUT_RAW && os.kind != TDX_OUT_SILU) continue;
        uint4* optr = reinterpret_cast<uint4*>(os.ptr) + ((size_t)img * C8 + (oc >> 3)) * plane + pix;
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          float w[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float t = acc[g * 8 + i];
            w[i] = os.kind == TDX_OUT_RAW ? t : mp_silu_f(t * os.scale);
          }
          uint4 u;
          u.x = pack_bf16x2(w[0], w[1]); u.y = pack_bf16x2(w[2], w[3]);
          u.z = pack_bf16x2(w[4], w[5]); u.w = pack_bf16x2(w[6], w[7]);
          optr[(size_t)g * plane] = u;
        }
      }
    }
  }
  bool want_pnorm = false;
  const uint4* raw_ptr = nullptr;
#pragma unroll
  for (int o = 0; o < 3; ++o) {
    if (p.out[o].kind == TDX_OUT_PNORM_SILU) want_pnorm = true;
    if (p.out[o].kind == TDX_OUT_RAW) raw_ptr = reinterpret_cast<const uint4*>(p.out[o].ptr);
  }
  if (want_pnorm) {
    // per-pixel sum of squares over all channels = sum over the 4 warps; then re-read this warp's own raw outputs
    ssq[wq][lane] = sumsq;
    __syncthreads();
    const float tot = ssq[0][lane] + ssq[1][lane] + ssq[2][lane] + ssq[3][lane];
    const float inv = 1.0f / (1e-4f + sqrtf(tot / (float)CO));
    if (inb) {
#pragma unroll
      for (int o = 0; o < 3; ++o) {
        const TdxOutSpec& os = p.out[o];
        if (os.kind != TDX_OUT_PNORM_SILU) continue;
        for (int oc0 = 0; oc0 < CO; oc0 += 64) {
#pragma unroll
          for (int g = 0; g < 2; ++g) {
            const size_t idx = ((size_t)img * C8 + ((oc0 + wq * 16) >> 3) + g) * plane + pix;
            const uint4 u = raw_ptr[idx];
            float a[8];
            unpack_bf16x2(u.x, a[0], a[1]); unpack_bf16x2(u.y, a[2], a[3]);
            unpack_bf16x2(u.z, a[4], a[5]); unpack_bf16x2(u.w, a[6], a[7]);
            uint4 r;
            r.x = pack_bf16x2(mp_silu_f(a[0] * inv), mp_silu_f(a[1] * inv));
            r.y = pack_bf16x2(mp_silu_f(a[2] * inv), mp_silu_f(a[3] * inv));
            r.z = pack_bf16x2(mp_silu_f(a[4] * inv), mp_silu_f(a[5] * inv));
            r.w = pack_bf16x2(mp_silu_f(a[6] * inv), mp_silu_f(a[7] * inv));
            reinterpret_cast<uint4*>(os.ptr)[idx] = r;
          }
        }
      }
    }
  }
  __syncthreads();  // ssq is reused by the next pixel group
  }
}

int direct_prepare();

int conv_in_validate(const TdxConvInDesc& d) {
  TDX_REQUIRE(d.src[0] && d.src_channels[0] > 0, "conv_in: src[0] missing");
  TDX_REQUIRE(d.src_channels[1] == 0 || d.src[1], "conv_in: src[1] missing");
  TDX_REQUIRE(d.weight, "conv_in: weight is null");
  TDX_REQUIRE(d.c_out >= 64 && d.c_out <= 256 && d.c_out % 64 == 0, "conv_in: c_out=%d (multiple of 64)", d.c_out);
  TDX_REQUIRE(d.src_channels[0] + d.src_channels[1] + 1 == 6 || d.src_channels[0] + d.src_channels[1] + 1 == 12,
              "conv_in: %d input channels; instantiated for 5 (decoder / latent models) or 11 (coarse model)",
              d.src_channels[0] + d.src_channels[1]);
  TDX_REQUIRE(d.n_img >= 1 && d.height >= 1 && d.width >= 1, "conv_in: bad shape");
  const int ci = d.src_channels[0] + d.src_channels[1] + 1;
  TDX_REQUIRE(9 * ci * d.c_out * 4 <= 200 * 1024, "conv_in: weights (%d in, %d out) exceed shared memory", ci, d.c_out);
  bool has_raw = false, has_pn = false;
  for (int o = 0; o < 3; ++o) {
    if (d.out[o].kind == TDX_OUT_NONE) continue;
    TDX_REQUIRE(d.out[o].ptr, "conv_in: out[%d].ptr is null", o);
    TDX_REQUIRE(d.out[o].spatial == TDX_SP_SAME, "conv_in: only TDX_SP_SAME outputs");
    has_raw |= d.out[o].kind == TDX_OUT_RAW;
    has_pn |= d.out[o].kind == TDX_OUT_PNORM_SILU;
  }
  TDX_REQUIRE(!has_pn || has_raw, "conv_in: a PNORM_SILU output needs a RAW output too");
  return TDX_OK;
}

int conv_in_launch(const TdxConvInDesc& d, cudaStream_t stream) {
  ConvInParams p;
  for (int i = 0; i < 2; ++i) {
    p.src[i] = d.src[i];
    p.src_ch[i] = d.src_channels[i];
    p.src_dtype[i] = d.src_dtype[i];
    p.src_scale[i] = d.src_scale[i];
  }
  p.weight = d.weight;
  p.ci = d.src_channels[0] + d.src_channels[1] + 1;
  p.cout = d.c_out;
  p.H = d.height;
  p.W = d.width;
  for (int o = 0; o < 3; ++o) p.out[o] = d.out[o];
  const int smem = 9 * p.ci * p.cout * 4;
  int rc_prep = direct_prepare();
  if (rc_prep != TDX_OK) return rc_prep;
  dim3 grid((d.height * d.width + 32 * kConvInGroups - 1) / (32 * kConvInGroups), d.n_img);
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute attr[1];
  fill_launch_config(&cfg, attr, grid, dim3(128), smem, stream);
  switch (p.ci) {
    case 6: TDX_CHECK_CUDA(cudaLaunchKernelEx(&cfg, conv_in_kernel<6>, p)); break;
    case 12: TDX_CHECK_CUDA(cudaLaunchKernelEx(&cfg, conv_in_kernel<12>, p)); break;
    default:
      set_error("conv_in: %d input channels (incl. ones) not instantiated (6 or 12)", p.ci);
      return TDX_E_UNSUPPORTED;
  }
  return TDX_OK;
}

// ------------------------------------------------------------------------------------------------ im2col of the input
struct Im2colParams {
  const void* src[2];
  int src_ch[2], src_dtype[2];
  const float* src_scale[2];
  uint4* out;
  int ci, kpad8, H, W;
};

// Thread = one pixel, all k (k = tap * CI + c); CI is a template constant, so the (tap, c) of every k is known at
// compile time and the gather is straight-line code: 9*(CI-1) coalesced source reads and k_pad/8 16-byte stores
// (a warp covers 32 consecutive pixels: 512 B per store instruction).
template <int CI>
__global__ void __launch_bounds__(128) im2col_in_kernel(const Im2colParams p) {
  pdl_launch_dependents();
  pdl_wait();
  const int pix = blockIdx.x * 128 + threadIdx.x;
  const int img = blockIdx.y;
  if (pix >= p.H * p.W) return;
  const int y = pix / p.W, x = pix - y * p.W;
  const size_t plane = (size_t)p.H * p.W;
  const int c0n = p.src_ch[0], c1n = p.src_ch[1];
  // per input channel: base pointer of this image's plane, element type, scale
  const uint8_t* cbase[CI - 1];
  int cdt[CI - 1];
  float csc[CI - 1];
  const float s0 = p.src_scale[0] ? __ldg(p.src_scale[0]) : 1.0f;
  const float s1 = p.src_scale[1] ? __ldg(p.src_scale[1]) : 1.0f;
#pragma unroll
  for (int c = 0; c < CI - 1; ++c) {
    const int which = c < c0n ? 0 : 1;
    const int cc = which ? c - c0n : c;
    const int cn = which ? c1n : c0n;
    cdt[c] = p.src_dtype[which];
    csc[c] = which ? s1 : s0;
    cbase[c] = reinterpret_cast<const uint8_t*>(p.src[which]) + ((size_t)img * cn + cc) * plane * (cdt[c] == 0 ? 4 : 2);
  }
  bool ok[9];
  int off[9];
#pragma unroll
  for (int tap = 0; tap < 9; ++tap) {
    const int yy = y + tap / 3 - 1, xx = x + tap % 3 - 1;
    ok[tap] = yy >= 0 && yy < p.H && xx >= 0 && xx < p.W;
    off[tap] = yy * p.W + xx;
  }
  constexpr int KPAD = ((9 * CI + 63) / 64) * 64;
  uint4* dst = p.out + (size_t)img * (KPAD / 8) * plane + pix;
#pragma unroll
  for (int kg = 0; kg < KPAD / 8; ++kg) {
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = kg * 8 + j;        // compile-time after unrolling
      const int tap = k / CI, c = k % CI;
      float val = 0.f;
      if (tap < 9) {
        if (c == CI - 1) {
          val = ok[tap] ? 1.0f : 0.f;
        } else if (ok[tap]) {
          val = (cdt[c] == 0 ? __ldg(reinterpret_cast<const float*>(cbase[c]) + off[tap])
                             : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(cbase[c])[off[tap]])) * csc[c];
        }
      }
      v[j] = val;
    }
    uint4 u;
    u.x = pack_bf16x2(v[0], v[1]);
    u.y = pack_bf16x2(v[2], v[3]);
    u.z = pack_bf16x2(v[4], v[5]);
    u.w = pack_bf16x2(v[6], v[7]);
    dst[(size_t)kg * plane] = u;
  }
}

int im2col_validate(const TdxIm2colDesc& d) {
  TDX_REQUIRE(d.src[0] && d.src_channels[0] > 0, "im2col: src[0] missing");
  TDX_REQUIRE(d.src_channels[1] == 0 || d.src[1], "im2col: src[1] missing");
  TDX_REQUIRE(d.out, "im2col: out is null");
  const int ci = d.src_channels[0] + d.src_channels[1] + 1;
  TDX_REQUIRE(ci == 6 || ci == 12, "im2col: %d input channels; instantiated for 5 (decoder / latent models) or 11 "
              "(coarse model)", ci - 1);
  TDX_REQUIRE(d.k_pad == ((9 * ci + 63) / 64) * 64, "im2col: k_pad=%d must be 9*%d rounded up to a multiple of 64",
              d.k_pad, ci);
  TDX_REQUIRE(d.n_img >= 1 && d.n_img <= 65535 && d.height >= 1 && d.width >= 1, "im2col: bad shape");
  return TDX_OK;
}

int im2col_launch(const TdxIm2colDesc& d, cudaStream_t stream) {
  Im2colParams p;
  for (int i = 0; i < 2; ++i) {
    p.src[i] = d.src[i];
    p.src_ch[i] = d.src_channels[i];
    p.src_dtype[i] = d.src_dtype[i];
    p.src_scale[i] = d.src_scale[i];
  }
  p.out = reinterpret_cast<uint4*>(d.out);
  p.ci = d.src_channels[0] + d.src_channels[1] + 1;
  p.kpad8 = d.k_pad / 8;
  p.H = d.height;
  p.W = d.width;
  dim3 grid((d.height * d.width + 127) / 128, d.n_img);
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute attr[1];
  fill_launch_config(&cfg, attr, grid, dim3(128), 0, stream);
  if (p.ci == 6) TDX_CHECK_CUDA(cudaLaunchKernelEx(&cfg, im2col_in_kernel<6>, p));
  else TDX_CHECK_CUDA(cudaLaunchKernelEx(&cfg, im2col_in_kernel<12>, p));
  return TDX_OK;
}

// ------------------------------------------------------------------------------------------------ last conv (+ scheduler)
struct ConvOutParams {
  const uint4* x;
  int C8, cout, H, W;
  const float* weight;
  float* model_out;
  const float* coef;
  float* sample;
  float* x0_prev;
  const float* guide_out;   // GUIDED: the guide model's F_g (fp32 NCHW); the guidance scale is coef[4]
};

// One DPM-Solver++(2M) update in the EDM closed form (scheduler/dpmsolver.py:419-561; SURVEY.md Appendix B).
__device__ __forceinline__ void sched_update(float x, float f, float x0p, float c_skip, float c_out, float r, float k,
                                             float& x_new, float& x0) {
  x0 = __fadd_rn(__fmul_rn(c_skip, x), __fmul_rn(c_out, f));
  float t = __fadd_rn(__fmul_rn(r, x), __fmul_rn(1.0f - r, x0));
  x_new = __fadd_rn(t, __fmul_rn(k, __fsub_rn(x0, x0p)));
}

// Block = 128 threads = 32 pixels x 4 sub-threads; sub-thread s accumulates channel groups s, s+4, ... so four times as
// many 16-byte loads are in flight; the partial sums are combined with two warp shuffles.  COUT = 1 (decoder) or 8.
// GUIDED: two-model autoguidance before the update, F = F_g + s*(F_m - F_g) with F_m = conv3x3(x), separately rounded
// in the reference's order (sample_diffusion_base.py:110, sample_diffusion_decoder.py:117); model_out receives F.
template <int COUT, bool GUIDED>
__global__ void __launch_bounds__(128) conv_out_kernel(const ConvOutParams p) {
  extern __shared__ float ws[];  // [tap][c][COUT]
  const int C = p.C8 * 8;
  for (int i = threadIdx.x; i < (9 * C * COUT) / 4; i += blockDim.x)
    reinterpret_cast<float4*>(ws)[i] = __ldg(reinterpret_cast<const float4*>(p.weight) + i);
  pdl_launch_dependents();
  pdl_wait();
  __syncthreads();
  const int img = blockIdx.y;
  const int lane = threadIdx.x & 31, wq = threadIdx.x >> 5;
  const int sub = lane >> 3;                                // 0..3
  const size_t plane = (size_t)p.H * p.W;
  for (int grp = 0; grp < kConvOutGroups; ++grp) {
    const int pix = (blockIdx.x * kConvOutGroups + grp) * 32 + wq * 8 + (lane & 7);
    const bool inb = pix < p.H * p.W;
    const int y = inb ? pix / p.W : 0, x = inb ? pix % p.W : 0;
    float acc[COUT];
#pragma unroll
    for (int j = 0; j < COUT; ++j) acc[j] = 0.f;
    // the guide's output is issued with the activation loads, not after the reduction
    float fg[GUIDED ? COUT : 1];
    if (GUIDED) {
#pragma unroll
      for (int oc = 0; oc < COUT; ++oc)
        fg[oc] = (inb && sub == 0 && oc < p.cout) ? __ldg(p.guide_out + ((size_t)img * p.cout + oc) * plane + pix) : 0.f;
    }
    if (COUT == 1 && p.C8 == 8) {
      // the decoder's 64 -> 1 case: all 18 loads of a thread are issued before the first is used (the generic loop
      // below walks taps and groups with data-dependent control flow: one L2 latency after the other).  Out-of-image
      // taps contribute exact zeros, so the sum is bit-identical to the generic path.
      uint4 u[9][2];
      const uint4* base = p.x + (size_t)img * p.C8 * plane;
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) {
        const int yy = y + tap / 3 - 1, xx = x + tap % 3 - 1;
        const bool ok = inb && yy >= 0 && yy < p.H && xx >= 0 && xx < p.W;
        const uint4* src = base + (ok ? (size_t)yy * p.W + xx : 0);
        u[tap][0] = ok ? __ldg(src + (size_t)sub * plane) : make_uint4(0, 0, 0, 0);
        u[tap][1] = ok ? __ldg(src + (size_t)(sub + 4) * plane) : make_uint4(0, 0, 0, 0);
      }
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          float a[8];
          unpack_bf16x2(u[tap][j].x, a[0], a[1]); unpack_bf16x2(u[tap][j].y, a[2], a[3]);
          unpack_bf16x2(u[tap][j].z, a[4], a[5]); unpack_bf16x2(u[tap][j].w, a[6], a[7]);
          const float* w = ws + (tap * C + (sub + 4 * j) * 8);
          const float4 wa = *reinterpret_cast<const float4*>(w), wb = *reinterpret_cast<const float4*>(w + 4);
          const float t0 = fmaf(wa.x, a[0], wa.y * a[1]), t1 = fmaf(wa.z, a[2], wa.w * a[3]);
          const float t2 = fmaf(wb.x, a[4], wb.y * a[5]), t3 = fmaf(wb.z, a[6], wb.w * a[7]);
          acc[0] += (t0 + t1) + (t2 + t3);
        }
      }
    } else
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
      const int yy = y + tap / 3 - 1, xx = x + tap % 3 - 1;
      if (!inb || yy < 0 || yy >= p.H || xx < 0 || xx >= p.W) continue;
      const uint4* src = p.x + (size_t)img * p.C8 * plane + (size_t)yy * p.W + xx;
      for (int g = sub; g < p.C8; g += 4) {
        const uint4 u = __ldg(src + (size_t)g * plane);
        float a[8];
        unpack_bf16x2(u.x, a[0], a[1]); unpack_bf16x2(u.y, a[2], a[3]);
        unpack_bf16x2(u.z, a[4], a[5]); unpack_bf16x2(u.w, a[6], a[7]);
        const float* w = ws + (tap * C + g * 8) * COUT;
        if (COUT == 1) {
          const float4 wa = *reinterpret_cast<const float4*>(w), wb = *reinterpret_cast<const float4*>(w + 4);
          // (a tree per load instead of one 144-deep FMA chain through acc[0])
          const float t0 = fmaf(wa.x, a[0], wa.y * a[1]), t1 = fmaf(wa.z, a[2], wa.w * a[3]);
          const float t2 = fmaf(wb.x, a[4], wb.y * a[5]), t3 = fmaf(wb.z, a[6], wb.w * a[7]);
          acc[0] += (t0 + t1) + (t2 + t3);
        } else {
#pragma unroll
          for (int e = 0; e < 8; ++e) {
#pragma unroll
            for (int j = 0; j < COUT; ++j) acc[j] = fmaf(w[e * COUT + j], a[e], acc[j]);
          }
        }
      }
    }
#pragma unroll
    for (int j = 0; j < COUT; ++j) {
      acc[j] += __shfl_xor_sync(0xffffffff, acc[j], 8);
      acc[j] += __shfl_xor_sync(0xffffffff, acc[j], 16);
    }
    if (!inb || sub != 0) continue;
    float cs = 0.f, co = 0.f, r = 0.f, k = 0.f, gs = 1.f;
    if (p.coef) { cs = __ldg(p.coef); co = __ldg(p.coef + 1); r = __ldg(p.coef + 2); k = __ldg(p.coef + 3); }
    if (GUIDED) gs = __ldg(p.coef + 4);
#pragma unroll
    for (int oc = 0; oc < COUT; ++oc) {
      if (oc >= p.cout) break;
      const size_t idx = ((size_t)img * p.cout + oc) * plane + pix;
      if (GUIDED) acc[oc] = __fadd_rn(fg[oc], __fmul_rn(gs, __fsub_rn(acc[oc], fg[oc])));
      if (p.model_out) p.model_out[idx] = acc[oc];
      if (p.coef) {
        float xn, x0;
        sched_update(p.sample[idx], acc[oc], p.x0_prev[idx], cs, co, r, k, xn, x0);
        p.sample[idx] = xn;
        p.x0_prev[idx] = x0;
      }
    }
  }
}

// Opt in to > 48 KB dynamic shared memory once (must not happen inside a stream capture).
int direct_prepare() {
  static bool seen[16] = {false};
  if (first_use_on_device(seen)) {
    TDX_CHECK_CUDA(cudaFuncSetAttribute(conv_in_kernel<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    TDX_CHECK_CUDA(cudaFuncSetAttribute(conv_in_kernel<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    TDX_CHECK_CUDA(cudaFuncSetAttribute(conv_out_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    TDX_CHECK_CUDA(cudaFuncSetAttribute(conv_out_kernel<8, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    TDX_CHECK_CUDA(cudaFuncSetAttribute(conv_out_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    TDX_CHECK_CUDA(cudaFuncSetAttribute(conv_out_kernel<8, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  }
  return TDX_OK;
}

int conv_out_validate(const TdxConvOutDesc& d) {
  TDX_REQUIRE(d.x && d.weight, "conv_out: null x / weight");
  TDX_REQUIRE(d.c_in > 0 && d.c_in % 8 == 0, "conv_out: c_in=%d not a multiple of 8", d.c_in);
  TDX_REQUIRE(d.c_out >= 1 && d.c_out <= 8, "conv_out: c_out=%d not in 1..8", d.c_out);
  TDX_REQUIRE(9 * d.c_in * 8 * 4 <= 200 * 1024, "conv_out: c_in=%d too large", d.c_in);
  TDX_REQUIRE(d.model_out || d.sched_coef, "conv_out: nothing to write");
  if (d.sched_coef) TDX_REQUIRE(d.sample && d.x0_prev, "conv_out: scheduler fusion needs sample and x0_prev");
  return TDX_OK;
}

int conv_out_guided_validate(const TdxConvOutGuidedDesc& d) {
  int rc = conv_out_validate(d.base);
  if (rc != TDX_OK) return rc;
  TDX_REQUIRE(d.guide_out, "conv_out_guided: null guide_out");
  TDX_REQUIRE(d.base.sched_coef, "conv_out_guided: the guidance scale is read from sched_coef[4]: sched_coef is required");
  return TDX_OK;
}

// guide_out == NULL: the plain kernel (bit-identical to a TdxConvOutDesc launch).
int conv_out_launch_impl(const TdxConvOutDesc& d, const float* guide_out, cudaStream_t stream) {
  ConvOutParams p;
  p.x = reinterpret_cast<const uint4*>(d.x);
  p.C8 = d.c_in / 8;
  p.cout = d.c_out;
  p.H = d.height;
  p.W = d.width;
  p.weight = d.weight;
  p.model_out = d.model_out;
  p.coef = d.sched_coef;
  p.sample = d.sample;
  p.x0_prev = d.x0_prev;
  p.guide_out = guide_out;
  const int wout = d.c_out == 1 ? 1 : 8;
  const int smem = 9 * d.c_in * wout * 4;
  int rc_prep = direct_prepare();
  if (rc_prep != TDX_OK) return rc_prep;
  dim3 grid((d.height * d.width + 32 * kConvOutGroups - 1) / (32 * kConvOutGroups), d.n_img);
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute attr[1];
  fill_launch_config(&cfg, attr, grid, dim3(128), smem, stream);
  if (guide_out) {
    if (wout == 1) TDX_CHECK_CUDA(cudaLaunchKernelEx(&cfg, conv_out_kernel<1, true>, p));
    else TDX_CHECK_CUDA(cudaLaunchKernelEx(&cfg, conv_out_kernel<8, true>, p));
  } else {
    if (wout == 1) TDX_CHECK_CUDA(cudaLaunchKernelEx(&cfg, conv_out_kernel<1, false>, p));
    else TDX_CHECK_CUDA(cudaLaunchKernelEx(&cfg, conv_out_kernel<8, false>, p));
  }
  return TDX_OK;
}

int conv_out_launch(const TdxConvOutDesc& d, cudaStream_t stream) { return conv_out_launch_impl(d, nullptr, stream); }

int conv_out_guided_launch(const TdxConvOutGuidedDesc& d, cudaStream_t stream) {
  return conv_out_launch_impl(d.base, d.guide_out, stream);
}

// ------------------------------------------------------------------------------------------------ embedding vectors
constexpr int kMaxEmbedBlocks = 64;
struct EmbedParams {
  const float* labels;
  const float* emb_in;
  const float* noise_weight;
  const float* noise_freqs;
  int noise_dims, E;
  TdxEmbedBlock blocks[kMaxEmbedBlocks];
};

// One block per (U-Net block, image).  Weights are stored TRANSPOSED ([in][out]) so thread n's loads are coalesced and
// independent; every block recomputes the 256-wide embedding (64 x 256 MACs) instead of paying a second launch.
__global__ void __launch_bounds__(256) embed_kernel(const __grid_constant__ EmbedParams p) {
  __shared__ float pe[256];
  __shared__ float emb[1024];
  __shared__ float red[8];
  const int b = blockIdx.x, img = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_launch_dependents();
  pdl_wait();  // labels / cvec buffers are shared with earlier launches
  if (p.emb_in) {
    for (int j = threadIdx.x; j < p.E; j += blockDim.x) emb[j] = p.emb_in[(size_t)img * p.E + j];
  } else {
    // MPPositionalEmbedding (mp_layers.py:88-107), fp32
    const int half = p.noise_dims >> 1;
    const float t = p.labels[img];
    for (int i = threadIdx.x; i < half; i += blockDim.x) {
      const float yv = t * p.noise_freqs[i];
      pe[i] = sinf(yv) * 1.41421356237309515f;
      pe[half + i] = cosf(yv) * 1.41421356237309515f;
    }
    __syncthreads();
    for (int j = threadIdx.x; j < p.E; j += blockDim.x) {
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll 4
      for (int i = 0; i < p.noise_dims; i += 4) {
        s0 = fmaf(__ldg(p.noise_weight + (size_t)(i + 0) * p.E + j), pe[i + 0], s0);
        s1 = fmaf(__ldg(p.noise_weight + (size_t)(i + 1) * p.E + j), pe[i + 1], s1);
        s2 = fmaf(__ldg(p.noise_weight + (size_t)(i + 2) * p.E + j), pe[i + 2], s2);
        s3 = fmaf(__ldg(p.noise_weight + (size_t)(i + 3) * p.E + j), pe[i + 3], s3);
      }
      emb[j] = mp_silu_precise((s0 + s1) + (s2 + s3));  // mp_sum of a single embed with weight [1] is the identity
    }
  }
  __syncthreads();
  // c[n] = sum_j W^T[j][n] * emb[j] + 1: the 256 threads cover (n, part-of-j) so all of them stream weights
  const TdxEmbedBlock& blk = p.blocks[b];
  __shared__ float part[4][256];
  __shared__ float cfull[1024];
  const int parts = blk.c_out <= 64 ? 4 : (blk.c_out <= 128 ? 2 : 1);
  const int per = 256 / parts;
  float sq = 0.f;
  for (int n0 = 0; n0 < blk.c_out; n0 += per) {
    const int n = n0 + threadIdx.x % per, part_id = threadIdx.x / per;
    const int jlen = p.E / parts, j0 = part_id * jlen;
    float acc = 0.f;
    if (n < blk.c_out) {
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll 8
      for (int j = j0; j < j0 + jlen; j += 4) {
        s0 = fmaf(__ldg(blk.weight + (size_t)(j + 0) * blk.c_out + n), emb[j + 0], s0);
        s1 = fmaf(__ldg(blk.weight + (size_t)(j + 1) * blk.c_out + n), emb[j + 1], s1);
        s2 = fmaf(__ldg(blk.weight + (size_t)(j + 2) * blk.c_out + n), emb[j + 2], s2);
        s3 = fmaf(__ldg(blk.weight + (size_t)(j + 3) * blk.c_out + n), emb[j + 3], s3);
      }
      acc = (s0 + s1) + (s2 + s3);
    }
    part[part_id][threadIdx.x % per] = acc;
    __syncthreads();
    const int nn = n0 + threadIdx.x;
    if (threadIdx.x < per && nn < blk.c_out) {
      float c = 1.0f;
      for (int q = 0; q < parts; ++q) c += part[q][threadIdx.x];
      cfull[nn] = c;
      sq += c * c;
    }
    __syncthreads();
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffff, sq, o);
  if (lane == 0) red[warp] = sq;
  __syncthreads();
  float tot = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) tot += red[w];
  const float inv = rsqrtf(tot / (float)blk.c_out + 1e-8f);
  for (int nn = threadIdx.x; nn < blk.c_out; nn += blockDim.x) blk.cvec[(size_t)img * blk.c_out + nn] = cfull[nn] * inv;
}

int embed_validate(const TdxEmbedDesc& d) {
  TDX_REQUIRE(d.n_blocks >= 1 && d.n_blocks <= kMaxEmbedBlocks, "embed: n_blocks=%d not in 1..%d", d.n_blocks,
              kMaxEmbedBlocks);
  TDX_REQUIRE(d.blocks, "embed: blocks is null");
  TDX_REQUIRE(d.emb_channels >= 4 && d.emb_channels <= 1024 && d.emb_channels % 4 == 0, "embed: emb_channels=%d",
              d.emb_channels);
  TDX_REQUIRE(d.emb_channels % 16 == 0, "embed: emb_channels must be a multiple of 16");
  TDX_REQUIRE(d.n_img >= 1, "embed: n_img");
  if (!d.emb_in) {
    TDX_REQUIRE(d.noise_labels && d.noise_weight && d.noise_freqs, "embed: noise path needs labels, weight, freqs");
    TDX_REQUIRE(d.noise_dims >= 4 && d.noise_dims <= 256 && d.noise_dims % 4 == 0, "embed: noise_dims=%d",
                d.noise_dims);
  }
  for (int b = 0; b < d.n_blocks; ++b)
    TDX_REQUIRE(d.blocks[b].weight && d.blocks[b].cvec && d.blocks[b].c_out >= 1 && d.blocks[b].c_out <= 1024,
                "embed: block %d invalid", b);
  return TDX_OK;
}

int embed_launch(const TdxEmbedDesc& d, cudaStream_t stream) {
  EmbedParams p;
  memset(&p, 0, sizeof(p));
  p.labels = d.noise_labels;
  p.emb_in = d.emb_in;
  p.noise_weight = d.noise_weight;
  p.noise_freqs = d.noise_freqs;
  p.noise_dims = d.noise_dims;
  p.E = d.emb_channels;
  for (int b = 0; b < d.n_blocks; ++b) p.blocks[b] = d.blocks[b];
  dim3 grid(d.n_blocks, d.n_img);
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute attr[1];
  fill_launch_config(&cfg, attr, grid, dim3(256), 0, stream);
  TDX_CHECK_CUDA(cudaLaunchKernelEx(&cfg, embed_kernel, p));
  return TDX_OK;
}

// ------------------------------------------------------------------------------------------------ elementwise fp32
__global__ void sched_step_kernel(float* sample, const float* f, float* x0_prev, int64_t n, float cs, float co, float r,
                                  float k) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    float xn, x0;
    sched_update(sample[i], f[i], x0_prev[i], cs, co, r, k, xn, x0);
    sample[i] = xn;
    x0_prev[i] = x0;
  }
}

// ---- overlap blend / canvas kernels: HBM-bound, one float4 (four pixels of a row) per thread and channel.  Every
// element still goes through separately rounded __fmul_rn / __fadd_rn / __fdiv_rn in the reference's order, so the
// vector path is bit-identical to the scalar one (taken when pointers, widths or offsets are not multiples of 4).
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, const float4& v) { *reinterpret_cast<float4*>(p) = v; }

template <bool VEC>
__global__ void blend_accumulate_kernel(float* cval, float* cw, int channels, int CH, int CW, const float* tile,
                                        const float* window, int th, int tw, int y0, int x0) {
  constexpr int V = VEC ? 4 : 1;
  const int x = (blockIdx.x * blockDim.x + threadIdx.x) * V;
  const int y = blockIdx.y;
  if (x >= tw) return;
  const int Y = y0 + y, X = x0 + x;
  if (Y < 0 || Y >= CH) return;
  if constexpr (VEC) {
    if (X < 0 || X + 3 >= CW) {           // row segment straddling the canvas edge: element by element
      for (int i = 0; i < 4; ++i) {
        if (X + i < 0 || X + i >= CW) continue;
        const float w = window[(size_t)y * tw + x + i];
        const size_t ci = (size_t)Y * CW + X + i;
        for (int c = 0; c < channels; ++c)
          cval[(size_t)c * CH * CW + ci] = __fadd_rn(cval[(size_t)c * CH * CW + ci],
                                                     __fmul_rn(tile[((size_t)c * th + y) * tw + x + i], w));
        cw[ci] = __fadd_rn(cw[ci], w);
      }
      return;
    }
    const float4 w = ld4(window + (size_t)y * tw + x);
    const size_t cidx = (size_t)Y * CW + X;
    for (int c = 0; c < channels; ++c) {
      const float4 t = ld4(tile + ((size_t)c * th + y) * tw + x);
      float* d = cval + (size_t)c * CH * CW + cidx;
      float4 v = ld4(d);
      v.x = __fadd_rn(v.x, __fmul_rn(t.x, w.x));
      v.y = __fadd_rn(v.y, __fmul_rn(t.y, w.y));
      v.z = __fadd_rn(v.z, __fmul_rn(t.z, w.z));
      v.w = __fadd_rn(v.w, __fmul_rn(t.w, w.w));
      st4(d, v);
    }
    float4 s = ld4(cw + cidx);
    s.x = __fadd_rn(s.x, w.x); s.y = __fadd_rn(s.y, w.y); s.z = __fadd_rn(s.z, w.z); s.w = __fadd_rn(s.w, w.w);
    st4(cw + cidx, s);
  } else {
    if (X < 0 || X >= CW) return;
    const float w = window[(size_t)y * tw + x];
    const size_t cidx = (size_t)Y * CW + X;
    for (int c = 0; c < channels; ++c) {
      const float v = __fmul_rn(tile[((size_t)c * th + y) * tw + x], w);
      cval[(size_t)c * CH * CW + cidx] = __fadd_rn(cval[(size_t)c * CH * CW + cidx], v);
    }
    cw[cidx] = __fadd_rn(cw[cidx], w);
  }
}

template <bool VEC>
__global__ void canvas_add_kernel(float* dst, int channels, int DH, int DW, const float* tile, int th, int tw, int y0,
                                  int x0) {
  constexpr int V = VEC ? 4 : 1;
  const int x = (blockIdx.x * blockDim.x + threadIdx.x) * V;
  const int y = blockIdx.y;
  if (x >= tw) return;
  const int Y = y0 + y, X = x0 + x;
  if (Y < 0 || Y >= DH) return;
  if constexpr (VEC) {
    if (X >= 0 && X + 3 < DW) {
      for (int c = 0; c < channels; ++c) {
        float* d = dst + ((size_t)c * DH + Y) * DW + X;
        const float4 t = ld4(tile + ((size_t)c * th + y) * tw + x);
        float4 v = ld4(d);
        v.x = __fadd_rn(v.x, t.x); v.y = __fadd_rn(v.y, t.y); v.z = __fadd_rn(v.z, t.z); v.w = __fadd_rn(v.w, t.w);
        st4(d, v);
      }
      return;
    }
  }
  for (int i = 0; i < V; ++i) {
    if (X + i < 0 || X + i >= DW) continue;
    for (int c = 0; c < channels; ++c) {
      const size_t di = ((size_t)c * DH + Y) * DW + X + i;
      dst[di] = __fadd_rn(dst[di], tile[((size_t)c * th + y) * tw + x + i]);
    }
  }
}

template <bool VEC>
__global__ void blend_normalize_kernel(float* out, const float* cval, const float* cw, int channels, int64_t plane,
                                       float divisor) {
  constexpr int V = VEC ? 4 : 1;
  int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * V;
  const int64_t n = plane * channels;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x * V;
  for (; i < n; i += stride) {
    if constexpr (VEC) {
      const float4 a = ld4(cval + i), w = ld4(cw + i % plane);       // plane % 4 == 0: the four share one channel
      float4 q;
      q.x = __fdiv_rn(a.x, w.x); q.y = __fdiv_rn(a.y, w.y); q.z = __fdiv_rn(a.z, w.z); q.w = __fdiv_rn(a.w, w.w);
      if (divisor != 1.0f) {
        q.x = __fdiv_rn(q.x, divisor); q.y = __fdiv_rn(q.y, divisor); q.z = __fdiv_rn(q.z, divisor);
        q.w = __fdiv_rn(q.w, divisor);
      }
      st4(out + i, q);
    } else {
      const float q = __fdiv_rn(cval[i], cw[i % plane]);
      out[i] = divisor == 1.0f ? q : __fdiv_rn(q, divisor);
    }
  }
}

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace tdx

using namespace tdx;

extern "C" int tdx_conv_in_run(const TdxConvInDesc* d, void* stream) {
  if (!d) { set_error("conv_in: null descriptor"); return TDX_E_INVALID; }
  int rc = conv_in_validate(*d);
  if (rc != TDX_OK) return rc;
  return conv_in_launch(*d, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int tdx_im2col_run(const TdxIm2colDesc* d, void* stream) {
  if (!d) { set_error("im2col: null descriptor"); return TDX_E_INVALID; }
  int rc = im2col_validate(*d);
  if (rc != TDX_OK) return rc;
  return im2col_launch(*d, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int tdx_conv_out_run(const TdxConvOutDesc* d, void* stream) {
  if (!d) { set_error("conv_out: null descriptor"); return TDX_E_INVALID; }
  int rc = conv_out_validate(*d);
  if (rc != TDX_OK) return rc;
  return conv_out_launch(*d, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int tdx_conv_out_guided_run(const TdxConvOutGuidedDesc* d, void* stream) {
  if (!d) { set_error("conv_out_guided: null descriptor"); return TDX_E_INVALID; }
  int rc = conv_out_guided_validate(*d);
  if (rc != TDX_OK) return rc;
  return conv_out_guided_launch(*d, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int tdx_embed_run(const TdxEmbedDesc* d, void* stream) {
  if (!d) { set_error("embed: null descriptor"); return TDX_E_INVALID; }
  int rc = embed_validate(*d);
  if (rc != TDX_OK) return rc;
  return embed_launch(*d, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int tdx_sched_step(float* sample, const float* model_out, float* x0_prev, int64_t numel, float c_skip,
                              float c_out, float r, float k, void* stream) {
  TDX_REQUIRE(sample && model_out && x0_prev && numel > 0, "sched_step: bad arguments");
  int blocks = (int)((numel + 255) / 256);
  if (blocks > sm_count() * 8) blocks = sm_count() * 8;
  sched_step_kernel<<<blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(sample, model_out, x0_prev, numel,
                                                                               c_skip, c_out, r, k);
  TDX_CHECK_CUDA(cudaGetLastError());
  return TDX_OK;
}

extern "C" int tdx_blend_accumulate(float* canvas_val, float* canvas_w, int32_t channels, int32_t canvas_h,
                                    int32_t canvas_w_px, const float* tile, const float* window, int32_t tile_h,
                                    int32_t tile_w, int32_t y0, int32_t x0, void* stream) {
  TDX_REQUIRE(canvas_val && canvas_w && tile && window, "blend_accumulate: null pointer");
  TDX_REQUIRE(channels >= 1 && tile_h >= 1 && tile_w >= 1 && canvas_h >= 1 && canvas_w_px >= 1,
              "blend_accumulate: bad shape");
  dim3 grid((tile_w + 127) / 128, tile_h);
  const bool vec = (tile_w % 4 == 0) && (canvas_w_px % 4 == 0) && (x0 % 4 == 0) && aligned16(canvas_val) &&
                   aligned16(canvas_w) && aligned16(tile) && aligned16(window) &&
                   ((size_t)canvas_h * canvas_w_px) % 4 == 0 && ((size_t)tile_h * tile_w) % 4 == 0;
  if (vec) {
    grid.x = (tile_w / 4 + 127) / 128;
    blend_accumulate_kernel<true><<<grid, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        canvas_val, canvas_w, channels, canvas_h, canvas_w_px, tile, window, tile_h, tile_w, y0, x0);
  } else {
    blend_accumulate_kernel<false><<<grid, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        canvas_val, canvas_w, channels, canvas_h, canvas_w_px, tile, window, tile_h, tile_w, y0, x0);
  }
  TDX_CHECK_CUDA(cudaGetLastError());
  return TDX_OK;
}

extern "C" int tdx_canvas_add(float* dst, int32_t channels, int32_t dst_h, int32_t dst_w, const float* tile,
                              int32_t tile_h, int32_t tile_w, int32_t y0, int32_t x0, void* stream) {
  TDX_REQUIRE(dst && tile && channels >= 1 && dst_h >= 1 && dst_w >= 1 && tile_h >= 1 && tile_w >= 1,
              "canvas_add: bad arguments");
  dim3 grid((tile_w + 127) / 128, tile_h);
  const bool vec = (tile_w % 4 == 0) && (dst_w % 4 == 0) && (x0 % 4 == 0) && aligned16(dst) && aligned16(tile) &&
                   ((size_t)dst_h * dst_w) % 4 == 0 && ((size_t)tile_h * tile_w) % 4 == 0;
  if (vec) {
    grid.x = (tile_w / 4 + 127) / 128;
    canvas_add_kernel<true><<<grid, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(dst, channels, dst_h, dst_w, tile,
                                                                                     tile_h, tile_w, y0, x0);
  } else {
    canvas_add_kernel<false><<<grid, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(dst, channels, dst_h, dst_w, tile,
                                                                                      tile_h, tile_w, y0, x0);
  }
  TDX_CHECK_CUDA(cudaGetLastError());
  return TDX_OK;
}

extern "C" int tdx_blend_normalize(float* out, const float* canvas_val, const float* canvas_w, int32_t channels,
                                   int64_t plane, float divisor, void* stream) {
  TDX_REQUIRE(out && canvas_val && canvas_w && channels >= 1 && plane >= 1, "blend_normalize: bad arguments");
  int64_t n = plane * channels;
  const bool vec = plane % 4 == 0 && aligned16(out) && aligned16(canvas_val) && aligned16(canvas_w);
  int blocks = (int)((n / (vec ? 4 : 1) + 255) / 256);
  if (blocks > sm_count() * 8) blocks = sm_count() * 8;
  if (blocks < 1) blocks = 1;
  if (vec)
    blend_normalize_kernel<true><<<blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(out, canvas_val, canvas_w,
                                                                                            channels, plane, divisor);
  else
    blend_normalize_kernel<false><<<blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(out, canvas_val, canvas_w,
                                                                                             channels, plane, divisor);
  TDX_CHECK_CUDA(cudaGetLastError());
  return TDX_OK;
}
