// Program = recorded launch list (conv_in / im2col / igemm / conv_out / embed / attn) with pre-built TMA descriptors, replayed through
// one CUDA graph.  Host-side only; all kernels live in tdx_igemm.cu / tdx_direct.cu.
#include <vector>

#include "tdx_common.h"

namespace tdx {
int igemm_validate(const TdxIgemmDesc& d);
int igemm_prepare();
int igemm_launch(const TdxIgemmDesc& d, const CUtensorMap* tms, cudaStream_t stream);
int conv_in_validate(const TdxConvInDesc& d);
int conv_in_launch(const TdxConvInDesc& d, cudaStream_t stream);
int im2col_validate(const TdxIm2colDesc& d);
int im2col_launch(const TdxIm2colDesc& d, cudaStream_t stream);
int conv_out_validate(const TdxConvOutDesc& d);
int conv_out_launch(const TdxConvOutDesc& d, cudaStream_t stream);
int conv_out_guided_validate(const TdxConvOutGuidedDesc& d);
int conv_out_launch_impl(const TdxConvOutDesc& d, const float* guide_out, cudaStream_t stream);
int embed_validate(const TdxEmbedDesc& d);
int direct_prepare();
int attn_validate(const TdxAttnDesc& d);
int attn_prepare();
int attn_launch(const TdxAttnDesc& d, cudaStream_t stream);
int embed_launch(const TdxEmbedDesc& d, cudaStream_t stream);

enum OpType { OP_CONV_IN, OP_IGEMM, OP_CONV_OUT, OP_EMBED, OP_ATTN, OP_IM2COL };

struct Op {
  OpType type;
  TdxIgemmDesc ig;
  CUtensorMap tms[3];
  TdxConvInDesc ci;
  TdxConvOutDesc co;
  const float* guide_out = nullptr;   // OP_CONV_OUT with two-model guidance (tdx_program_add_conv_out_guided)
  TdxEmbedDesc em;
  TdxAttnDesc at;
  TdxIm2colDesc im;
  std::vector<TdxEmbedBlock> blocks;
};
}  // namespace tdx

struct TdxProgram {
  std::vector<tdx::Op> ops;
  cudaGraphExec_t exec = nullptr;
  cudaGraph_t graph = nullptr;
};

using namespace tdx;

static int launch_all(TdxProgram* p, cudaStream_t stream) {
  for (auto& op : p->ops) {
    int rc = TDX_OK;
    switch (op.type) {
      case OP_CONV_IN: rc = conv_in_launch(op.ci, stream); break;
      case OP_IGEMM: rc = igemm_launch(op.ig, op.tms, stream); break;
      case OP_CONV_OUT: rc = conv_out_launch_impl(op.co, op.guide_out, stream); break;
      case OP_EMBED:
        op.em.blocks = op.blocks.data();
        rc = embed_launch(op.em, stream);
        break;
      case OP_ATTN: rc = attn_launch(op.at, stream); break;
      case OP_IM2COL: rc = im2col_launch(op.im, stream); break;
    }
    if (rc != TDX_OK) return rc;
  }
  return TDX_OK;
}

extern "C" int tdx_program_create(TdxProgram** out) {
  TDX_REQUIRE(out, "program_create: null out");
  *out = new TdxProgram();
  return TDX_OK;
}

static int invalidate_graph(TdxProgram* p) {
  if (p->exec) { cudaGraphExecDestroy(p->exec); p->exec = nullptr; }
  if (p->graph) { cudaGraphDestroy(p->graph); p->graph = nullptr; }
  return TDX_OK;
}

extern "C" int tdx_program_add_conv_in(TdxProgram* p, const TdxConvInDesc* d) {
  TDX_REQUIRE(p && d, "program_add_conv_in: null argument");
  int rc = conv_in_validate(*d);
  if (rc != TDX_OK) return rc;
  rc = direct_prepare();
  if (rc != TDX_OK) return rc;
  Op op;
  op.type = OP_CONV_IN;
  op.ci = *d;
  p->ops.push_back(op);
  return invalidate_graph(p);
}

extern "C" int tdx_program_add_im2col(TdxProgram* p, const TdxIm2colDesc* d) {
  TDX_REQUIRE(p && d, "program_add_im2col: null argument");
  int rc = im2col_validate(*d);
  if (rc != TDX_OK) return rc;
  Op op;
  op.type = OP_IM2COL;
  op.im = *d;
  p->ops.push_back(op);
  return invalidate_graph(p);
}

extern "C" int tdx_program_add_igemm(TdxProgram* p, const TdxIgemmDesc* d) {
  TDX_REQUIRE(p && d, "program_add_igemm: null argument");
  int rc = igemm_validate(*d);
  if (rc != TDX_OK) return rc;
  rc = igemm_prepare();
  if (rc != TDX_OK) return rc;
  Op op;
  op.type = OP_IGEMM;
  op.ig = *d;
  for (int s = 0; s < d->n_seg; ++s) {
    rc = make_act_tensor_map(&op.tms[s], d->a_ptr[s], d->n_img, d->a_channels[s], d->height, d->width);
    if (rc != TDX_OK) return rc;
  }
  p->ops.push_back(op);
  return invalidate_graph(p);
}

extern "C" int tdx_program_add_conv_out(TdxProgram* p, const TdxConvOutDesc* d) {
  TDX_REQUIRE(p && d, "program_add_conv_out: null argument");
  int rc = conv_out_validate(*d);
  if (rc != TDX_OK) return rc;
  rc = direct_prepare();
  if (rc != TDX_OK) return rc;
  Op op;
  op.type = OP_CONV_OUT;
  op.co = *d;
  p->ops.push_back(op);
  return invalidate_graph(p);
}

extern "C" int tdx_program_add_conv_out_guided(TdxProgram* p, const TdxConvOutGuidedDesc* d) {
  TDX_REQUIRE(p && d, "program_add_conv_out_guided: null argument");
  int rc = conv_out_guided_validate(*d);
  if (rc != TDX_OK) return rc;
  rc = direct_prepare();
  if (rc != TDX_OK) return rc;
  Op op;
  op.type = OP_CONV_OUT;
  op.co = d->base;
  op.guide_out = d->guide_out;
  p->ops.push_back(op);
  return invalidate_graph(p);
}

extern "C" int tdx_program_add_embed(TdxProgram* p, const TdxEmbedDesc* d) {
  TDX_REQUIRE(p && d, "program_add_embed: null argument");
  int rc = embed_validate(*d);
  if (rc != TDX_OK) return rc;
  Op op;
  op.type = OP_EMBED;
  op.em = *d;
  op.blocks.assign(d->blocks, d->blocks + d->n_blocks);
  op.em.blocks = nullptr;
  p->ops.push_back(op);
  return invalidate_graph(p);
}

extern "C" int tdx_program_add_attn(TdxProgram* p, const TdxAttnDesc* d) {
  TDX_REQUIRE(p && d, "program_add_attn: null argument");
  int rc = attn_validate(*d);
  if (rc != TDX_OK) return rc;
  rc = attn_prepare();
  if (rc != TDX_OK) return rc;
  Op op;
  op.type = OP_ATTN;
  op.at = *d;
  p->ops.push_back(op);
  return invalidate_graph(p);
}

extern "C" int tdx_program_num_launches(const TdxProgram* p) { return p ? (int)p->ops.size() : -1; }

static int ensure_graph(TdxProgram* p) {
  if (p->exec) return TDX_OK;
  // Capture on a private stream: the caller's stream may be the legacy default stream, which cannot be captured.
  cudaStream_t cap = nullptr;
  TDX_CHECK_CUDA(cudaStreamCreateWithFlags(&cap, cudaStreamNonBlocking));
  cudaError_t e = cudaStreamBeginCapture(cap, cudaStreamCaptureModeThreadLocal);
  if (e != cudaSuccess) {
    cudaStreamDestroy(cap);
    set_error("program: cudaStreamBeginCapture failed: %s", cudaGetErrorString(e));
    return TDX_E_CUDA;
  }
  int rc = launch_all(p, cap);
  cudaGraph_t g = nullptr;
  e = cudaStreamEndCapture(cap, &g);
  cudaStreamDestroy(cap);
  if (rc != TDX_OK) {
    if (g) cudaGraphDestroy(g);
    return rc;
  }
  if (e != cudaSuccess) {
    set_error("program: stream capture failed: %s", cudaGetErrorString(e));
    return TDX_E_CUDA;
  }
  p->graph = g;
  TDX_CHECK_CUDA(cudaGraphInstantiate(&p->exec, g, 0));
  return TDX_OK;
}

extern "C" int tdx_program_instantiate(TdxProgram* p, void* stream_) {
  TDX_REQUIRE(p, "program_instantiate: null program");
  int rc = ensure_graph(p);
  if (rc != TDX_OK) return rc;
  TDX_CHECK_CUDA(cudaGraphUpload(p->exec, reinterpret_cast<cudaStream_t>(stream_)));
  return TDX_OK;
}

extern "C" int tdx_program_run(TdxProgram* p, int use_graph, void* stream_) {
  TDX_REQUIRE(p, "program_run: null program");
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
  TDX_CHECK_CUDA(cudaStreamIsCapturing(stream, &st));
  if (!use_graph || st != cudaStreamCaptureStatusNone) return launch_all(p, stream);
  int rc = ensure_graph(p);
  if (rc != TDX_OK) return rc;
  TDX_CHECK_CUDA(cudaGraphLaunch(p->exec, stream));
  return TDX_OK;
}

extern "C" int tdx_program_profile(TdxProgram* p, float* ms_per_launch, int32_t* kinds, void* stream_) {
  TDX_REQUIRE(p && ms_per_launch, "program_profile: null argument");
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  const size_t n = p->ops.size();
  std::vector<cudaEvent_t> ev(n + 1);
  for (auto& e : ev) TDX_CHECK_CUDA(cudaEventCreate(&e));
  int rc = TDX_OK;
  TDX_CHECK_CUDA(cudaEventRecord(ev[0], stream));
  for (size_t i = 0; i < n && rc == TDX_OK; ++i) {
    auto& op = p->ops[i];
    switch (op.type) {
      case OP_CONV_IN: rc = conv_in_launch(op.ci, stream); break;
      case OP_IGEMM: rc = igemm_launch(op.ig, op.tms, stream); break;
      case OP_CONV_OUT: rc = conv_out_launch_impl(op.co, op.guide_out, stream); break;
      case OP_EMBED:
        op.em.blocks = op.blocks.data();
        rc = embed_launch(op.em, stream);
        break;
      case OP_ATTN: rc = attn_launch(op.at, stream); break;
      case OP_IM2COL: rc = im2col_launch(op.im, stream); break;
    }
    cudaEventRecord(ev[i + 1], stream);
    if (kinds) kinds[i] = (int32_t)op.type;
  }
  cudaError_t e = cudaStreamSynchronize(stream);
  if (rc == TDX_OK && e == cudaSuccess) {
    for (size_t i = 0; i < n; ++i) cudaEventElapsedTime(&ms_per_launch[i], ev[i], ev[i + 1]);
  }
  for (auto& evt : ev) cudaEventDestroy(evt);
  if (rc != TDX_OK) return rc;
  TDX_CHECK_CUDA(e);
  return TDX_OK;
}

extern "C" int tdx_program_destroy(TdxProgram* p) {
  if (!p) return TDX_OK;
  invalidate_graph(p);
  delete p;
  return TDX_OK;
}
