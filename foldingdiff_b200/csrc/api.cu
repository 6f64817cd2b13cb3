// C ABI of foldingdiff_b200 (see include/foldingdiff_b200.h): handle, weight packing, per-batch
// packed-row bookkeeping, workspace, and the launch sequence of one reverse-diffusion step.
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/foldingdiff_b200.h"
#include "attention_pool.cuh"
#include "attention_tc.cuh"
#include "writers.hpp"
#include "common.cuh"
#include "gemm_tc.cuh"
#include "kernels_simt.cuh"
#include "loss.cuh"
#include "nerf.cuh"
#include "philox.cuh"

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

#define FD_CUDA(expr)                                                                      \
  do {                                                                                     \
    cudaError_t e_ = (expr);                                                               \
    if (e_ != cudaSuccess)                                                                 \
      return fail(FD_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_),     \
                  __FILE__, __LINE__);                                                     \
  } while (0)

// Entry points make the handle's device current for their own duration only (the caller's current device is
// restored on return, like any library that is handed explicit device pointers).
struct DevGuard {
  int prev = -1, want;
  explicit DevGuard(int dev) : want(dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != want) cudaSetDevice(want);
  }
  ~DevGuard() { if (prev >= 0 && prev != want) cudaSetDevice(prev); }
};

struct LayerW {
  // tensor-core path, LayerNorm folded into the projections (gemm_tc.cuh: TcLn): epilogue vectors c[n] / d[n] of the
  // QKV projection (input LN = the previous layer's output LN; layer 0: c = 0, d = bias) and of the FFN-in projection
  float *c_qkv = nullptr, *d_qkv = nullptr, *c_i = nullptr, *d_i = nullptr;
  float *w_qkv, *b_qkv, *dist, *w_o, *b_o, *ln1_g, *ln1_b, *w_i, *b_i, *w_o2, *b_o2, *ln2_g, *ln2_b;
  fd::TcWeight tq, to, ti, to2;  // tensor-core operand planes (hi / lo) of the four projections
  __half *e_hi = nullptr, *e_lo = nullptr;  // distance embedding as fp16 hi / lo, padded to 256 rows
};

}  // namespace

struct fd_handle {
  fd_dims d;
  int device = 0;
  int gemm_mode = FD_GEMM_FP32_SIMT;
  int sm_count = 148;
  std::vector<void*> allocs;  // everything cudaMalloc'ed for weights / tables
  float *w_in = nullptr, *b_in = nullptr, *emb_g = nullptr, *emb_b = nullptr;
  std::vector<LayerW> layers;
  float *w_d1 = nullptr, *b_d1 = nullptr, *hln_g = nullptr, *hln_b = nullptr, *w_d2 = nullptr,
        *b_d2 = nullptr;
  fd::TcWeight td1;
  float *c_d1 = nullptr, *d_d1 = nullptr;  // fold vectors of the decoder's dense1 (input LN = the last layer's output LN)
  float2 *stats1 = nullptr, *stats2 = nullptr;  // per-row partial (sum, sum of squares) of the two LayerNorm sites
  int stat_parts = 0;
  float* time_table = nullptr;  // (T, H) device
  std::vector<float> coef;      // (T, 4) host

  // batch state
  int batch = 0, n_pad = 0, rows = 0, rows_pad = 0, all_rows = 0;
  bool has_key_bias = false;
  int cap_batch = 0, cap_rows = 0, cap_bn = 0;
  int *row_src = nullptr, *row_start = nullptr, *n_rows = nullptr, *n_keys = nullptr;
  float* key_bias = nullptr;
  // workspace (rows_pad x width), fp32
  float *h = nullptr, *qkv = nullptr, *ctx = nullptr, *tmp = nullptr, *a = nullptr, *inter = nullptr;
  fd::TcActs tc;  // hi / lo operand planes of the activations (tensor-core modes)
  CUtensorMap att_hi, att_lo;  // per-head K / V boxes of the qkv planes (attention_pool.cuh)
  long long launches = 0;
  // Device-side pipeline error flag (gemm_tc.cuh: bounded mbarrier waits), mirrored into pinned host memory by an
  // async copy at the end of every forward / step window and checked at the next entry point and by fd_status().
  int* host_flag = nullptr;
  // One reverse step as a CUDA graph (run_steps): captured once per (batch, arithmetic, x buffer, wrap mask), replayed
  // for every further step with the step's own arguments in `dyn_dev` (kernels_simt.cuh: StepDyn).
  cudaStream_t gstream = nullptr;
  cudaEvent_t ev_in = nullptr, ev_out = nullptr;
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t gexec = nullptr;
  fd::StepDyn* dyn_dev = nullptr;
  long long batch_gen = 0, graph_gen = -1;
  int graph_mode = -1;
  const float* graph_x = nullptr;
  uint32_t graph_wrap = 0;
  long long graph_launches = 0;  // kernels per replay
  bool graph_broken = false;     // a capture failed once: stay on the eager path
  // optional CUDA-event profiler (fd_profile_begin / fd_profile_end)
  bool prof_on = false;
  std::vector<cudaEvent_t> prof_ev;  // pairs: start, stop
  std::vector<int> prof_cat;         // category of each pair
  size_t prof_used = 0;
};

namespace {

enum { CAT_EMBED = 0, CAT_GEMM_QKV, CAT_ATTN, CAT_GEMM_OUT, CAT_LN, CAT_GEMM_FFN1, CAT_GEMM_FFN2,
       CAT_GEMM_HEAD, CAT_TAIL, CAT_SPLIT, CAT_COUNT };
const char* const kCatNames[CAT_COUNT] = {"embed", "gemm_qkv", "attention", "gemm_attn_out", "layernorm",
                                          "gemm_ffn1", "gemm_ffn2", "gemm_head", "tail_posterior", "split"};

// Records a CUDA-event pair around one kernel launch when profiling is on (events on the launch stream).
struct ProfScope {
  fd_handle* h; cudaStream_t st; cudaEvent_t stop = nullptr;
  ProfScope(fd_handle* H, int cat, cudaStream_t s) : h(H), st(s) {
    if (!h || !h->prof_on) return;
    if (h->prof_used + 2 > h->prof_ev.size()) {
      for (int i = 0; i < 2; ++i) { cudaEvent_t e; cudaEventCreate(&e); h->prof_ev.push_back(e); }
    }
    cudaEvent_t start = h->prof_ev[h->prof_used];
    stop = h->prof_ev[h->prof_used + 1];
    h->prof_used += 2;
    h->prof_cat.push_back(cat);
    cudaEventRecord(start, st);
  }
  ~ProfScope() { if (stop) cudaEventRecord(stop, st); }
};

int dev_alloc(fd_handle* h, void** p, size_t bytes) {
  FD_CUDA(cudaMalloc(p, bytes));
  h->allocs.push_back(*p);
  return FD_OK;
}

int upload(fd_handle* h, float** dst, const float* src, size_t n) {
  int rc = dev_alloc(h, (void**)dst, n * sizeof(float));
  if (rc) return rc;
  FD_CUDA(cudaMemcpy(*dst, src, n * sizeof(float), cudaMemcpyHostToDevice));
  return FD_OK;
}

void free_batch(fd_handle* h) {
  cudaFree(h->row_src); cudaFree(h->row_start); cudaFree(h->n_rows); cudaFree(h->n_keys);
  cudaFree(h->key_bias);
  cudaFree(h->h); cudaFree(h->qkv); cudaFree(h->ctx); cudaFree(h->tmp); cudaFree(h->a);
  cudaFree(h->inter); cudaFree(h->stats1); cudaFree(h->stats2);
  h->stats1 = h->stats2 = nullptr;
  fd::tc_free_acts(&h->tc);
  h->row_src = h->row_start = h->n_rows = h->n_keys = nullptr;
  h->key_bias = nullptr;
  h->h = h->qkv = h->ctx = h->tmp = h->a = h->inter = nullptr;
  h->cap_batch = h->cap_rows = h->cap_bn = 0;
}

template <int VPL>
void launch_embed(fd_handle* H, const float* x, const float* temb, int temb_stride, fd::TcPlane* planes,
                  cudaStream_t st, const fd::StepDyn* dyn = nullptr) {
  const int want = (H->rows + 3) / 4, cap = H->sm_count * 3;  // persistent warps: 4 per block, 3 blocks per SM
  const int blocks = want < cap ? want : cap;
  ProfScope ps(H, CAT_EMBED, st);
  fd::launch_pdl(fd::embed_kernel<VPL>, dim3(blocks), dim3(128), 0, st, x, H->row_src, H->rows, H->n_pad, H->d.n_features,
                 H->w_in, H->b_in, H->emb_g, H->emb_b, H->d.ln_eps, temb, temb_stride, H->h,
                 planes ? planes->hi : (__half*)nullptr,
                 (planes && H->gemm_mode == FD_GEMM_TC_3X) ? planes->lo : (__half*)nullptr, dyn);
  H->launches++;
}

template <int VPL>
void launch_ln(fd_handle* H, const float* in, const float* resid, const float* g, const float* b, float* out,
               fd::TcPlane* planes, cudaStream_t st) {
  const int blocks = (H->rows * 32 + 255) / 256;
  ProfScope ps(H, CAT_LN, st);
  fd::launch_pdl(fd::layernorm_kernel<VPL>, dim3(blocks), dim3(256), 0, st, in, resid, H->rows, g, b, H->d.ln_eps, out,
                 planes ? planes->hi : (__half*)nullptr,
                 (planes && H->gemm_mode == FD_GEMM_TC_3X) ? planes->lo : (__half*)nullptr);
  H->launches++;
}

void launch_sgemm(fd_handle* H, int epi, const float* A, const float* W, const float* bias,
                  const float* resid, float* C, int M, int N, int K, cudaStream_t st) {
  dim3 grid(N / 64, M / 128);
  switch (epi) {
    case fd::EPI_BIAS:
      fd::sgemm_tn_kernel<fd::EPI_BIAS><<<grid, 256, 0, st>>>(A, W, bias, resid, C, M, N, K);
      break;
    case fd::EPI_BIAS_GELU:
      fd::sgemm_tn_kernel<fd::EPI_BIAS_GELU><<<grid, 256, 0, st>>>(A, W, bias, resid, C, M, N, K);
      break;
    default:
      fd::sgemm_tn_kernel<fd::EPI_BIAS_RESID><<<grid, 256, 0, st>>>(A, W, bias, resid, C, M, N, K);
  }
  if (H) H->launches++;
}

size_t attn_smem_bytes(int n_rows, int n_keys) {
  return sizeof(float) * ((size_t)2 * n_keys * FD_HEAD_DIM + (size_t)(n_rows + n_keys - 1) * (FD_HEAD_DIM + 1) + n_keys);
}

void launch_attention(fd_handle* H, const float* dist, cudaStream_t st) {
  dim3 grid(H->d.heads, H->batch);
  const size_t smem = attn_smem_bytes(H->n_pad, H->n_pad);
  ProfScope ps(H, CAT_ATTN, st);
  fd::attention_simt_kernel<<<grid, 128, smem, st>>>(H->qkv, H->row_start, H->n_rows, H->n_keys,
                                                     H->has_key_bias ? H->key_bias : nullptr,
                                                     H->n_pad, dist, H->d.max_pos, H->d.hidden, H->ctx);
  H->launches++;
}

// tensor-core attention on the fp16 hi / lo planes (tc modes): qkv planes -> ctx planes
int launch_attention_mma(fd_handle* H, const LayerW& w, cudaStream_t st) {
  const int items = H->batch * H->d.heads;
  const float* bias = H->has_key_bias ? H->key_bias : nullptr;
  ProfScope ps(H, CAT_ATTN, st);
  int rc;
  if (H->gemm_mode == FD_GEMM_TC_3X && fd::atc_enabled())
    rc = fd::atc_launch(H->att_hi, H->att_lo, H->row_start, H->n_rows, H->n_keys, bias, H->n_pad, w.e_hi, w.e_lo,
                        H->d.hidden, H->d.heads, items, H->tc.ctx.hi, H->tc.ctx.lo, H->sm_count, st);
  else if (H->gemm_mode == FD_GEMM_TC_3X)
    rc = fd::attp_launch<true>(H->att_hi, H->att_lo, H->tc.qkv.hi, H->tc.qkv.lo, H->row_start, H->n_rows, H->n_keys, bias,
                               H->n_pad, w.e_hi, w.e_lo, H->d.hidden, H->d.heads, items, H->tc.ctx.hi, H->tc.ctx.lo,
                               H->sm_count, st);
  else
    rc = fd::attp_launch<false>(H->att_hi, H->att_lo, H->tc.qkv.hi, H->tc.qkv.lo, H->row_start, H->n_rows, H->n_keys, bias,
                                H->n_pad, w.e_hi, w.e_lo, H->d.hidden, H->d.heads, items, H->tc.ctx.hi, H->tc.ctx.lo,
                                H->sm_count, st);
  if (rc) return fail(FD_ERR_CUDA, "attention launch failed (%d)", rc);
  H->launches++;
  return FD_OK;
}

template <int VPL, bool SAMPLE>
void launch_tail(fd_handle* H, float* eps_out, float* x, fd::StepNoise noise, float* hist,
                 fd::StepCoef coef, uint32_t wrap_bits, cudaStream_t st, const fd::StepDyn* dyn = nullptr) {
  const int want = (H->rows + 7) / 8, cap = H->sm_count * 4;  // persistent warps (kernels_simt.cuh: tail_kernel)
  const int blocks = want < cap ? want : cap;
  const size_t smem = sizeof(float) * H->d.n_features * H->d.hidden;
  ProfScope ps(H, CAT_TAIL, st);
  fd::launch_pdl(fd::tail_kernel<VPL, SAMPLE>, dim3(blocks), dim3(256), smem, st, (const float*)H->tmp,
                 (const int*)H->row_src, H->rows, H->d.n_features, (const float*)H->hln_g, (const float*)H->hln_b,
                 H->d.head_ln_eps, (const float*)H->w_d2, (const float*)H->b_d2, eps_out, x, noise, hist, coef, wrap_bits, dyn);
  H->launches++;
}

// One projection  C = A W^T + bias (+resid)(+gelu)  in the handle's arithmetic.
// `a_tc` / `c_tc` are the tensor-core operand planes that shadow A / C (nullptr where unused).
int project(fd_handle* H, int cat, int epi, const float* A, const float* W, const fd::TcWeight* tw,
            const float* bias, const float* resid, float* C, int N, int K, const fd::TcPlane* a_tc,
            fd::TcPlane* c_tc, cudaStream_t st, const fd::TcLn& ln = fd::TcLn()) {
  ProfScope ps(H, cat, st);
  if (H->gemm_mode == FD_GEMM_FP32_SIMT) {
    launch_sgemm(H, epi, A, W, bias, resid, C, H->rows_pad, N, K, st);
    return FD_OK;
  }
  int rc = fd::tc_gemm(H->gemm_mode, epi, a_tc, tw, bias, resid, C, c_tc, H->rows_pad, N, K,
                       H->sm_count, st, ln);
  if (rc != 0) return fail(FD_ERR_CUDA, "tensor-core GEMM launch failed (%d)", rc);
  H->launches++;
  return FD_OK;
}

// The noise-predictor forward on the current batch: leaves gelu(dense1(h_L)) in H->tmp.
//
// fp32 mode: every tensor fp32, CUDA-core kernels, standalone LayerNorm launches - the in-GPU reference arithmetic.
//
// tc modes: GEMM operands travel as fp16 hi / lo planes written by the producing kernel's epilogue (embed / QKV GEMM /
// attention / FFN1 GEMM / the two LayerNorm-site GEMMs) - no conversion passes - and there is NO LayerNorm kernel:
// the attention-output and FFN-output projections write the raw pre-LayerNorm rows v (fp32 + planes) and their row
// sums; the projections that consume LN(v) run on v with gamma folded into their weights and apply mean / rstd in the
// epilogue; the residual of the next site is LN(v) recomputed from v and the sums (gemm_tc.cuh: TcLn).
//   buffers: h / tc.h = the embedding output (layer 0) or v of the FFN-output site; a / tc.a = v of the attention-output
//   site; stats2 / stats1 = their row sums.
template <int VPL>
int run_encoder(fd_handle* H, const float* x, const float* temb, int temb_stride, cudaStream_t st,
                const fd::StepDyn* dyn = nullptr) {
  const int Hd = H->d.hidden, I = H->d.intermediate;
  const bool tcm = H->gemm_mode != FD_GEMM_FP32_SIMT;
  launch_embed<VPL>(H, x, temb, temb_stride, tcm ? &H->tc.h : nullptr, st, dyn);
  if (!tcm) {
    for (int l = 0; l < H->d.layers; ++l) {
      LayerW& w = H->layers[l];
      int rc = project(H, CAT_GEMM_QKV, fd::EPI_BIAS, H->h, w.w_qkv, nullptr, w.b_qkv, nullptr, H->qkv, 3 * Hd, Hd, nullptr, nullptr, st);
      if (rc) return rc;
      launch_attention(H, w.dist, st);
      rc = project(H, CAT_GEMM_OUT, fd::EPI_BIAS_RESID, H->ctx, w.w_o, nullptr, w.b_o, H->h, H->tmp, Hd, Hd, nullptr, nullptr, st);
      if (rc) return rc;
      launch_ln<VPL>(H, H->tmp, nullptr, w.ln1_g, w.ln1_b, H->a, nullptr, st);
      rc = project(H, CAT_GEMM_FFN1, fd::EPI_BIAS_GELU, H->a, w.w_i, nullptr, w.b_i, nullptr, H->inter, I, Hd, nullptr, nullptr, st);
      if (rc) return rc;
      rc = project(H, CAT_GEMM_FFN2, fd::EPI_BIAS_RESID, H->inter, w.w_o2, nullptr, w.b_o2, H->a, H->tmp, Hd, I, nullptr, nullptr, st);
      if (rc) return rc;
      launch_ln<VPL>(H, H->tmp, nullptr, w.ln2_g, w.ln2_b, H->h, nullptr, st);
    }
    return project(H, CAT_GEMM_HEAD, fd::EPI_BIAS_GELU, H->h, H->w_d1, nullptr, H->b_d1, nullptr, H->tmp, Hd, Hd, nullptr, nullptr, st);
  }
  const float inv_n = 1.0f / (float)Hd;
  const int parts = H->stat_parts;
  for (int l = 0; l < H->d.layers; ++l) {
    LayerW& w = H->layers[l];
    const LayerW* prev = l > 0 ? &H->layers[l - 1] : nullptr;
    fd::TcLn in2;  // "the A rows are raw rows of the FFN-output site": layers > 0
    if (prev) { in2.in_stats = H->stats2; in2.in_c = w.c_qkv; in2.in_parts = parts; in2.inv_n = inv_n; in2.eps = H->d.ln_eps; }
    int rc = project(H, CAT_GEMM_QKV, prev ? fd::EPI_LNIN : fd::EPI_BIAS, nullptr, nullptr, &w.tq, w.d_qkv, nullptr, nullptr,
                     3 * Hd, Hd, &H->tc.h, &H->tc.qkv, st, in2);
    if (rc) return rc;
    rc = launch_attention_mma(H, w, st);
    if (rc) return rc;
    fd::TcLn r1;  // attention-output site: residual = the layer input = embedding output (l = 0) or LN2 of layer l - 1
    r1.res_v = H->h;
    r1.out_stats = H->stats1; r1.inv_n = inv_n; r1.eps = H->d.ln_eps;
    if (prev) { r1.res_stats = H->stats2; r1.res_g = prev->ln2_g; r1.res_b = prev->ln2_b; r1.res_parts = parts; }
    rc = project(H, CAT_GEMM_OUT, fd::EPI_LNRES, nullptr, nullptr, &w.to, w.b_o, nullptr, H->a, Hd, Hd,
                 &H->tc.ctx, &H->tc.a, st, r1);
    if (rc) return rc;
    fd::TcLn in1;
    in1.in_stats = H->stats1; in1.in_c = w.c_i; in1.in_parts = parts; in1.inv_n = inv_n; in1.eps = H->d.ln_eps;
    rc = project(H, CAT_GEMM_FFN1, fd::EPI_LNIN_GELU, nullptr, nullptr, &w.ti, w.d_i, nullptr, nullptr, I, Hd, &H->tc.a,
                 &H->tc.inter, st, in1);
    if (rc) return rc;
    fd::TcLn r2;  // FFN-output site: residual = LN1 of this layer
    r2.res_v = H->a; r2.res_stats = H->stats1; r2.res_g = w.ln1_g; r2.res_b = w.ln1_b; r2.res_parts = parts;
    r2.out_stats = H->stats2; r2.inv_n = inv_n; r2.eps = H->d.ln_eps;
    rc = project(H, CAT_GEMM_FFN2, fd::EPI_LNRES, nullptr, nullptr, &w.to2, w.b_o2, nullptr, H->h, Hd, I,
                 &H->tc.inter, &H->tc.h, st, r2);
    if (rc) return rc;
  }
  fd::TcLn inh;
  inh.in_stats = H->stats2; inh.in_c = H->c_d1; inh.in_parts = parts; inh.inv_n = inv_n; inh.eps = H->d.ln_eps;
  return project(H, CAT_GEMM_HEAD, fd::EPI_LNIN_GELU, nullptr, nullptr, &H->td1, H->d_d1, nullptr, H->tmp, Hd, Hd, &H->tc.h,
                 nullptr, st, inh);
}

int check_launch() {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(FD_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
  return FD_OK;
}

// The tcgen05 pipelines end with an error code instead of hanging when an mbarrier wait exceeds ~2 s (a preempted /
// time-sliced GPU can do that).  Results of such a launch are garbage, so the code must reach the caller:
//   flag_enqueue_copy  device flag -> the handle's pinned word, stream-ordered after the kernels just enqueued
//   flag_poll          reports (and clears) a non-zero word: called on entry of every compute call, after the
//                      synchronising calls, and by fd_status() once the caller has synchronised its stream
int flag_enqueue_copy(fd_handle* h, cudaStream_t st) {
  if (h->gemm_mode == FD_GEMM_FP32_SIMT || !h->host_flag) return FD_OK;
  int* dflag = fd::tc_err_flag();
  if (!dflag) return fail(FD_ERR_CUDA, "pipeline error flag unavailable");
  FD_CUDA(cudaMemcpyAsync(h->host_flag, dflag, sizeof(int), cudaMemcpyDeviceToHost, st));
  return FD_OK;
}
int flag_poll(fd_handle* h) {
  if (!h->host_flag) return FD_OK;
  const int code = *(volatile int*)h->host_flag;
  if (code == 0) return FD_OK;
  *h->host_flag = 0;
  int* dflag = fd::tc_err_flag();
  if (dflag) cudaMemset(dflag, 0, sizeof(int));
  return fail(FD_ERR_CUDA, "tensor-core pipeline timed out on device %d (stage code %d): the results of the previous "
              "forward / step window are invalid", h->device, code);
}

}  // namespace

extern "C" {

int32_t fd_num_weights(int32_t layers) { return FD_W_HEAD + FD_W_PER_LAYER * layers + FD_W_TAIL; }

int32_t fd_abi_version(void) { return FD_ABI_VERSION; }

const char* fd_build_info(void) {
  return "foldingdiff_b200 sm_100a; gemm: fp32-simt, tcgen05-3x, tcgen05-1x; attention: fp32-simt, tcgen05-3x, mma.sync-3x";
}

const char* fd_last_error(void) { return g_err.c_str(); }

int32_t fd_create(const fd_dims* dims, const float* const* weights, int32_t n_weights,
                  const float* time_table, const float* coef, int32_t device, int32_t gemm_mode,
                  fd_handle** out) {
  if (!dims || !weights || !time_table || !coef || !out) return fail(FD_ERR_INVALID, "null argument");
  const fd_dims& d = *dims;
  if (d.hidden % 64 || d.hidden > 512 || d.hidden < 64)
    return fail(FD_ERR_UNSUPPORTED, "hidden=%d must be a multiple of 64 in [64, 512]", d.hidden);
  if (d.heads <= 0 || d.hidden != d.heads * FD_HEAD_DIM)
    return fail(FD_ERR_UNSUPPORTED, "head_dim must be %d (hidden=%d heads=%d)", FD_HEAD_DIM, d.hidden, d.heads);
  if (d.intermediate % 64) return fail(FD_ERR_UNSUPPORTED, "intermediate=%d must be a multiple of 64", d.intermediate);
  if (d.max_pos < 1 || d.max_pos > 128) return fail(FD_ERR_UNSUPPORTED, "max_pos=%d must be in [1, 128]", d.max_pos);
  if (d.n_features < 1 || d.n_features > FD_MAX_FEATURES) return fail(FD_ERR_UNSUPPORTED, "n_features=%d", d.n_features);
  if (d.layers < 1 || d.timesteps < 1) return fail(FD_ERR_INVALID, "layers/timesteps must be positive");
  if (n_weights != fd_num_weights(d.layers))
    return fail(FD_ERR_INVALID, "expected %d weight tensors, got %d", fd_num_weights(d.layers), n_weights);
  if (gemm_mode < FD_GEMM_FP32_SIMT || gemm_mode > FD_GEMM_TC_1X) return fail(FD_ERR_INVALID, "bad gemm_mode");
  if (gemm_mode != FD_GEMM_FP32_SIMT && d.max_pos != 128)
    return fail(FD_ERR_UNSUPPORTED, "the tensor-core path is specialised for max_position_embeddings = 128 (got %d); use FD_GEMM_FP32_SIMT", d.max_pos);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(FD_ERR_CUDA, "no CUDA device visible: foldingdiff_b200 has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(FD_ERR_INVALID, "device %d out of range (%d visible)", device, ndev);
  cudaDeviceProp prop;
  FD_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(FD_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
  DevGuard guard(device);

  fd_handle* h = new fd_handle();
  if (cudaHostAlloc((void**)&h->host_flag, sizeof(int), cudaHostAllocDefault) != cudaSuccess) {
    delete h;
    return fail(FD_ERR_CUDA, "pinned status word: %s", cudaGetErrorString(cudaGetLastError()));
  }
  *h->host_flag = 0;
  if (cudaStreamCreateWithFlags(&h->gstream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&h->ev_in, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&h->ev_out, cudaEventDisableTiming) != cudaSuccess ||
      cudaMalloc((void**)&h->dyn_dev, sizeof(fd::StepDyn)) != cudaSuccess) {
    const int rc0 = fail(FD_ERR_CUDA, "step-graph resources: %s", cudaGetErrorString(cudaGetLastError()));
    if (h->gstream) cudaStreamDestroy(h->gstream);
    if (h->ev_in) cudaEventDestroy(h->ev_in);
    if (h->ev_out) cudaEventDestroy(h->ev_out);
    cudaFreeHost(h->host_flag);
    delete h;
    return rc0;
  }
  if (!fd::tc_err_flag()) { cudaFreeHost(h->host_flag); delete h; return fail(FD_ERR_CUDA, "pipeline error flag allocation failed"); }
  h->d = d;
  h->device = device;
  h->gemm_mode = gemm_mode;
  h->sm_count = prop.multiProcessorCount;
  const int H = d.hidden, I = d.intermediate, F = d.n_features;
  int rc = FD_OK;
#define UP(dst, idx, n) if (!rc) rc = upload(h, &(dst), weights[idx], (size_t)(n))
  UP(h->w_in, 0, H * F); UP(h->b_in, 1, H); UP(h->emb_g, 2, H); UP(h->emb_b, 3, H);
  h->layers.resize(d.layers);
  for (int l = 0; l < d.layers && !rc; ++l) {
    const int b = FD_W_HEAD + l * FD_W_PER_LAYER;
    LayerW& w = h->layers[l];
    // fused QKV: rows [0,H) = query, [H,2H) = key, [2H,3H) = value
    rc = dev_alloc(h, (void**)&w.w_qkv, sizeof(float) * 3 * H * H);
    if (!rc) rc = dev_alloc(h, (void**)&w.b_qkv, sizeof(float) * 3 * H);
    for (int j = 0; j < 3 && !rc; ++j) {
      if (cudaMemcpy(w.w_qkv + (size_t)j * H * H, weights[b + 2 * j], sizeof(float) * H * H, cudaMemcpyHostToDevice) != cudaSuccess ||
          cudaMemcpy(w.b_qkv + (size_t)j * H, weights[b + 2 * j + 1], sizeof(float) * H, cudaMemcpyHostToDevice) != cudaSuccess)
        rc = fail(FD_ERR_CUDA, "weight upload failed");
    }
    UP(w.dist, b + 6, (2 * d.max_pos - 1) * FD_HEAD_DIM);
    UP(w.w_o, b + 7, H * H); UP(w.b_o, b + 8, H); UP(w.ln1_g, b + 9, H); UP(w.ln1_b, b + 10, H);
    UP(w.w_i, b + 11, I * H); UP(w.b_i, b + 12, I);
    UP(w.w_o2, b + 13, H * I); UP(w.b_o2, b + 14, H); UP(w.ln2_g, b + 15, H); UP(w.ln2_b, b + 16, H);
  }
  const int tb = FD_W_HEAD + d.layers * FD_W_PER_LAYER;
  UP(h->w_d1, tb + 0, H * H); UP(h->b_d1, tb + 1, H); UP(h->hln_g, tb + 2, H); UP(h->hln_b, tb + 3, H);
  UP(h->w_d2, tb + 4, F * H); UP(h->b_d2, tb + 5, F);
#undef UP
  if (!rc) rc = upload(h, &h->time_table, time_table, (size_t)d.timesteps * H);
  h->coef.assign(coef, coef + (size_t)d.timesteps * 4);
  // tensor-core operand planes of the weights (prepared once; cheap).  The projections that consume a LayerNorm
  // output carry its gamma in their K columns and its mean / beta terms in the epilogue vectors c / d (gemm_tc.cuh:
  // TcLn); the query rows of the fused QKV weight also carry the de-bias of the attention kernel's K = 32 products.
  {
    const fd::TcRz rz = fd::tc_rz();
    auto fold = [&](const float* w_dev, const float* b_dev, const float* g, const float* be, int n, int k, int q_rows,
                    float** c_out, float** d_out) -> int {
      int r = dev_alloc(h, (void**)c_out, sizeof(float) * n);
      if (!r) r = dev_alloc(h, (void**)d_out, sizeof(float) * n);
      if (r) return r;
      fd::tc_fold_vectors_kernel<<<(n * 32 + 255) / 256, 256>>>(w_dev, b_dev, g, be, n, k, q_rows, rz.alpha, rz.beta_att, *c_out, *d_out);
      return FD_OK;
    };
    for (int l = 0; l < d.layers && !rc; ++l) {
      LayerW& w = h->layers[l];
      const float* g_in = l > 0 ? h->layers[l - 1].ln2_g : nullptr;  // LayerNorm whose output this layer's QKV reads
      const float* b_in = l > 0 ? h->layers[l - 1].ln2_b : nullptr;
      if (fd::tc_pack_weight(w.w_qkv, 3 * H, H, &w.tq, H, g_in) || fd::tc_pack_weight(w.w_o, H, H, &w.to) ||
          fd::tc_pack_weight(w.w_i, I, H, &w.ti, 0, w.ln1_g) || fd::tc_pack_weight(w.w_o2, H, I, &w.to2))
        rc = fail(FD_ERR_CUDA, "tensor-core weight packing failed: %s", cudaGetErrorString(cudaGetLastError()));
      if (!rc) rc = fold(w.w_qkv, w.b_qkv, g_in, b_in, 3 * H, H, H, &w.c_qkv, &w.d_qkv);
      if (!rc) rc = fold(w.w_i, w.b_i, w.ln1_g, w.ln1_b, I, H, 0, &w.c_i, &w.d_i);
    }
    const LayerW& last = h->layers[d.layers - 1];
    if (!rc && fd::tc_pack_weight(h->w_d1, H, H, &h->td1, 0, last.ln2_g)) rc = fail(FD_ERR_CUDA, "tensor-core weight packing failed");
    if (!rc) rc = fold(h->w_d1, h->b_d1, last.ln2_g, last.ln2_b, H, H, 0, &h->c_d1, &h->d_d1);
  }
  // distance embeddings as fp16 hi / lo planes, padded to 256 rows (row 2*max_pos-1.. are zero)
  for (int l = 0; l < d.layers && !rc; ++l) {
    LayerW& w = h->layers[l];
    const size_t n = (size_t)fd::ATT_E_TABLE * FD_HEAD_DIM;
    float* padded = nullptr;
    if (cudaMalloc(&padded, n * sizeof(float)) != cudaSuccess || cudaMalloc(&w.e_hi, n * sizeof(__half)) != cudaSuccess ||
        cudaMalloc(&w.e_lo, n * sizeof(__half)) != cudaSuccess) { rc = fail(FD_ERR_CUDA, "distance-embedding planes: out of memory"); cudaFree(padded); break; }
    h->allocs.push_back(w.e_hi); h->allocs.push_back(w.e_lo);
    cudaMemset(padded, 0, n * sizeof(float));
    cudaMemcpy(padded, w.dist, sizeof(float) * (2 * d.max_pos - 1) * FD_HEAD_DIM, cudaMemcpyDeviceToDevice);
    fd::tc_split_kernel<<<16, 256>>>(padded, w.e_hi, w.e_lo, n / 4, 1.0f);
    cudaDeviceSynchronize();
    cudaFree(padded);
  }
  if (!rc) {
    cudaFuncSetAttribute(fd::attention_simt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         (int)attn_smem_bytes(128, 128));
    if (cudaDeviceSynchronize() != cudaSuccess) rc = fail(FD_ERR_CUDA, "create: %s", cudaGetErrorString(cudaGetLastError()));
  }
  if (rc) {
    fd_destroy(h);
    return rc;
  }
  *out = h;
  return FD_OK;
}

void fd_destroy(fd_handle* h) {
  if (!h) return;
  DevGuard guard(h->device);
  cudaDeviceSynchronize();  // the pinned status word may still be the target of an enqueued copy
  if (h->host_flag) cudaFreeHost(h->host_flag);
  if (h->gexec) cudaGraphExecDestroy(h->gexec);
  if (h->graph) cudaGraphDestroy(h->graph);
  if (h->gstream) cudaStreamDestroy(h->gstream);
  if (h->ev_in) cudaEventDestroy(h->ev_in);
  if (h->ev_out) cudaEventDestroy(h->ev_out);
  cudaFree(h->dyn_dev);
  free_batch(h);
  for (auto& w : h->layers) { fd::tc_free_weight(&w.tq); fd::tc_free_weight(&w.to); fd::tc_free_weight(&w.ti); fd::tc_free_weight(&w.to2); }
  fd::tc_free_weight(&h->td1);
  for (void* p : h->allocs) cudaFree(p);
  for (cudaEvent_t e : h->prof_ev) cudaEventDestroy(e);
  delete h;
}

int32_t fd_set_schedule(fd_handle* h, int32_t timesteps, const float* time_table, const float* coef) {
  if (!h || !time_table || !coef) return fail(FD_ERR_INVALID, "null argument");
  if (timesteps < 1) return fail(FD_ERR_INVALID, "timesteps=%d", timesteps);
  DevGuard guard(h->device);
  FD_CUDA(cudaDeviceSynchronize());  // no step may still be reading the old table
  float* fresh = nullptr;
  FD_CUDA(cudaMalloc(&fresh, sizeof(float) * (size_t)timesteps * h->d.hidden));
  if (cudaMemcpy(fresh, time_table, sizeof(float) * (size_t)timesteps * h->d.hidden, cudaMemcpyHostToDevice) != cudaSuccess) {
    cudaFree(fresh);
    return fail(FD_ERR_CUDA, "time table upload failed");
  }
  for (auto& p : h->allocs)
    if (p == h->time_table) p = fresh;
  cudaFree(h->time_table);
  h->time_table = fresh;
  h->d.timesteps = timesteps;
  h->coef.assign(coef, coef + (size_t)timesteps * 4);
  return FD_OK;
}

int32_t fd_set_gemm_mode(fd_handle* h, int32_t gemm_mode) {
  if (!h) return fail(FD_ERR_INVALID, "null handle");
  if (gemm_mode < FD_GEMM_FP32_SIMT || gemm_mode > FD_GEMM_TC_1X) return fail(FD_ERR_INVALID, "bad gemm_mode");
  if (gemm_mode != FD_GEMM_FP32_SIMT && h->d.max_pos != 128) return fail(FD_ERR_UNSUPPORTED, "tensor-core path needs max_pos = 128");
  h->gemm_mode = gemm_mode;
  return FD_OK;
}

int64_t fd_launch_count(const fd_handle* h) { return h ? h->launches : 0; }

int32_t fd_set_batch(fd_handle* h, int32_t batch, int32_t n_pad, const int32_t* lengths,
                     int32_t all_rows, const float* key_mask, void* stream) {
  if (!h || !lengths) return fail(FD_ERR_INVALID, "null argument");
  if (batch < 1 || n_pad < 1 || n_pad > h->d.max_pos)
    return fail(FD_ERR_INVALID, "batch=%d n_pad=%d (max_pos=%d)", batch, n_pad, h->d.max_pos);
  cudaStream_t st = (cudaStream_t)stream;
  DevGuard guard(h->device);
  std::vector<int> row_start(batch), n_rows(batch), n_keys(batch);
  long long rows = 0;
  for (int b = 0; b < batch; ++b) {
    if (lengths[b] < 1 || lengths[b] > n_pad)
      return fail(FD_ERR_INVALID, "lengths[%d]=%d outside [1, %d]", b, lengths[b], n_pad);
    n_rows[b] = all_rows ? n_pad : lengths[b];
    n_keys[b] = key_mask ? n_pad : lengths[b];
    row_start[b] = (int)rows;
    rows += n_rows[b];
  }
  const int rows_pad = (int)((rows + FD_ROW_TILE - 1) / FD_ROW_TILE * FD_ROW_TILE);
  std::vector<int> row_src(rows_pad, 0);
  for (int b = 0; b < batch; ++b)
    for (int n = 0; n < n_rows[b]; ++n) row_src[row_start[b] + n] = b * n_pad + n;

  const int Hd = h->d.hidden, I = h->d.intermediate;
  // no batch is installed until every allocation and copy below has succeeded: a failure part-way leaves the handle
  // in the "fd_set_batch has not been called" state (FD_ERR_STATE), never pointing at freed or partial buffers
  h->batch = 0; h->rows = 0; h->rows_pad = 0;
  if (batch > h->cap_batch || rows_pad > h->cap_rows || batch * n_pad > h->cap_bn) {
    FD_CUDA(cudaStreamSynchronize(st));
    free_batch(h);
    const size_t r = (size_t)rows_pad;
    FD_CUDA(cudaMalloc(&h->row_src, sizeof(int) * r));
    FD_CUDA(cudaMalloc(&h->row_start, sizeof(int) * batch));
    FD_CUDA(cudaMalloc(&h->n_rows, sizeof(int) * batch));
    FD_CUDA(cudaMalloc(&h->n_keys, sizeof(int) * batch));
    FD_CUDA(cudaMalloc(&h->key_bias, sizeof(float) * batch * n_pad));
    FD_CUDA(cudaMalloc(&h->h, sizeof(float) * r * Hd));
    FD_CUDA(cudaMalloc(&h->qkv, sizeof(float) * r * 3 * Hd));
    FD_CUDA(cudaMalloc(&h->ctx, sizeof(float) * r * Hd));
    FD_CUDA(cudaMalloc(&h->tmp, sizeof(float) * r * Hd));
    FD_CUDA(cudaMalloc(&h->a, sizeof(float) * r * Hd));
    FD_CUDA(cudaMalloc(&h->inter, sizeof(float) * r * I));
    if (fd::tc_alloc_acts(&h->tc, rows_pad, Hd, I)) return fail(FD_ERR_CUDA, "tensor-core workspace allocation failed");
    h->stat_parts = 2 * Hd / fd::tc_pick_bn(Hd);  // one slot per (column block, epilogue column group)
    FD_CUDA(cudaMalloc(&h->stats1, sizeof(float2) * r * h->stat_parts));
    FD_CUDA(cudaMalloc(&h->stats2, sizeof(float2) * r * h->stat_parts));
    FD_CUDA(cudaMemsetAsync(h->stats1, 0, sizeof(float2) * r * h->stat_parts, st));
    FD_CUDA(cudaMemsetAsync(h->stats2, 0, sizeof(float2) * r * h->stat_parts, st));
    if (fd::attp_make_map(&h->att_hi, h->tc.qkv.hi, rows_pad, 3 * Hd) || fd::attp_make_map(&h->att_lo, h->tc.qkv.lo, rows_pad, 3 * Hd))
      return fail(FD_ERR_CUDA, "attention tensor map creation failed");
    h->cap_batch = batch; h->cap_rows = rows_pad; h->cap_bn = batch * n_pad;
    // rows beyond the last valid one are never written by the row-limited kernels: keep them 0
    FD_CUDA(cudaMemsetAsync(h->h, 0, sizeof(float) * r * Hd, st));
    FD_CUDA(cudaMemsetAsync(h->ctx, 0, sizeof(float) * r * Hd, st));
    FD_CUDA(cudaMemsetAsync(h->a, 0, sizeof(float) * r * Hd, st));
  }
  FD_CUDA(cudaMemcpyAsync(h->row_src, row_src.data(), sizeof(int) * rows_pad, cudaMemcpyHostToDevice, st));
  FD_CUDA(cudaMemcpyAsync(h->row_start, row_start.data(), sizeof(int) * batch, cudaMemcpyHostToDevice, st));
  FD_CUDA(cudaMemcpyAsync(h->n_rows, n_rows.data(), sizeof(int) * batch, cudaMemcpyHostToDevice, st));
  FD_CUDA(cudaMemcpyAsync(h->n_keys, n_keys.data(), sizeof(int) * batch, cudaMemcpyHostToDevice, st));
  h->has_key_bias = key_mask != nullptr;
  if (key_mask) {
    std::vector<float> bias((size_t)batch * n_pad);
    for (size_t i = 0; i < bias.size(); ++i) bias[i] = (1.0f - key_mask[i]) * -10000.0f;  // modelling.py:452
    FD_CUDA(cudaMemcpyAsync(h->key_bias, bias.data(), sizeof(float) * bias.size(), cudaMemcpyHostToDevice, st));
  }
  // pageable-memory async copies have been staged by the time the call returns
  h->batch = batch; h->n_pad = n_pad; h->rows = (int)rows; h->rows_pad = rows_pad; h->all_rows = all_rows;
  h->batch_gen++;  // any captured step graph refers to the previous batch's geometry / buffers
  return FD_OK;
}

int32_t fd_forward(fd_handle* h, const float* x_dev, const float* temb_dev, float* eps_out_dev,
                   void* stream) {
  if (!h || !x_dev || !temb_dev || !eps_out_dev) return fail(FD_ERR_INVALID, "null argument");
  if (h->batch == 0) return fail(FD_ERR_STATE, "fd_set_batch has not been called");
  cudaStream_t st = (cudaStream_t)stream;
  DevGuard guard(h->device);
  int rc = flag_poll(h);
  if (rc) return rc;
  const int Hd = h->d.hidden;
  FD_CUDA(cudaMemsetAsync(eps_out_dev, 0, sizeof(float) * h->batch * h->n_pad * h->d.n_features, st));
  fd::StepCoef none{};
  fd::StepNoise no_noise{nullptr, 0ull, 0ull};
#define FD_FWD(V)                                                                                  \
  case V:                                                                                          \
    rc = run_encoder<V>(h, x_dev, temb_dev, Hd, st);                                               \
    if (!rc) launch_tail<V, false>(h, eps_out_dev, nullptr, no_noise, nullptr, none, 0u, st);      \
    break;
  switch (Hd / 32) {
    FD_FWD(2) FD_FWD(4) FD_FWD(6) FD_FWD(8) FD_FWD(10) FD_FWD(12) FD_FWD(14) FD_FWD(16)
    default: return fail(FD_ERR_UNSUPPORTED, "hidden=%d", Hd);
  }
#undef FD_FWD
  if (rc) return rc;
  rc = check_launch();
  if (rc) return rc;
  return flag_enqueue_copy(h, st);
}

}  // extern "C"

namespace {

// FOLDINGDIFF_B200_GRAPH=0 replays nothing: every step is launched kernel by kernel on the caller's stream.
bool graphs_enabled() {
  static const bool on = [] { const char* e = getenv("FOLDINGDIFF_B200_GRAPH"); return !(e && e[0] == '0'); }();
  return on;
}

template <int V>
int capture_step_graph(fd_handle* h, float* x_dev, uint32_t wrap_bits) {
  if (h->gexec) { cudaGraphExecDestroy(h->gexec); h->gexec = nullptr; }
  if (h->graph) { cudaGraphDestroy(h->graph); h->graph = nullptr; }
  const long long before = h->launches;
  FD_CUDA(cudaStreamBeginCapture(h->gstream, cudaStreamCaptureModeThreadLocal));
  fd::StepCoef none{};
  fd::StepNoise no_noise{nullptr, 0ull, 0ull};
  int rc = run_encoder<V>(h, x_dev, h->time_table, 0, h->gstream, h->dyn_dev);
  if (!rc) launch_tail<V, true>(h, nullptr, x_dev, no_noise, nullptr, none, wrap_bits, h->gstream, h->dyn_dev);
  cudaGraph_t g = nullptr;
  const cudaError_t e = cudaStreamEndCapture(h->gstream, &g);
  h->graph_launches = h->launches - before;
  h->launches = before;  // nothing ran: replays are counted when they are launched
  if (rc) { if (g) cudaGraphDestroy(g); return rc; }
  if (e != cudaSuccess || !g) return fail(FD_ERR_CUDA, "step graph capture failed: %s", cudaGetErrorString(e));
  h->graph = g;
  if (cudaGraphInstantiate(&h->gexec, h->graph, 0) != cudaSuccess) {
    h->gexec = nullptr;
    return fail(FD_ERR_CUDA, "step graph instantiation failed: %s", cudaGetErrorString(cudaGetLastError()));
  }
  return FD_OK;
}

// Reverse steps t = t_hi-1 .. t_lo; the k-th executed step takes its normals from noise_dev slice k, or (noise_dev
// == nullptr, philox) from elements [offset + k * slice, +slice) of the library stream `seed`.
//
// Execution: the first step of a new (batch, arithmetic, x buffer, wrap mask) combination is launched kernel by kernel
// on the caller's stream (it also performs every lazy one-time initialisation); the 63-launch sequence is then captured
// ONCE into a CUDA graph on the handle's own stream and every further step is one cudaGraphLaunch preceded by a
// 56-byte stream-ordered upload of the step's arguments (StepDyn).  The handle's stream is ordered after the caller's
// stream on entry and the caller's stream after it on exit (events), so the call keeps its contract: work is enqueued
// behind whatever the caller enqueued before, and whatever the caller enqueues next runs after the steps.
int run_steps(fd_handle* h, float* x_dev, int t_hi, int t_lo, const float* noise_dev, bool philox, uint64_t seed,
              uint64_t offset, float* history_dev, const uint8_t* wrap_mask, cudaStream_t st) {
  if (h->batch == 0) return fail(FD_ERR_STATE, "fd_set_batch has not been called");
  if (t_lo < 0 || t_hi > h->d.timesteps || t_lo >= t_hi)
    return fail(FD_ERR_INVALID, "need 0 <= t_lo < t_hi <= %d (got %d, %d)", h->d.timesteps, t_lo, t_hi);
  if (!noise_dev && !philox && !(t_hi == 1 && t_lo == 0)) return fail(FD_ERR_INVALID, "noise_dev is required for steps with t > 0");
  DevGuard guard(h->device);
  int rc = flag_poll(h);
  if (rc) return rc;
  const int Hd = h->d.hidden, F = h->d.n_features;
  uint32_t wrap_bits = 0;
  for (int f = 0; f < F; ++f) wrap_bits |= (wrap_mask[f] ? 1u : 0u) << f;
  const size_t slice = (size_t)h->batch * h->n_pad * F;
  const bool use_graph = graphs_enabled() && !h->prof_on && (t_hi - t_lo) > 1;
  bool on_gstream = false;  // the handle's stream has been ordered after the caller's and has work of this call
  for (int t = t_hi - 1, k = 0; t >= t_lo; --t, ++k) {
    const float* c = &h->coef[(size_t)t * 4];
    fd::StepCoef coef{c[0], c[1], c[2], c[3], t > 0 ? 1 : 0};
    fd::StepNoise noise{noise_dev ? noise_dev + (size_t)k * slice : nullptr, (unsigned long long)seed,
                        (unsigned long long)(offset + (uint64_t)k * slice)};
    float* hist = history_dev ? history_dev + (size_t)k * slice : nullptr;
    const float* temb = h->time_table + (size_t)t * Hd;
    const bool have_graph = use_graph && h->gexec && h->graph_gen == h->batch_gen && h->graph_mode == h->gemm_mode &&
                            h->graph_x == x_dev && h->graph_wrap == wrap_bits;
    if (have_graph) {
      if (!on_gstream) {
        FD_CUDA(cudaEventRecord(h->ev_in, st));
        FD_CUDA(cudaStreamWaitEvent(h->gstream, h->ev_in, 0));
        on_gstream = true;
      }
      const fd::StepDyn dyn{temb, noise, hist, coef};
      // pageable source: staged by the driver before the call returns, ordered on the stream behind the previous replay
      cudaError_t ge = cudaMemcpyAsync(h->dyn_dev, &dyn, sizeof(dyn), cudaMemcpyHostToDevice, h->gstream);
      if (ge == cudaSuccess) ge = cudaGraphLaunch(h->gexec, h->gstream);
      if (ge != cudaSuccess) {  // keep the caller's stream ordered behind whatever was enqueued before reporting
        cudaEventRecord(h->ev_out, h->gstream);
        cudaStreamWaitEvent(st, h->ev_out, 0);
        return fail(FD_ERR_CUDA, "step graph replay failed: %s", cudaGetErrorString(ge));
      }
      h->launches += h->graph_launches;
      continue;
    }
#define FD_STEP(V)                                                                               \
  case V:                                                                                        \
    rc = run_encoder<V>(h, x_dev, temb, 0, st);                                                  \
    if (!rc) launch_tail<V, true>(h, nullptr, x_dev, noise, hist, coef, wrap_bits, st);          \
    if (!rc && use_graph && !h->graph_broken && t > t_lo) {                                      \
      if (capture_step_graph<V>(h, x_dev, wrap_bits) == FD_OK) {                                 \
        h->graph_gen = h->batch_gen; h->graph_mode = h->gemm_mode; h->graph_x = x_dev; h->graph_wrap = wrap_bits; \
      } else {  /* not fatal: keep launching kernel by kernel, do not try again */               \
        h->graph_broken = true; h->graph_gen = -1; cudaGetLastError();                           \
      }                                                                                          \
    }                                                                                            \
    break;
    switch (Hd / 32) {
      FD_STEP(2) FD_STEP(4) FD_STEP(6) FD_STEP(8) FD_STEP(10) FD_STEP(12) FD_STEP(14) FD_STEP(16)
      default: return fail(FD_ERR_UNSUPPORTED, "hidden=%d", Hd);
    }
#undef FD_STEP
    if (rc) return rc;
  }
  if (on_gstream) {
    FD_CUDA(cudaEventRecord(h->ev_out, h->gstream));
    FD_CUDA(cudaStreamWaitEvent(st, h->ev_out, 0));
  }
  rc = check_launch();
  if (rc) return rc;
  return flag_enqueue_copy(h, st);
}

}  // namespace

extern "C" {

int32_t fd_p_sample_steps(fd_handle* h, float* x_dev, int32_t t_hi, int32_t t_lo,
                          const float* noise_dev, float* history_dev, const uint8_t* wrap_mask,
                          void* stream) {
  if (!h || !x_dev || !wrap_mask) return fail(FD_ERR_INVALID, "null argument");
  return run_steps(h, x_dev, t_hi, t_lo, noise_dev, false, 0, 0, history_dev, wrap_mask, (cudaStream_t)stream);
}

int32_t fd_p_sample_steps_philox(fd_handle* h, float* x_dev, int32_t t_hi, int32_t t_lo, uint64_t seed,
                                 uint64_t offset, float* history_dev, const uint8_t* wrap_mask, void* stream) {
  if (!h || !x_dev || !wrap_mask) return fail(FD_ERR_INVALID, "null argument");
  return run_steps(h, x_dev, t_hi, t_lo, nullptr, true, seed, offset, history_dev, wrap_mask, (cudaStream_t)stream);
}

int32_t fd_status(fd_handle* h) {
  if (!h) return fail(FD_ERR_INVALID, "null handle");
  return flag_poll(h);
}

int32_t fd_randn(float* dst_dev, int64_t n, uint64_t seed, uint64_t offset, void* stream) {
  if (!dst_dev || n < 0) return fail(FD_ERR_INVALID, "bad argument");
  if (n == 0) return FD_OK;
  fd::launch_philox_randn(dst_dev, n, seed, offset, (cudaStream_t)stream);
  return check_launch();
}

int32_t fd_sample_host(fd_handle* h, int32_t batch, int32_t n_pad, const int32_t* lengths,
                       const float* x0_host, int32_t t_start, const float* noise_host,
                       uint64_t seed, const uint8_t* wrap_mask, int32_t full_history,
                       float* out_host) {
  if (!h || !lengths || !x0_host || !wrap_mask || !out_host) return fail(FD_ERR_INVALID, "null argument");
  if (t_start < 1 || t_start > h->d.timesteps) return fail(FD_ERR_INVALID, "t_start=%d", t_start);
  DevGuard guard(h->device);
  cudaStream_t st;
  FD_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  int rc = fd_set_batch(h, batch, n_pad, lengths, 0, nullptr, st);
  const size_t slice = (size_t)batch * n_pad * h->d.n_features;
  const int chunk = t_start < 32 ? t_start : 32;
  float *x = nullptr, *z = nullptr, *hist = nullptr;
  auto cleanup = [&]() { cudaFree(x); cudaFree(z); cudaFree(hist); cudaStreamDestroy(st); };
  if (!rc && cudaMalloc(&x, sizeof(float) * slice) != cudaSuccess) rc = fail(FD_ERR_CUDA, "cudaMalloc x");
  if (!rc && noise_host && cudaMalloc(&z, sizeof(float) * slice * chunk) != cudaSuccess) rc = fail(FD_ERR_CUDA, "cudaMalloc noise");
  if (!rc && full_history && cudaMalloc(&hist, sizeof(float) * slice * chunk) != cudaSuccess) rc = fail(FD_ERR_CUDA, "cudaMalloc history");
  if (!rc && cudaMemcpyAsync(x, x0_host, sizeof(float) * slice, cudaMemcpyHostToDevice, st) != cudaSuccess) rc = fail(FD_ERR_CUDA, "H2D x0");
  if (!rc && hist) cudaMemsetAsync(hist, 0, sizeof(float) * slice * chunk, st);
  int done = 0;
  while (!rc && done < t_start) {
    const int t_hi = t_start - done;
    const int n = t_hi < chunk ? t_hi : chunk;
    if (noise_host) {
      if (cudaMemcpyAsync(z, noise_host + (size_t)done * slice, sizeof(float) * slice * n, cudaMemcpyHostToDevice, st) != cudaSuccess)
        rc = fail(FD_ERR_CUDA, "H2D noise");
      if (!rc) rc = fd_p_sample_steps(h, x, t_hi, t_hi - n, z, hist, wrap_mask, st);
    } else {  // the library's own stream: element (step, b, n, f) of `seed`, drawn inside the tail kernel
      rc = fd_p_sample_steps_philox(h, x, t_hi, t_hi - n, seed, (uint64_t)done * slice, hist, wrap_mask, st);
    }
    if (!rc && hist &&
        cudaMemcpyAsync(out_host + (size_t)done * slice, hist, sizeof(float) * slice * n, cudaMemcpyDeviceToHost, st) != cudaSuccess)
      rc = fail(FD_ERR_CUDA, "D2H history");
    done += n;
  }
  if (!rc && !full_history && cudaMemcpyAsync(out_host, x, sizeof(float) * slice, cudaMemcpyDeviceToHost, st) != cudaSuccess)
    rc = fail(FD_ERR_CUDA, "D2H result");
  if (!rc && cudaStreamSynchronize(st) != cudaSuccess) rc = fail(FD_ERR_CUDA, "sample_host: %s", cudaGetErrorString(cudaGetLastError()));
  if (!rc) rc = flag_poll(h);  // a timed-out pipeline must not return garbage as a success
  cleanup();
  return rc;
}

int32_t fd_debug_gemm(int32_t gemm_mode, const float* a_dev, const float* w_dev,
                      const float* bias_dev, float* c_dev, int32_t rows, int32_t n, int32_t k,
                      void* stream) {
  if (!a_dev || !w_dev || !c_dev) return fail(FD_ERR_INVALID, "null argument");
  if (rows % 128 || n % 64 || k % 64) return fail(FD_ERR_INVALID, "rows %% 128, n %% 64, k %% 64 must be 0");
  cudaStream_t st = (cudaStream_t)stream;
  float* zero_bias = nullptr;
  if (!bias_dev) {
    FD_CUDA(cudaMalloc(&zero_bias, sizeof(float) * n));
    FD_CUDA(cudaMemsetAsync(zero_bias, 0, sizeof(float) * n, st));
    bias_dev = zero_bias;
  }
  int rc = FD_OK;
  if (gemm_mode == FD_GEMM_FP32_SIMT) {
    launch_sgemm(nullptr, fd::EPI_BIAS, a_dev, w_dev, bias_dev, nullptr, c_dev, rows, n, k, st);
  } else {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    fd::TcWeight tw{};
    fd::TcPlane ap{};
    if (fd::tc_pack_weight(w_dev, n, k, &tw) || fd::tc_alloc_plane(&ap, rows, k)) {
      rc = fail(FD_ERR_CUDA, "debug gemm: allocation failed");
    } else {
      fd::tc_split(a_dev, &ap, rows, k, gemm_mode, st);
      int r = fd::tc_gemm(gemm_mode, fd::EPI_BIAS, &ap, &tw, bias_dev, nullptr, c_dev, nullptr, rows, n, k, sms, st);
      if (r) rc = fail(FD_ERR_CUDA, "tensor-core GEMM launch failed (%d)", r);
    }
    cudaStreamSynchronize(st);
    fd::tc_free_weight(&tw);
    fd::tc_free_plane(&ap);
  }
  if (!rc) rc = check_launch();
  if (zero_bias) { cudaStreamSynchronize(st); cudaFree(zero_bias); }
  return rc;
}

// ctx = hi + lo (fp16 planes back to fp32), for the debug hook below
__global__ void fd_join_planes_kernel(const __half* hi, const __half* lo, float* out, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    out[i] = __half2float(hi[i]) + (lo ? __half2float(lo[i]) : 0.0f);
}

int32_t fd_debug_attention(int32_t mode, const float* qkv_dev, int32_t batch, int32_t n_pad,
                           const int32_t* lengths, int32_t all_rows, const float* dist_dev, int32_t heads,
                           float* ctx_out_dev, void* stream) {
  if (!qkv_dev || !lengths || !dist_dev || !ctx_out_dev) return fail(FD_ERR_INVALID, "null argument");
  if (batch < 1 || n_pad < 1 || n_pad > 128 || heads < 1) return fail(FD_ERR_INVALID, "bad shape");
  cudaStream_t st = (cudaStream_t)stream;
  const int H = heads * FD_HEAD_DIM;
  std::vector<int> row_start(batch), n_rows(batch), n_keys(batch);
  int rows = 0;
  for (int b = 0; b < batch; ++b) {
    if (lengths[b] < 1 || lengths[b] > n_pad) return fail(FD_ERR_INVALID, "bad length");
    n_rows[b] = all_rows ? n_pad : lengths[b]; n_keys[b] = lengths[b]; row_start[b] = rows; rows += n_rows[b];
  }
  int *d_rs = nullptr, *d_nr = nullptr, *d_nk = nullptr;
  FD_CUDA(cudaMalloc(&d_rs, sizeof(int) * batch)); FD_CUDA(cudaMalloc(&d_nr, sizeof(int) * batch)); FD_CUDA(cudaMalloc(&d_nk, sizeof(int) * batch));
  FD_CUDA(cudaMemcpy(d_rs, row_start.data(), sizeof(int) * batch, cudaMemcpyHostToDevice));
  FD_CUDA(cudaMemcpy(d_nr, n_rows.data(), sizeof(int) * batch, cudaMemcpyHostToDevice));
  FD_CUDA(cudaMemcpy(d_nk, n_keys.data(), sizeof(int) * batch, cudaMemcpyHostToDevice));
  int rc = FD_OK;
  if (mode == FD_GEMM_FP32_SIMT) {
    cudaFuncSetAttribute(fd::attention_simt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)attn_smem_bytes(128, 128));
    dim3 grid(heads, batch);
    fd::attention_simt_kernel<<<grid, 128, attn_smem_bytes(n_pad, n_pad), st>>>(qkv_dev, d_rs, d_nr, d_nk, nullptr, n_pad, dist_dev, 128, H, ctx_out_dev);
  } else {
    const size_t nq = (size_t)rows * 3 * H, nqa = (size_t)(rows + 128) * 3 * H, nc = (size_t)rows * H, ne = (size_t)fd::ATT_E_TABLE * FD_HEAD_DIM;
    __half *q_hi, *q_lo, *c_hi, *c_lo, *e_hi, *e_lo; float* e_pad;
    FD_CUDA(cudaMalloc(&q_hi, nqa * 2)); FD_CUDA(cudaMalloc(&q_lo, nqa * 2));
    FD_CUDA(cudaMemsetAsync(q_hi, 0, nqa * 2, st)); FD_CUDA(cudaMemsetAsync(q_lo, 0, nqa * 2, st)); FD_CUDA(cudaMalloc(&c_hi, nc * 2)); FD_CUDA(cudaMalloc(&c_lo, nc * 2));
    FD_CUDA(cudaMalloc(&e_hi, ne * 2)); FD_CUDA(cudaMalloc(&e_lo, ne * 2)); FD_CUDA(cudaMalloc(&e_pad, ne * 4));
    FD_CUDA(cudaMemsetAsync(e_pad, 0, ne * 4, st)); FD_CUDA(cudaMemsetAsync(c_hi, 0, nc * 2, st)); FD_CUDA(cudaMemsetAsync(c_lo, 0, nc * 2, st));
    FD_CUDA(cudaMemcpyAsync(e_pad, dist_dev, sizeof(float) * 255 * FD_HEAD_DIM, cudaMemcpyDeviceToDevice, st));
    fd::tc_split_kernel<<<16, 256, 0, st>>>(e_pad, e_hi, e_lo, ne / 4, 1.0f);
    fd::tc_split_kernel<<<256, 256, 0, st>>>(qkv_dev, q_hi, q_lo, nq / 4, 1.0f);
    int sms = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int items = batch * heads;
    if (fd::atc_enabled() && mode == FD_GEMM_TC_3X) {
      CUtensorMap m_hi, m_lo;
      int arc = fd::attp_make_map(&m_hi, q_hi, rows + 128, 3 * H) || fd::attp_make_map(&m_lo, q_lo, rows + 128, 3 * H);
      if (!arc) arc = fd::atc_launch(m_hi, m_lo, d_rs, d_nr, d_nk, nullptr, n_pad, e_hi, e_lo, H, heads, items, c_hi, c_lo, sms, st);
      if (arc) rc = fail(FD_ERR_CUDA, "debug attention: tcgen05 launch failed (%d)", arc);
    } else {
      CUtensorMap m_hi, m_lo;
      int arc = fd::attp_make_map(&m_hi, q_hi, rows + 128, 3 * H) || fd::attp_make_map(&m_lo, q_lo, rows + 128, 3 * H);
      if (!arc) arc = mode == FD_GEMM_TC_3X
          ? fd::attp_launch<true>(m_hi, m_lo, q_hi, q_lo, d_rs, d_nr, d_nk, nullptr, n_pad, e_hi, e_lo, H, heads, items, c_hi, c_lo, sms, st)
          : fd::attp_launch<false>(m_hi, m_lo, q_hi, q_lo, d_rs, d_nr, d_nk, nullptr, n_pad, e_hi, e_lo, H, heads, items, c_hi, c_lo, sms, st);
      if (arc) rc = fail(FD_ERR_CUDA, "debug attention: pool launch failed (%d)", arc);
    }
    fd_join_planes_kernel<<<256, 256, 0, st>>>(c_hi, mode == FD_GEMM_TC_3X ? c_lo : nullptr, ctx_out_dev, nc);
    cudaStreamSynchronize(st);
    cudaFree(q_hi); cudaFree(q_lo); cudaFree(c_hi); cudaFree(c_lo); cudaFree(e_hi); cudaFree(e_lo); cudaFree(e_pad);
  }
  if (cudaStreamSynchronize(st) != cudaSuccess || cudaGetLastError() != cudaSuccess) rc = fail(FD_ERR_CUDA, "debug attention: %s", cudaGetErrorString(cudaGetLastError()));
  cudaFree(d_rs); cudaFree(d_nr); cudaFree(d_nk);
  return rc;
}

int32_t fd_profile_begin(fd_handle* h) {
  if (!h) return fail(FD_ERR_INVALID, "null handle");
  DevGuard guard(h->device);
  FD_CUDA(cudaDeviceSynchronize());
  h->prof_used = 0;
  h->prof_cat.clear();
  h->prof_on = true;
  return FD_OK;
}

int32_t fd_profile_end(fd_handle* h, float* ms_out, int64_t* launches_out) {
  if (!h || !ms_out || !launches_out) return fail(FD_ERR_INVALID, "null argument");
  h->prof_on = false;
  DevGuard guard(h->device);
  FD_CUDA(cudaDeviceSynchronize());
  for (int c = 0; c < CAT_COUNT; ++c) { ms_out[c] = 0.0f; launches_out[c] = 0; }
  for (size_t i = 0; i < h->prof_cat.size(); ++i) {
    float ms = 0.0f;
    if (cudaEventElapsedTime(&ms, h->prof_ev[2 * i], h->prof_ev[2 * i + 1]) == cudaSuccess) {
      ms_out[h->prof_cat[i]] += ms;
      launches_out[h->prof_cat[i]] += 1;
    }
  }
  return FD_OK;
}

int32_t fd_profile_num_categories(void) { return CAT_COUNT; }

const char* fd_profile_category_name(int32_t i) { return (i >= 0 && i < CAT_COUNT) ? kCatNames[i] : ""; }

int32_t fd_nerf_build(const float* angles_dev, int32_t batch, int32_t n_pad, int32_t n_features,
                      const int32_t* lengths, const int32_t* columns, int32_t center, float* coords_out_dev,
                      void* stream) {
  if (!angles_dev || !lengths || !columns || !coords_out_dev) return fail(FD_ERR_INVALID, "null argument");
  if (batch < 1 || n_pad < 1 || n_features < 3) return fail(FD_ERR_INVALID, "bad shape");
  for (int i = 0; i < 6; ++i)
    if (columns[i] >= n_features || (i < 3 && columns[i] < 0))
      return fail(FD_ERR_INVALID, "columns[%d]=%d (phi, psi, omega are required; all must be < n_features)", i, columns[i]);
  for (int b = 0; b < batch; ++b)
    if (lengths[b] < 1 || lengths[b] > n_pad) return fail(FD_ERR_INVALID, "lengths[%d]=%d outside [1, %d]", b, lengths[b], n_pad);
  cudaStream_t st = (cudaStream_t)stream;
  int* d_len = nullptr;
  FD_CUDA(cudaMalloc(&d_len, sizeof(int) * batch));
  if (cudaMemcpyAsync(d_len, lengths, sizeof(int) * batch, cudaMemcpyHostToDevice, st) != cudaSuccess) {
    cudaFree(d_len);
    return fail(FD_ERR_CUDA, "nerf: H2D lengths");
  }
  fd::NerfCols cols{columns[0], columns[1], columns[2], columns[3], columns[4], columns[5]};
  fd::nerf_kernel<<<(batch + 31) / 32, 32, 0, st>>>(angles_dev, d_len, batch, n_pad, n_features, cols, center, coords_out_dev);
  int rc = check_launch();
  cudaStreamSynchronize(st);  // d_len must outlive the kernel
  cudaFree(d_len);
  return rc;
}

// ---- output writers (host only; SURVEY section 8f rank 2) -------------------------------------------------
int32_t fd_write_angles_csv_gz(const float* angles_host, int32_t n_rows, int32_t n_features, int32_t row_stride,
                               const char* const* feature_names, const char* path, int32_t gz_level) {
  if (!angles_host || !feature_names || !path) return fail(FD_ERR_INVALID, "null argument");
  if (n_rows < 0 || n_features < 1 || row_stride < n_features) return fail(FD_ERR_INVALID, "bad shape");
  const int rc = fdw::write_gz(path, fdw::angles_csv_text(angles_host, n_rows, n_features, row_stride, feature_names), gz_level);
  return rc ? fail(FD_ERR_INVALID, "cannot write %s (%d)", path, rc) : FD_OK;
}

int32_t fd_write_backbone_pdb(const float* coords_host, int32_t n_atoms, const char* path) {
  if (!coords_host || !path) return fail(FD_ERR_INVALID, "null argument");
  if (n_atoms < 0 || n_atoms % 3 != 0) return fail(FD_ERR_INVALID, "expected 3N atoms (N, CA, C per residue), got %d", n_atoms);
  if (n_atoms > 99999) return fail(FD_ERR_INVALID, "%d atoms do not fit the PDB serial field", n_atoms);
  const int rc = fdw::write_text(path, fdw::backbone_pdb_text(coords_host, n_atoms));
  return rc ? fail(FD_ERR_INVALID, "cannot write %s (%d)", path, rc) : FD_OK;
}

int32_t fd_write_batch(int32_t n_chains, const float* angles_host, int32_t n_pad, int32_t n_features,
                       const char* const* feature_names, const float* coords_host, int32_t atoms_pad,
                       const int32_t* lengths, const char* const* csv_paths, const char* const* pdb_paths,
                       int32_t n_threads, int32_t gz_level) {
  if (!lengths || n_chains < 0) return fail(FD_ERR_INVALID, "bad argument");
  if (csv_paths && (!angles_host || !feature_names || n_features < 1 || n_pad < 1)) return fail(FD_ERR_INVALID, "csv output needs angles");
  if (pdb_paths && (!coords_host || atoms_pad < 3)) return fail(FD_ERR_INVALID, "pdb output needs coordinates");
  std::vector<fdw::BatchJob> jobs((size_t)n_chains);
  for (int i = 0; i < n_chains; ++i) {
    const int n = lengths[i];
    if (n < 1 || (csv_paths && n > n_pad) || (pdb_paths && (3 * n > atoms_pad || 3 * n > 99999)))
      return fail(FD_ERR_INVALID, "lengths[%d]=%d does not fit the padded arrays", i, n);
    fdw::BatchJob& j = jobs[(size_t)i];
    j.angles = csv_paths ? angles_host + (size_t)i * n_pad * n_features : nullptr;
    j.n_rows = n; j.n_features = n_features; j.row_stride = n_features; j.names = feature_names;
    j.csv_path = csv_paths ? csv_paths[i] : nullptr;
    j.coords = pdb_paths ? coords_host + (size_t)i * atoms_pad * 3 : nullptr;
    j.n_atoms = 3 * n;
    j.pdb_path = pdb_paths ? pdb_paths[i] : nullptr;
  }
  const int bad = fdw::run_batch(jobs, n_threads, gz_level);
  return bad ? fail(FD_ERR_INVALID, "%d output files could not be written", bad) : FD_OK;
}

// ---- forward half of the training step (loss.cuh; SURVEY section 8f rank 3) --------------------------------------
int32_t fd_q_sample(const float* x0_dev, int32_t batch, int32_t n_pad, int32_t n_features, const float* sqrt_abar_dev,
                    const float* sqrt_1m_abar_dev, const float* var_scale, const uint8_t* angular, const float* z_dev,
                    uint64_t seed, uint64_t offset, float* known_noise_dev, float* corrupted_dev, void* stream) {
  if (!x0_dev || !sqrt_abar_dev || !sqrt_1m_abar_dev || !var_scale || !angular || !known_noise_dev || !corrupted_dev)
    return fail(FD_ERR_INVALID, "null argument");
  if (batch < 1 || n_pad < 1 || n_features < 1 || n_features > FD_MAX_FEATURES)
    return fail(FD_ERR_INVALID, "bad shape: batch=%d n_pad=%d n_features=%d", batch, n_pad, n_features);
  fd::FeatureScales sc{};
  uint32_t ang_bits = 0;
  for (int f = 0; f < n_features; ++f) {
    sc.s[f] = var_scale[f];
    ang_bits |= (angular[f] ? 1u : 0u) << f;
  }
  const long long total = (long long)batch * n_pad * n_features;
  const long long want = (total + 255) / 256;
  fd::q_sample_kernel<<<(unsigned)(want < 4096 ? want : 4096), 256, 0, (cudaStream_t)stream>>>(
      x0_dev, total, n_pad, n_features, sqrt_abar_dev, sqrt_1m_abar_dev, sc, ang_bits, z_dev, seed, offset,
      known_noise_dev, corrupted_dev);
  return check_launch();
}

int32_t fd_loss_terms(const float* eps_hat_dev, const float* known_noise_dev, const float* attn_mask_dev, int32_t batch,
                      int32_t n_pad, int32_t n_features, const uint8_t* angular, int32_t loss, float circle_penalty,
                      double* chain_sums_dev, float* terms_dev, void* stream) {
  if (!eps_hat_dev || !known_noise_dev || !attn_mask_dev || !angular || !chain_sums_dev || !terms_dev)
    return fail(FD_ERR_INVALID, "null argument");
  if (batch < 1 || n_pad < 1 || n_features < 1 || n_features > FD_MAX_FEATURES)
    return fail(FD_ERR_INVALID, "bad shape: batch=%d n_pad=%d n_features=%d", batch, n_pad, n_features);
  if (loss != FD_LOSS_SMOOTH_L1 && loss != FD_LOSS_L1) return fail(FD_ERR_INVALID, "loss=%d", loss);
  if (!(circle_penalty >= 0.0f)) return fail(FD_ERR_INVALID, "circle_penalty must be >= 0");
  uint32_t ang_bits = 0;
  for (int f = 0; f < n_features; ++f) ang_bits |= (angular[f] ? 1u : 0u) << f;
  cudaStream_t st = (cudaStream_t)stream;
  fd::loss_chain_kernel<<<batch, fd::LOSS_THREADS, 0, st>>>(eps_hat_dev, known_noise_dev, attn_mask_dev, n_pad, n_features,
                                                             ang_bits, loss, circle_penalty > 0.0f ? 1 : 0, chain_sums_dev);
  fd::loss_reduce_kernel<<<1, 32, 0, st>>>(chain_sums_dev, batch, n_features, circle_penalty, terms_dev);
  return check_launch();
}

int32_t fd_pdist_loss(const float* corrupted_dev, const float* eps_hat_dev, const float* known_angles_dev,
                      const float* sqrt_abar_dev, const float* sqrt_1m_abar_dev, const float* coef_dev, int32_t batch,
                      int32_t n_pad, int32_t n_features, const int32_t* lengths, const int32_t* columns,
                      float* denoised_dev, double* chain_sums_dev, float* loss_dev, void* stream) {
  if (!corrupted_dev || !eps_hat_dev || !known_angles_dev || !sqrt_abar_dev || !sqrt_1m_abar_dev || !coef_dev || !lengths ||
      !columns || !loss_dev)
    return fail(FD_ERR_INVALID, "null argument");
  if (batch < 1 || n_pad < 1 || n_pad > 128 || n_features < 3 || n_features > FD_MAX_FEATURES)
    return fail(FD_ERR_INVALID, "bad shape: batch=%d n_pad=%d (<= 128) n_features=%d", batch, n_pad, n_features);
  for (int i = 0; i < 6; ++i)
    if (columns[i] >= n_features || (i < 3 && columns[i] < 0))
      return fail(FD_ERR_INVALID, "columns[%d]=%d (phi, psi, omega are required; all must be < n_features)", i, columns[i]);
  for (int b = 0; b < batch; ++b)
    if (lengths[b] < 1 || lengths[b] > n_pad) return fail(FD_ERR_INVALID, "lengths[%d]=%d outside [1, %d]", b, lengths[b], n_pad);
  cudaStream_t st = (cudaStream_t)stream;
  const size_t n_ang = (size_t)batch * n_pad * n_features, n_xyz = (size_t)batch * n_pad * 9;
  // stream-ordered scratch: freed behind the kernels, so the call does not synchronise
  char* work = nullptr;
  const size_t bytes = sizeof(float) * (2 * n_xyz + (denoised_dev ? 0 : n_ang)) + sizeof(double) * (chain_sums_dev ? 0 : 2 * (size_t)batch) +
                       sizeof(int) * (size_t)batch + 64;
  FD_CUDA(cudaMallocAsync((void**)&work, bytes, st));
  float* xyz_a = (float*)work;
  float* xyz_b = xyz_a + n_xyz;
  float* den = denoised_dev ? denoised_dev : xyz_b + n_xyz;
  char* tail = (char*)(denoised_dev ? xyz_b + n_xyz : den + n_ang);
  tail = (char*)(((uintptr_t)tail + 15) & ~(uintptr_t)15);
  double* chain = chain_sums_dev ? chain_sums_dev : (double*)tail;
  int* d_len = (int*)(chain_sums_dev ? tail : tail + sizeof(double) * 2 * (size_t)batch);
  int rc = FD_OK;
  if (cudaMemcpyAsync(d_len, lengths, sizeof(int) * batch, cudaMemcpyHostToDevice, st) != cudaSuccess)
    rc = fail(FD_ERR_CUDA, "pdist: H2D lengths");
  if (!rc) {
    const long long total = (long long)n_ang, want = (total + 255) / 256;
    fd::denoise_kernel<<<(unsigned)(want < 4096 ? want : 4096), 256, 0, st>>>(corrupted_dev, eps_hat_dev, total,
                                                                              (long long)n_pad * n_features, sqrt_abar_dev,
                                                                              sqrt_1m_abar_dev, den);
    // both structures through the library's one NeRF (nerf.cuh), uncentred: the term is translation invariant
    const fd::NerfCols cols{columns[0], columns[1], columns[2], columns[3], columns[4], columns[5]};
    fd::nerf_kernel<<<(batch + 31) / 32, 32, 0, st>>>(den, d_len, batch, n_pad, n_features, cols, 0, xyz_a);
    fd::nerf_kernel<<<(batch + 31) / 32, 32, 0, st>>>(known_angles_dev, d_len, batch, n_pad, n_features, cols, 0, xyz_b);
    fd::pdist_chain_kernel<<<batch, fd::LOSS_THREADS, 0, st>>>(xyz_a, xyz_b, d_len, n_pad, coef_dev, chain);
    fd::pdist_reduce_kernel<<<1, 32, 0, st>>>(chain, batch, loss_dev);
    rc = check_launch();
  }
  cudaFreeAsync(work, st);
  return rc;
}

int32_t fd_debug_tc_status(void) { return fd::tc_check_error(); }

int32_t fd_debug_graph_state(const fd_handle* h) {
  if (!h) return 0;
  if (h->graph_broken) return -1;
  return (h->gexec && h->graph_gen == h->batch_gen) ? 1 : 0;
}

int32_t fd_debug_attention_dump(float* dump_dev) {
  fd::atc_debug_dump() = dump_dev;
  return FD_OK;
}

}  // extern "C"
