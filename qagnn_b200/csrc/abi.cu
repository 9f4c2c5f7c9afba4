// extern "C" entry points declared in include/qagnn_b200.h: the forward orchestration of
// GATConvE (modeling/modeling_qagnn.py:411-484) and QAGNN_Message_Passing (modeling_qagnn.py:53-95).
#include <atomic>
#include <mutex>
#include <cuda_bf16.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

namespace qagnn {

static std::atomic<long long> g_launches{0};
static thread_local char g_cuda_err[256] = "";

void note_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

int32_t cuda_fail(cudaError_t e, const char* file, int line) {
  const char* base = strrchr(file, '/');
  snprintf(g_cuda_err, sizeof(g_cuda_err), "%s (%s:%d)", cudaGetErrorString(e), base ? base + 1 : file, line);
  return QAGNN_ERR_CUDA;
}

// ---- stage timing -----------------------------------------------------------------------------------
namespace {
constexpr int kProfMax = 8192;
struct ProfState {
  bool on = false;
  int n = 0;                       // recorded intervals
  cudaEvent_t ev[kProfMax][2];
  int created = 0;
  int stage[kProfMax];
  int open_idx[QAGNN_PROF_STAGES];
  std::mutex mu;  // the stage timers are process-wide diagnostics: calls from several host threads serialise here
} g_prof;
}  // namespace

void prof_begin(int stage, cudaStream_t st) {
  if (!g_prof.on) return;
  std::lock_guard<std::mutex> lk(g_prof.mu);
  if (!g_prof.on || g_prof.n >= kProfMax) { if (g_prof.on) g_prof.open_idx[stage] = -1; return; }
  const int i = g_prof.n++;
  if (i >= g_prof.created) {
    cudaEventCreate(&g_prof.ev[i][0]);
    cudaEventCreate(&g_prof.ev[i][1]);
    g_prof.created = i + 1;
  }
  g_prof.stage[i] = stage;
  g_prof.open_idx[stage] = i;
  cudaEventRecord(g_prof.ev[i][0], st);
}

void prof_end(int stage, cudaStream_t st) {
  if (!g_prof.on) return;
  std::lock_guard<std::mutex> lk(g_prof.mu);
  const int i = g_prof.open_idx[stage];
  if (i >= 0) cudaEventRecord(g_prof.ev[i][1], st);
}

WorkLayout make_work_layout(const qagnn_shape& s) {
  WorkLayout W;
  const size_t N = (size_t)s.N, D = (size_t)s.D, Ep = (size_t)(s.N + s.E), H = (size_t)s.H;
  size_t o = 0;
  auto take = [&](size_t n) { size_t r = o; o += align_up(n * 4) / 4; return r; };
  const size_t DP = (size_t)head_dim_padded((int)(D / H));
  W.qkm = take(N * 3 * (D > H * DP ? D : H * DP));
  W.aggr = take(N * D);
  W.hmid = take(N * D);
  W.xa = take(N * D);
  W.xb = take(N * D);
  W.extra = take(N * D);
  W.sinb = take(N * (D / 2));
  const size_t half = N * D / 2 + 8;  // one bf16 plane [N, D], in floats
  W.hp_hi = take(half); W.hp_lo = take(half);
  W.ep_hi = take(half); W.ep_lo = take(half);
  W.xp_hi[0] = take(half); W.xp_lo[0] = take(half);
  W.xp_hi[1] = take(half); W.xp_lo[1] = take(half);
  W.ap_hi = take(half); W.ap_lo = take(half);
  W.mp_hi = take(half); W.mp_lo = take(half);
  const size_t sbh = N * (size_t)round_up8((int)(D / 2)) / 2 + 8;  // one bf16 plane [N, KSh], in floats
  W.sb_hi = take(sbh); W.sb_lo = take(sbh);
  const size_t xsh = N * (size_t)round_up8((int)(D + D / 2)) / 2 + 8;  // one bf16 plane [N, KS], in floats
  for (int i = 0; i < 3; ++i) { W.xs_hi[i] = take(xsh); W.xs_lo[i] = take(xsh); }
  const size_t Eps = (Ep + 3) / 4 * 4;  // per-head stride of the tiled path
  W.score = take(Eps * H);
  W.alpha = take(Eps * H);
  W.alpha2 = take(2 * Eps * H);
  W.total = o;
  return W;
}

namespace {

__global__ void node_feature_prologue_kernel(int64_t N, int D, int T, const int64_t* __restrict__ node_type,
                                             const float* __restrict__ node_score, const float* __restrict__ type_tab,
                                             const float* __restrict__ basis, float* __restrict__ extra,
                                             float* __restrict__ sinb) {
  // extra[v, :D/2] = GELU(emb_node_type(onehot(type)))  == row `type` of the folded table (:65-66)
  // sinb[v, j]     = sin(1.1^j * score[v])                                                (:70-72)
  const int Dh = D / 2;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < N * Dh; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t v = i / Dh;
    const int j = (int)(i % Dh);
    int64_t t = node_type[v];
    t = t < 0 ? 0 : (t >= T ? T - 1 : t);
    extra[v * D + j] = type_tab[t * Dh + j];
    sinb[i] = sinf(basis[j] * node_score[v]);  // precise sinf: arguments reach ~1e4 * |score|
  }
}

// sin basis of the relevance score as split-bf16 planes [N, ld]: the A operand of emb_score on the tensor-core path (:70-73)
__global__ void sin_basis_planes_kernel(int64_t N, int Dh, int ld, const float* __restrict__ node_score,
                                        const float* __restrict__ basis, __nv_bfloat16* __restrict__ hi,
                                        __nv_bfloat16* __restrict__ lo) {
  const int half = Dh / 2;  // Dh even: two columns per thread
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < N * half; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t v = i / half;
    const int j = (int)(i % half) * 2;
    const float sc = node_score[v];
    const float a = sinf(basis[j] * sc), b = sinf(basis[j + 1] * sc);  // precise sinf: arguments reach ~1e4 * |score|
    __nv_bfloat162 h2, l2;
    h2.x = __float2bfloat16_rn(a); h2.y = __float2bfloat16_rn(b);
    l2.x = __float2bfloat16_rn(a - __bfloat162float(h2.x)); l2.y = __float2bfloat16_rn(b - __bfloat162float(h2.y));
    *reinterpret_cast<__nv_bfloat162*>(hi + v * ld + j) = h2;
    *reinterpret_cast<__nv_bfloat162*>(lo + v * ld + j) = l2;
  }
}

// copies `w4` 8-byte words per row (a column block of bf16 planes with row stride `ld8` words) from one hi/lo plane pair into
// two others: score_emb is layer-invariant and has to sit next to x in every [x | score_emb] operand buffer
__global__ void copy_plane_columns_kernel(int64_t N, int w4, int ld8, const uint2* __restrict__ sh, const uint2* __restrict__ sl,
                                          uint2* __restrict__ d1h, uint2* __restrict__ d1l, uint2* __restrict__ d2h,
                                          uint2* __restrict__ d2l) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < N * w4; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / w4;
    const int c = (int)(i - r * w4);
    const uint2 h = sh[r * ld8 + c], l = sl[r * ld8 + c];
    d1h[r * ld8 + c] = h; d1l[r * ld8 + c] = l;
    d2h[r * ld8 + c] = h; d2l[r * ld8 + c] = l;
  }
}

// Fused node_feature_extra for D/2 <= 128 (modeling_qagnn.py:62-73,86): one CTA = 64 nodes; emb_score's [D/2, D/2] weight
// and the CTA's sin-basis tile live in shared memory, so the whole prologue (type-table lookup, sin basis, Linear, GELU)
// is one launch that writes `extra` as fp32 and/or as the split-bf16 planes the projection GEMM consumes.
constexpr int kNfNodes = 64;
__global__ void __launch_bounds__(256) node_feature_fused_kernel(int64_t N, int D, int T, const int64_t* __restrict__ node_type,
                                                                  const float* __restrict__ node_score,
                                                                  const float* __restrict__ type_tab, const float* __restrict__ basis,
                                                                  const float* __restrict__ ws, const float* __restrict__ bs,
                                                                  float* __restrict__ extra, __nv_bfloat16* __restrict__ ex_hi,
                                                                  __nv_bfloat16* __restrict__ ex_lo) {
  extern __shared__ __align__(16) float sm_nf[];
  const int Dh = D / 2;                   // Dh % 4 == 0 (checked by the launcher)
  float* Wt = sm_nf;                      // [Dh][Dh]        Wt[k*Dh + j] = ws[j][k]
  float* Bt = Wt + (size_t)Dh * Dh;       // [Dh][kNfNodes]  Bt[k*64 + v] = sin(basis[k] * score[v])
  const int64_t v0 = (int64_t)blockIdx.x * kNfNodes;
  for (int i = threadIdx.x; i < Dh * Dh; i += 256) Wt[(i % Dh) * Dh + i / Dh] = ws[i];
  for (int i = threadIdx.x; i < kNfNodes * Dh; i += 256) {
    const int k = i / kNfNodes, vi = i % kNfNodes;
    const int64_t v = v0 + vi;
    Bt[i] = v < N ? sinf(basis[k] * node_score[v]) : 0.f;  // precise sinf: arguments reach ~1e4 * |score|
  }
  __syncthreads();
  // 4 consecutive columns of one node: one 16-byte fp32 store and/or two 8-byte bf16 stores (hi / lo planes);
  // (v*D + col) is a multiple of 4 because D % 8 == 0 and col % 4 == 0
  auto put4 = [&](int64_t v, int col, const float (&x)[4]) {
    if (extra != nullptr) *reinterpret_cast<float4*>(extra + v * D + col) = make_float4(x[0], x[1], x[2], x[3]);
    if (ex_hi != nullptr) {
      __nv_bfloat16 h[4], l[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        h[c] = __float2bfloat16_rn(x[c]);
        l[c] = __float2bfloat16_rn(x[c] - __bfloat162float(h[c]));
      }
      *reinterpret_cast<uint2*>(ex_hi + v * D + col) = *reinterpret_cast<const uint2*>(h);
      *reinterpret_cast<uint2*>(ex_lo + v * D + col) = *reinterpret_cast<const uint2*>(l);
    }
  };
  // register tile: 4 nodes x 4 outputs per thread -> two LDS.128 per 16 FMAs
  const int jg = Dh / 4, ntile = (kNfNodes / 4) * jg;
  for (int tl = threadIdx.x; tl < ntile; tl += 256) {
    const int vi0 = (tl / jg) * 4, j0 = (tl % jg) * 4;
    float acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[a][c] = 0.f;
    for (int k = 0; k < Dh; ++k) {
      const float4 b = *reinterpret_cast<const float4*>(Bt + k * kNfNodes + vi0);
      const float4 w = *reinterpret_cast<const float4*>(Wt + k * Dh + j0);
      const float bb[4] = {b.x, b.y, b.z, b.w}, ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[a][c] = fmaf(bb[a], ww[c], acc[a][c]);
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const int64_t v = v0 + vi0 + a;
      if (v >= N) continue;
      int64_t t = node_type[v];
      t = t < 0 ? 0 : (t >= T ? T - 1 : t);
      float sc[4], ty[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        sc[c] = gelu_tanh(acc[a][c] + bs[j0 + c]);
        ty[c] = type_tab[t * Dh + j0 + c];
      }
      put4(v, Dh + j0, sc);
      put4(v, j0, ty);
    }
  }
}

int32_t check_shape_fwd(const qagnn_shape* s) {
  if (!s) return QAGNN_ERR_INVALID_ARGUMENT;
  if (s->N <= 0 || s->E < 0 || s->D <= 0 || s->H <= 0 || s->T <= 0 || s->R <= 0 || s->k < 0)
    return QAGNN_ERR_INVALID_ARGUMENT;
  if (s->D % s->H != 0 || s->D % 2 != 0) return QAGNN_ERR_INVALID_ARGUMENT;
  if (s->N + s->E >= (int64_t)1 << 31) return QAGNN_ERR_INVALID_ARGUMENT;
  return QAGNN_OK;
}

// Path selection: the shared-memory-tiled kernel when the batch is made of equal small sub-graphs
// (shape.n_per_graph > 0 and the tiles fit), else the general CSR kernels.  QAGNN_MP_PATH=csr forces
// the general path (A/B measurements).
bool use_headtile(const qagnn_shape& s) {
  const char* e = getenv("QAGNN_MP_PATH");  // read at every call: tests cover every path in one process
  const bool forced = e && (strcmp(e, "csr") == 0 || strcmp(e, "basic") == 0);
  return !forced && headtile_supported(s);
}
// Without per-graph tiles: the column-sliced kernels (edge tables in shared memory) when the head width allows, else the
// basic CSR kernels; QAGNN_MP_PATH=basic forces the latter.
bool use_slice(const qagnn_shape& s) {
  const char* e = getenv("QAGNN_MP_PATH");
  return !(e && strcmp(e, "basic") == 0) && slice_supported(s);
}
// Some message-passing path takes the shape.  Checked at the entry points before anything is launched: a width no path
// can run (D % 4 != 0 without per-graph tiles) is refused up front instead of after the projection GEMM.
bool mp_path_supported(const qagnn_shape& s) { return use_headtile(s) || use_slice(s) || basic_mp_supported(s); }

// one GATConvE layer; `final_act` = ACT_NONE for the bare layer, ACT_GELU when called from mp_helper
int32_t layer_forward(const qagnn_shape& s, const FoldLayout& L, const WorkLayout& W, int layer, const float* x,
                      const float* extra, const void* prep, const qagnn_prep_layout& pl, const float* folded,
                      float* out, float* alpha_out, float* aggr_out, float* ws, Act final_act, bool tiled,
                      cudaStream_t st) {
  const int D = s.D;
  const float* lb = folded + L.layer0 + (size_t)layer * L.layer_stride;
  float* qkm = ws + W.qkm;
  float* aggr = aggr_out ? aggr_out : ws + W.aggr;
  {  // Q | Kx | Mx = [x ‖ extra] @ Wp^T + bp                     (:440, :464-466 node part, :469)
    ProfScope ps(QAGNN_PROF_PROJECTION, st);
    HeadMajorOut hm{tiled ? 1 : 0, D, D / s.H, head_dim_padded(D / s.H), s.H};
    QAGNN_RETURN_IF(sgemm_tn(x, D, D, extra, D, D, lb + L.wp, 2 * D, lb + L.bp, qkm, 3 * D, s.N, 3 * D, ACT_NONE, st, hm));
  }
  {  // logits -> per-source softmax -> out-degree rescale -> per-target sum   (:442, :469-484)
    ProfScope ps(QAGNN_PROF_MESSAGE_PASSING, st);
    if (tiled) {
      QAGNN_RETURN_IF(launch_message_passing_headtile(s, (const int32_t*)prep, pl, qkm, lb + L.keh, lb + L.meh,
                                                      ws + W.score, ws + W.alpha2, aggr, alpha_out, nullptr, nullptr, st));
    } else if (use_slice(s)) {
      QAGNN_RETURN_IF(launch_message_passing_slice(s, (const int32_t*)prep, pl, qkm, lb + L.ke, lb + L.me, ws + W.score, aggr,
                                                   alpha_out, st));
    } else {
      QAGNN_RETURN_IF(launch_message_passing(s, (const int32_t*)prep, pl, qkm, lb + L.ke, lb + L.me, ws + W.score,
                                             ws + W.alpha, aggr, alpha_out, st));
    }
  }
  {  // node MLP: Linear -> BatchNorm(eval, folded) -> ReLU -> Linear          (:443, :408)
    ProfScope ps(QAGNN_PROF_NODE_MLP, st);
    QAGNN_RETURN_IF(sgemm_tn(aggr, D, D, nullptr, 0, 0, lb + L.w1, D, lb + L.b1, ws + W.hmid, D, s.N, D, ACT_RELU, st));
    QAGNN_RETURN_IF(sgemm_tn(ws + W.hmid, D, D, nullptr, 0, 0, lb + L.w2, D, lb + L.b2, out, D, s.N, D, final_act, st));
  }
  return QAGNN_OK;
}

// Dense-path selection: tcgen05 split-bf16 GEMMs when the driver exposes TMA descriptors and the row strides
// meet TMA's 16-byte rule (D % 8 == 0); else the exact-fp32 FFMA GEMM.  QAGNN_GEMM=ffma forces the latter.
bool use_tc(const qagnn_shape& s) { return gemm_tc_available() && s.D % 8 == 0; }

struct Planes {
  const void* hi;
  const void* lo;
  int ld = 0;  // row stride in elements; 0 = D
};

// one GATConvE layer on split-bf16 planes.  x / extra are [N, D] plane pairs; the layer output goes to any of
// out_f32 (fp32 [N, D]) and out_planes.
int32_t layer_forward_tc(const qagnn_shape& s, const FoldLayout& L, const WorkLayout& W, int layer, Planes x, Planes extra,
                         const void* prep, const qagnn_prep_layout& pl, const float* folded, float* out_f32,
                         void* out_hi, void* out_lo, float* alpha_out, float* aggr_out, float* ws, Act final_act,
                         bool tiled, cudaStream_t st, const int64_t* type_bias_classes = nullptr, int out_ldp = 0) {
  const int D = s.D;
  if (out_ldp == 0) out_ldp = D;
  const float* lb = folded + L.layer0 + (size_t)layer * L.layer_stride;
  float* qkm = ws + W.qkm;
  const bool fused_split = tiled && (D / s.H) % 2 == 0;  // the tiled kernel emits the bf16 planes of aggr itself
  float* aggr = aggr_out ? aggr_out : (fused_split ? nullptr : ws + W.aggr);
  {  // Q | Kx | Mx = [x ‖ extra] @ Wp^T + bp                     (:440, :464-466 node part, :469)
    ProfScope ps(QAGNN_PROF_PROJECTION, st);
    TcOperand A1{x.hi, x.lo, x.ld ? x.ld : D, D}, A2{extra.hi, extra.lo, D, D};
    TcOutput o{};
    if (tiled && type_bias_classes != nullptr) {
      // fast form (qagnn_mp_forward): x planes are [N, KS] rows of [x | score_emb] (K = D + D/2, ONE segment); the
      // type-embedding half of node_feature_extra enters as a per-node-type bias row (T distinct rows).  One segment lets
      // the GEMM keep its weight tile resident in shared memory (gemm_tc.cu, W-resident variant)
      const int DP = head_dim_padded(D / s.H), KS = round_up8(D + D / 2);
      TcOperand Ax{x.hi, x.lo, KS, D + D / 2}, none{nullptr, nullptr, 0, 0};
      TcOperand Wp{lb + L.wps_hi, lb + L.wps_lo, KS, D + D / 2};
      o.hm_buf = qkm;
      o.hm = HeadMajorOut{1, D, D / s.H, DP, s.H};
      o.row_class = type_bias_classes; o.class_stride = 3 * s.H * DP; o.n_class = s.T;
      QAGNN_RETURN_IF(gemm_tc(Ax, none, Wp, lb + L.tbias, s.N, 3 * s.H * DP, ACT_NONE, o, st));
    } else if (tiled) {  // per-head padded weight rows -> the GEMM writes [3][H][N][DP] (pads = exact zeros) itself
      const int DP = head_dim_padded(D / s.H);
      TcOperand Wp{lb + L.wph_hi, lb + L.wph_lo, 2 * D, 2 * D};
      o.hm_buf = qkm;
      o.hm = HeadMajorOut{1, D, D / s.H, DP, s.H};
      QAGNN_RETURN_IF(gemm_tc(A1, A2, Wp, lb + L.bph, s.N, 3 * s.H * DP, ACT_NONE, o, st));
    } else {
      TcOperand Wp{lb + L.wp_hi, lb + L.wp_lo, 2 * D, 2 * D};
      o.f32 = qkm;
      o.ldc = 3 * D;
      QAGNN_RETURN_IF(gemm_tc(A1, A2, Wp, lb + L.bp, s.N, 3 * D, ACT_NONE, o, st));
    }
  }
  {  // logits -> per-source softmax -> out-degree rescale -> per-target sum   (:442, :469-484)
    ProfScope ps(QAGNN_PROF_MESSAGE_PASSING, st);
    if (tiled) {
      QAGNN_RETURN_IF(launch_message_passing_headtile(s, (const int32_t*)prep, pl, qkm, lb + L.keh, lb + L.meh,
                                                      ws + W.score, ws + W.alpha2, aggr, alpha_out,
                                                      fused_split ? ws + W.ap_hi : nullptr, ws + W.ap_lo, st));
    } else if (use_slice(s)) {
      QAGNN_RETURN_IF(launch_message_passing_slice(s, (const int32_t*)prep, pl, qkm, lb + L.ke, lb + L.me, ws + W.score, aggr,
                                                   alpha_out, st));
    } else {
      QAGNN_RETURN_IF(launch_message_passing(s, (const int32_t*)prep, pl, qkm, lb + L.ke, lb + L.me, ws + W.score,
                                             ws + W.alpha, aggr, alpha_out, st));
    }
  }
  {  // node MLP: Linear -> BatchNorm(eval, folded) -> ReLU -> Linear          (:443, :408)
    ProfScope ps(QAGNN_PROF_NODE_MLP, st);
    if (!fused_split) QAGNN_RETURN_IF(split_bf16(aggr, D, s.N, D, ws + W.ap_hi, ws + W.ap_lo, D, st));
    TcOperand A{ws + W.ap_hi, ws + W.ap_lo, D, D}, none{nullptr, nullptr, 0, 0};
    TcOperand W1{lb + L.w1_hi, lb + L.w1_lo, D, D}, W2{lb + L.w2_hi, lb + L.w2_lo, D, D};
    TcOutput o1{};
    o1.hi = ws + W.mp_hi; o1.lo = ws + W.mp_lo; o1.ldp = D;
    QAGNN_RETURN_IF(gemm_tc(A, none, W1, lb + L.b1, s.N, D, ACT_RELU, o1, st));
    TcOperand Hm{ws + W.mp_hi, ws + W.mp_lo, D, D};
    TcOutput o2{};
    o2.f32 = out_f32; o2.ldc = D; o2.hi = out_hi; o2.lo = out_lo; o2.ldp = out_ldp;
    QAGNN_RETURN_IF(gemm_tc(Hm, none, W2, lb + L.b2, s.N, D, final_act, o2, st));
  }
  return QAGNN_OK;
}

int32_t extra_forward(const qagnn_shape& s, const FoldLayout& L, const WorkLayout& W, const int64_t* node_type,
                      const float* node_score, const float* folded, float* extra, float* ws, cudaStream_t st,
                      void* ex_hi = nullptr, void* ex_lo = nullptr) {
  ProfScope ps(QAGNN_PROF_PRO_EPILOGUE, st);
  const int D = s.D, Dh = D / 2;
  if (Dh <= 128 && D % 8 == 0) {
    const size_t smem = ((size_t)Dh * Dh + (size_t)kNfNodes * Dh) * sizeof(float);
    static size_t attr[kMaxDevices] = {0};
    const int dev = current_device();
    if (smem > 48 * 1024 && smem > attr[dev]) {
      QAGNN_CHECK_CUDA(cudaFuncSetAttribute(node_feature_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      attr[dev] = smem;
    }
    node_feature_fused_kernel<<<(unsigned)((s.N + kNfNodes - 1) / kNfNodes), 256, smem, st>>>(
        s.N, D, s.T, node_type, node_score, folded + L.type_tab, folded + L.basis, folded + L.ws, folded + L.bs, extra,
        (__nv_bfloat16*)ex_hi, (__nv_bfloat16*)ex_lo);
    QAGNN_CHECK_LAUNCH();
    return QAGNN_OK;
  }
  const int64_t n = s.N * Dh;
  int64_t g = (n + 255) / 256;
  if (g > 148 * 32) g = 148 * 32;
  node_feature_prologue_kernel<<<(unsigned)g, 256, 0, st>>>(s.N, D, s.T, node_type, node_score, folded + L.type_tab,
                                                            folded + L.basis, extra, ws + W.sinb);
  QAGNN_CHECK_LAUNCH();
  // extra[:, D/2:] = GELU(emb_score(sinb))                                  (:73)
  QAGNN_RETURN_IF(sgemm_tn(ws + W.sinb, Dh, Dh, nullptr, 0, 0, folded + L.ws, Dh, folded + L.bs, extra + Dh, D, s.N, Dh,
                           ACT_GELU, st));
  if (ex_hi != nullptr) QAGNN_RETURN_IF(split_bf16(extra, D, s.N, D, ex_hi, ex_lo, D, st));
  return QAGNN_OK;
}

}  // namespace
}  // namespace qagnn

using namespace qagnn;

extern "C" int32_t qagnn_abi_version(void) { return QAGNN_ABI_VERSION; }

extern "C" const char* qagnn_status_string(int32_t status) {
  switch (status) {
    case QAGNN_OK: return "ok";
    case QAGNN_ERR_INVALID_ARGUMENT: return "invalid argument";
    case QAGNN_ERR_CUDA: return "CUDA error";
    case QAGNN_ERR_INDEX_RANGE: return "index out of range in edge_index / edge_type / node_type";
    case QAGNN_ERR_WORKSPACE: return "workspace too small";
    case QAGNN_ERR_UNSUPPORTED: return "unsupported shape";
    default: return "unknown status";
  }
}

extern "C" const char* qagnn_last_cuda_error(void) { return g_cuda_err; }

extern "C" int64_t qagnn_launch_count(void) { return (int64_t)g_launches.load(std::memory_order_relaxed); }

extern "C" int32_t qagnn_profile_enable(int32_t on) {
  std::lock_guard<std::mutex> lk(g_prof.mu);
  g_prof.on = on != 0;
  g_prof.n = 0;
  for (int i = 0; i < QAGNN_PROF_STAGES; ++i) g_prof.open_idx[i] = -1;
  return QAGNN_OK;
}

extern "C" int32_t qagnn_profile_read(double* ms_out, int64_t* count_out) {
  if (!ms_out || !count_out) return QAGNN_ERR_INVALID_ARGUMENT;
  std::lock_guard<std::mutex> lk(g_prof.mu);
  for (int i = 0; i < QAGNN_PROF_STAGES; ++i) { ms_out[i] = 0.0; count_out[i] = 0; }
  for (int i = 0; i < g_prof.n; ++i) {
    QAGNN_CHECK_CUDA(cudaEventSynchronize(g_prof.ev[i][1]));
    float ms = 0.f;
    QAGNN_CHECK_CUDA(cudaEventElapsedTime(&ms, g_prof.ev[i][0], g_prof.ev[i][1]));
    ms_out[g_prof.stage[i]] += ms;
    count_out[g_prof.stage[i]] += 1;
  }
  return QAGNN_OK;
}

extern "C" size_t qagnn_forward_workspace_bytes(const qagnn_shape* shape) {
  if (check_shape_fwd(shape) != QAGNN_OK) return 0;
  return align_up(make_work_layout(*shape).total * sizeof(float));
}

extern "C" int32_t qagnn_gatconve_forward(const qagnn_shape* shape, int32_t layer, const float* x, const float* extra,
                                          const void* prep, const void* folded, float* out, float* alpha_out,
                                          float* aggr_out, void* workspace, size_t workspace_bytes, void* stream) {
  QAGNN_RETURN_IF(check_shape_fwd(shape));
  if (!x || !extra || !prep || !folded || !out || !workspace) return QAGNN_ERR_INVALID_ARGUMENT;
  if (layer < 0 || layer >= shape->k) return QAGNN_ERR_INVALID_ARGUMENT;
  if (!mp_path_supported(*shape)) return QAGNN_ERR_UNSUPPORTED;
  const FoldLayout L = make_fold_layout(*shape);
  const WorkLayout W = make_work_layout(*shape);
  if (workspace_bytes < W.total * sizeof(float)) return QAGNN_ERR_WORKSPACE;
  qagnn_prep_layout pl;
  QAGNN_RETURN_IF(qagnn_graph_prep_layout(shape->N, shape->E, &pl));
  const bool tiled = use_headtile(*shape);
  cudaStream_t st = (cudaStream_t)stream;
  float* ws = (float*)workspace;
  if (tiled && !use_tc(*shape)) QAGNN_RETURN_IF(zero_head_pads(*shape, ws + W.qkm, st));
  if (use_tc(*shape)) {
    const int D = shape->D;
    QAGNN_RETURN_IF(split_bf16(x, D, shape->N, D, ws + W.xp_hi[0], ws + W.xp_lo[0], D, st));
    QAGNN_RETURN_IF(split_bf16(extra, D, shape->N, D, ws + W.ep_hi, ws + W.ep_lo, D, st));
    return layer_forward_tc(*shape, L, W, layer, Planes{ws + W.xp_hi[0], ws + W.xp_lo[0]}, Planes{ws + W.ep_hi, ws + W.ep_lo},
                            prep, pl, (const float*)folded, out, nullptr, nullptr, alpha_out, aggr_out, ws, ACT_NONE, tiled, st);
  }
  return layer_forward(*shape, L, W, layer, x, extra, prep, pl, (const float*)folded, out, alpha_out, aggr_out, ws,
                       ACT_NONE, tiled, st);
}

extern "C" int32_t qagnn_node_feature_extra(const qagnn_shape* shape, const int64_t* node_type, const float* node_score,
                                            const void* folded, float* extra_out, void* workspace,
                                            size_t workspace_bytes, void* stream) {
  QAGNN_RETURN_IF(check_shape_fwd(shape));
  if (!node_type || !node_score || !folded || !extra_out || !workspace) return QAGNN_ERR_INVALID_ARGUMENT;
  const FoldLayout L = make_fold_layout(*shape);
  const WorkLayout W = make_work_layout(*shape);
  if (workspace_bytes < W.total * sizeof(float)) return QAGNN_ERR_WORKSPACE;
  return extra_forward(*shape, L, W, node_type, node_score, (const float*)folded, extra_out, (float*)workspace,
                       (cudaStream_t)stream);
}

extern "C" int32_t qagnn_mp_forward(const qagnn_shape* shape, const float* H_in, const int64_t* node_type,
                                    const float* node_score, const void* prep, const void* folded, float* out,
                                    float* x_layers_out, void* workspace, size_t workspace_bytes, void* stream) {
  QAGNN_RETURN_IF(check_shape_fwd(shape));
  if (!H_in || !node_type || !node_score || !prep || !folded || !out || !workspace) return QAGNN_ERR_INVALID_ARGUMENT;
  const qagnn_shape& s = *shape;
  if (s.k > 0 && !mp_path_supported(s)) return QAGNN_ERR_UNSUPPORTED;
  const FoldLayout L = make_fold_layout(s);
  const WorkLayout W = make_work_layout(s);
  if (workspace_bytes < W.total * sizeof(float)) return QAGNN_ERR_WORKSPACE;
  qagnn_prep_layout pl;
  QAGNN_RETURN_IF(qagnn_graph_prep_layout(s.N, s.E, &pl));
  cudaStream_t st = (cudaStream_t)stream;
  float* ws = (float*)workspace;
  const float* f = (const float*)folded;
  float* extra = ws + W.extra;
  const bool tc = use_tc(s);
  const bool tiled = use_headtile(s);
  // fast form: tensor-core emb_score + type-embedding half of node_feature_extra folded into per-type bias rows
  // (QAGNN_MP_FASTPROJ=0 keeps the general [x | extra] projection, for A/B runs and tests)
  const char* efp = getenv("QAGNN_MP_FASTPROJ");
  const bool fast = tc && tiled && s.k > 0 && (s.D / 2) % 4 == 0 && !(efp && atoi(efp) == 0);
  if (fast) {
    const int D = s.D, Dh = D / 2, KSh = round_up8(Dh), KS = round_up8(D + Dh);
    char* xh[3]; char* xl[3];
    for (int i = 0; i < 3; ++i) { xh[i] = (char*)(ws + W.xs_hi[i]); xl[i] = (char*)(ws + W.xs_lo[i]); }
    {
      ProfScope ps(QAGNN_PROF_PRO_EPILOGUE, st);
      int64_t g = (s.N * (Dh / 2) + 255) / 256;
      if (g > 148 * 32) g = 148 * 32;
      sin_basis_planes_kernel<<<(unsigned)g, 256, 0, st>>>(s.N, Dh, KSh, node_score, f + L.basis, (__nv_bfloat16*)(ws + W.sb_hi),
                                                           (__nv_bfloat16*)(ws + W.sb_lo));
      QAGNN_CHECK_LAUNCH();
      // score_emb = GELU(emb_score(sin basis)) -> columns [D, D + D/2) of the H_in planes                   (:73)
      TcOperand A{ws + W.sb_hi, ws + W.sb_lo, KSh, Dh}, none{nullptr, nullptr, 0, 0}, Wsc{f + L.ws_hi, f + L.ws_lo, KSh, Dh};
      TcOutput o{};
      o.hi = xh[0] + (size_t)D * 2; o.lo = xl[0] + (size_t)D * 2; o.ldp = KS;
      QAGNN_RETURN_IF(gemm_tc(A, none, Wsc, f + L.bs, s.N, Dh, ACT_GELU, o, st));
      // ... and into the two activation buffers (layer-invariant: modeling_qagnn.py:86)
      {
        const int w4 = Dh * 2 / 8, ld8 = KS * 2 / 8;  // Dh % 4 == 0 and KS % 8 == 0 (checked by `fast`)
        int64_t gc = (s.N * w4 + 255) / 256;
        if (gc > 148 * 16) gc = 148 * 16;
        const size_t off = (size_t)D * 2;
        copy_plane_columns_kernel<<<(unsigned)gc, 256, 0, st>>>(s.N, w4, ld8, (const uint2*)(xh[0] + off), (const uint2*)(xl[0] + off),
                                                              (uint2*)(xh[1] + off), (uint2*)(xl[1] + off), (uint2*)(xh[2] + off),
                                                              (uint2*)(xl[2] + off));
        QAGNN_CHECK_LAUNCH();
      }
      QAGNN_RETURN_IF(split_bf16(H_in, D, s.N, D, xh[0], xl[0], KS, st));
    }
    const size_t ND = (size_t)s.N * s.D;
    Planes xin{xh[0], xl[0], KS};
    const Planes ep{nullptr, nullptr, 0};
    for (int l = 0; l < s.k; ++l) {  // mp_helper, :45-50 (dropout is the identity in eval)
      float* xo32 = x_layers_out ? x_layers_out + (size_t)l * ND : nullptr;
      void* ohi = xh[1 + (l & 1)];
      void* olo = xl[1 + (l & 1)];
      QAGNN_RETURN_IF(layer_forward_tc(s, L, W, l, xin, ep, prep, pl, f, xo32, ohi, olo, nullptr, nullptr, ws, ACT_GELU, tiled, st,
                                       node_type, KS));
      xin = Planes{ohi, olo, KS};
    }
    // output = GELU(Vh(H) + Vx(X))                                           (:92)
    ProfScope ps(QAGNN_PROF_PRO_EPILOGUE, st);
    TcOperand A1{xh[0], xl[0], KS, D}, A2{xin.hi, xin.lo, KS, D}, Wv{f + L.vcat_hi, f + L.vcat_lo, 2 * D, 2 * D};
    TcOutput o{};
    o.f32 = out; o.ldc = D;
    return gemm_tc(A1, A2, Wv, f + L.vbias, s.N, D, ACT_GELU, o, st);
  }
  {
    // tensor-core path: `extra` is only ever consumed as split-bf16 planes, so the prologue writes those directly
    QAGNN_RETURN_IF(extra_forward(s, L, W, node_type, node_score, f, tc && s.D / 2 <= 128 ? nullptr : extra, ws, st,
                                  tc ? ws + W.ep_hi : nullptr, tc ? ws + W.ep_lo : nullptr));
  }
  if (tiled && !use_tc(s)) QAGNN_RETURN_IF(zero_head_pads(s, ws + W.qkm, st));
  const size_t ND = (size_t)s.N * s.D;
  if (tc) {
    const int D = s.D;
    {
      ProfScope ps(QAGNN_PROF_PRO_EPILOGUE, st);
      QAGNN_RETURN_IF(split_bf16(H_in, D, s.N, D, ws + W.hp_hi, ws + W.hp_lo, D, st));
    }
    Planes xin{ws + W.hp_hi, ws + W.hp_lo};
    const Planes ep{ws + W.ep_hi, ws + W.ep_lo};
    for (int l = 0; l < s.k; ++l) {  // mp_helper, :45-50 (dropout is the identity in eval)
      float* xo32 = x_layers_out ? x_layers_out + (size_t)l * ND : nullptr;
      void* ohi = ws + W.xp_hi[l & 1];
      void* olo = ws + W.xp_lo[l & 1];
      QAGNN_RETURN_IF(layer_forward_tc(s, L, W, l, xin, ep, prep, pl, f, xo32, ohi, olo, nullptr, nullptr, ws, ACT_GELU,
                                       tiled, st));
      xin = Planes{ohi, olo};
    }
    // output = GELU(Vh(H) + Vx(X))                                           (:92)
    ProfScope ps(QAGNN_PROF_PRO_EPILOGUE, st);
    TcOperand A1{ws + W.hp_hi, ws + W.hp_lo, D, D}, A2{xin.hi, xin.lo, D, D}, Wv{f + L.vcat_hi, f + L.vcat_lo, 2 * D, 2 * D};
    TcOutput o{};
    o.f32 = out; o.ldc = D;
    if (s.k == 0) { A2 = A1; }
    return gemm_tc(A1, A2, Wv, f + L.vbias, s.N, D, ACT_GELU, o, st);
  }
  const float* x = H_in;
  for (int l = 0; l < s.k; ++l) {  // mp_helper, :45-50 (dropout is the identity in eval)
    float* xo = x_layers_out ? x_layers_out + (size_t)l * ND : ws + ((l & 1) ? W.xb : W.xa);
    QAGNN_RETURN_IF(layer_forward(s, L, W, l, x, extra, prep, pl, f, xo, nullptr, nullptr, ws, ACT_GELU, tiled, st));
    x = xo;
  }
  // output = GELU(Vh(H) + Vx(X))                                             (:92)
  ProfScope ps(QAGNN_PROF_PRO_EPILOGUE, st);
  return sgemm_tn(H_in, s.D, s.D, x, s.D, s.D, f + L.vcat, 2 * s.D, f + L.vbias, out, s.D, s.N, s.D, ACT_GELU, st);
}

extern "C" int32_t qagnn_mp_core_forward(const qagnn_shape* shape, const void* prep, const float* qkm, const float* ke,
                                         const float* me, float* aggr, float* alpha_scaled, float* alpha_out, float* scratch,
                                         void* stream) {
  QAGNN_RETURN_IF(check_shape_fwd(shape));
  if (!prep || !qkm || !ke || !me || !aggr || !alpha_scaled || !scratch) return QAGNN_ERR_INVALID_ARGUMENT;
  qagnn_prep_layout pl;
  QAGNN_RETURN_IF(qagnn_graph_prep_layout(shape->N, shape->E, &pl));
  cudaStream_t st = (cudaStream_t)stream;
  ProfScope ps(QAGNN_PROF_MESSAGE_PASSING, st);
  return launch_message_passing(*shape, (const int32_t*)prep, pl, qkm, ke, me, scratch, alpha_scaled, aggr, alpha_out, st);
}

extern "C" int32_t qagnn_mp_core_backward(const qagnn_shape* shape, const void* prep, const int32_t* combo_order,
                                          const float* qkm, const float* ke, const float* me, const float* alpha_scaled,
                                          const float* d_aggr, float* d_qkm, float* d_ke, float* d_me, float* scratch,
                                          void* stream) {
  QAGNN_RETURN_IF(check_shape_fwd(shape));
  if (!prep || !combo_order || !qkm || !ke || !me || !alpha_scaled || !d_aggr || !d_qkm || !d_ke || !d_me || !scratch)
    return QAGNN_ERR_INVALID_ARGUMENT;
  qagnn_prep_layout pl;
  QAGNN_RETURN_IF(qagnn_graph_prep_layout(shape->N, shape->E, &pl));
  return launch_message_passing_backward(*shape, (const int32_t*)prep, pl, combo_order, qkm, ke, me, alpha_scaled, d_aggr,
                                         scratch, d_qkm, d_ke, d_me, (cudaStream_t)stream);
}

extern "C" size_t qagnn_linear_workspace_bytes(int64_t M, int32_t N, int32_t K1, int32_t K2) {
  if (M <= 0 || N <= 0 || K1 <= 0 || K2 < 0) return 0;
  const size_t K = (size_t)K1 + K2;
  return align_up(2 * 2 * ((size_t)M * K + (size_t)N * K) + 8 * 1024);
}

extern "C" int32_t qagnn_linear_bf16x3(const float* A1, int32_t lda1, int32_t K1, const float* A2, int32_t lda2, int32_t K2,
                                       const float* Wt, int32_t ldw, const float* bias, float* C, int32_t ldc, int64_t M,
                                       int32_t N, int32_t act, void* workspace, size_t workspace_bytes, void* stream) {
  if (!A1 || !Wt || !C || !workspace || M <= 0 || N <= 0 || K1 <= 0 || K2 < 0 || (K2 > 0 && !A2)) return QAGNN_ERR_INVALID_ARGUMENT;
  if (act < 0 || act > 2) return QAGNN_ERR_INVALID_ARGUMENT;
  if (workspace_bytes < qagnn_linear_workspace_bytes(M, N, K1, K2)) return QAGNN_ERR_WORKSPACE;
  if (!gemm_tc_available() || !gemm_tc_shape_ok(K1, K2, K1, K2, K1 + K2, N)) return QAGNN_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  char* w = (char*)workspace;
  auto take = [&](size_t elems) { char* r = w; w += align_up(elems * 2); return (void*)r; };
  const int K = K1 + K2;
  void *a1h = take((size_t)M * K1), *a1l = take((size_t)M * K1);
  void *a2h = K2 ? take((size_t)M * K2) : nullptr, *a2l = K2 ? take((size_t)M * K2) : nullptr;
  void *wh = take((size_t)N * K), *wl = take((size_t)N * K);
  QAGNN_RETURN_IF(split_bf16(A1, lda1, M, K1, a1h, a1l, K1, st));
  if (K2) QAGNN_RETURN_IF(split_bf16(A2, lda2, M, K2, a2h, a2l, K2, st));
  QAGNN_RETURN_IF(split_bf16(Wt, ldw, N, K, wh, wl, K, st));
  TcOperand o1{a1h, a1l, K1, K1}, o2{a2h, a2l, K2, K2}, ow{wh, wl, K, K};
  TcOutput out{};
  out.f32 = C;
  out.ldc = ldc;
  return gemm_tc(o1, o2, ow, bias, M, N, (Act)act, out, st);
}
