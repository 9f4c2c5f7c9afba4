// Shared declarations for the qagnn_b200 CUDA sources (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/qagnn_b200.h"

namespace qagnn {

constexpr size_t kAlign = 256;
__host__ __device__ inline size_t align_up(size_t x, size_t a = kAlign) { return (x + a - 1) / a * a; }

// ---- launch bookkeeping -------------------------------------------------------------------------
void note_launch(int n = 1);
int32_t cuda_fail(cudaError_t e, const char* file, int line);  // records the error text + call site, returns QAGNN_ERR_CUDA

#define QAGNN_CHECK_LAUNCH()                               \
  do {                                                     \
    cudaError_t e__ = cudaGetLastError();                  \
    if (e__ != cudaSuccess) return ::qagnn::cuda_fail(e__, __FILE__, __LINE__);\
    ::qagnn::note_launch();                                \
  } while (0)

#define QAGNN_CHECK_CUDA(expr)                              \
  do {                                                     \
    cudaError_t e__ = (expr);                              \
    if (e__ != cudaSuccess) return ::qagnn::cuda_fail(e__, __FILE__, __LINE__);\
  } while (0)

#define QAGNN_RETURN_IF(st)        \
  do {                             \
    int32_t s__ = (st);            \
    if (s__ != QAGNN_OK) return s__; \
  } while (0)

// ---- per-device caches (a process may drive several GPUs, e.g. the reference's encoder/decoder split) -------------
constexpr int kMaxDevices = 64;
inline int current_device() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) dev = 0;
  return dev;
}

// ---- optional stage timing (qagnn_profile_*) -------------------------------------------------------
void prof_begin(int stage, cudaStream_t st);
void prof_end(int stage, cudaStream_t st);
struct ProfScope {
  int stage; cudaStream_t st;
  ProfScope(int s, cudaStream_t t) : stage(s), st(t) { prof_begin(stage, st); }
  ~ProfScope() { prof_end(stage, st); }
};

// ---- folded-weight blob ---------------------------------------------------------------------------
// All offsets in floats from the start of the blob.  C = R*T*T + T rows in the edge tables.
struct FoldLayout {
  int D, H, T, R, k, C;
  size_t tab;        // [C, D]   edge_encoder(onehot(c))                      (layer-invariant)
  size_t hidden;     // [C, D]   scratch: ReLU(BN(lin0(onehot)))
  size_t type_tab;   // [T, D/2] GELU(emb_node_type(onehot(t)))
  size_t basis;      // [D/2]    copy of score_basis
  size_t ws;         // [D/2, D/2] emb_score.weight   (copy)
  size_t bs;         // [D/2]
  size_t vcat;       // [D, 2D]  [Vh | Vx]
  size_t vbias;      // [D]      Vh.bias + Vx.bias
  size_t layer0;     // per-layer block start
  size_t layer_stride;
  // per-layer offsets relative to the layer block
  size_t wp;         // [3D, 2D] rows: W_q/sqrt(d) ; W_k[:, :2D] ; W_m[:, :2D]
  size_t bp;         // [3D]     b_q/sqrt(d) ; 0 ; 0
  size_t ke;         // [C, D]   tab @ W_k[:, 2D:]^T + b_k
  size_t me;         // [C, D]   tab @ W_m[:, 2D:]^T + b_m
  size_t w1;         // [D, D]   BN-folded mlp.0
  size_t b1;         // [D]
  size_t w2;         // [D, D]   mlp.3 (copy)
  size_t b2;         // [D]
  size_t keh;        // [H, C, DP] head-major zero-padded copy of ke (DP = d rounded up to 4)
  size_t meh;        // [H, C, DP]
  // split-bf16 planes of the dense weights (tensor-core path); sizes in floats = elements / 2 per plane
  size_t wp_hi, wp_lo;   // [3D, 2D]
  size_t wph, bph;       // fp32 [3*H*DP, 2D] / [3*H*DP]: projection rows regrouped per head and zero-padded to DP
  size_t wph_hi, wph_lo; // its planes — the GEMM then emits the tiled path's [3][H][N][DP] layout directly
  size_t w1_hi, w1_lo;   // [D, D]
  size_t w2_hi, w2_lo;   // [D, D]
  size_t vcat_hi, vcat_lo;  // [D, 2D]  (global, not per layer)
  // fast projection of qagnn_mp_forward (tiled + tensor-core path): node_feature_extra = [type_emb | score_emb] and type_emb
  // has only T distinct rows, so its half of the projection is a per-node-type bias table and K shrinks from 2D to D + D/2
  size_t ws_hi, ws_lo;   // global: emb_score.weight planes [D/2, KSh] (KSh = D/2 rounded up to 8)
  size_t wps;            // per layer fp32 [3*H*DP, KS]: [x columns | score_emb columns] of wph (KS = D + D/2 rounded up to 8)
  size_t wps_hi, wps_lo; // its planes
  size_t tbias;          // per layer [T, 3*H*DP]: bph + wph[:, D:D+D/2] . type_tab[t]
  size_t total;      // floats
};
FoldLayout make_fold_layout(const qagnn_shape& s);

// ---- forward workspace ------------------------------------------------------------------------------
struct WorkLayout {
  size_t qkm;     // [N, 3D]  or head-major [3, H, N, DP] for the tiled path
  size_t aggr;    // [N, D]
  size_t hmid;    // [N, D]
  size_t xa, xb;  // [N, D] ping-pong layer activations
  size_t extra;   // [N, D]
  size_t sinb;    // [N, D/2]
  // split-bf16 planes [N, D] x {hi, lo} of the GEMM A operands (tensor-core path)
  size_t hp_hi, hp_lo;          // H_in
  size_t ep_hi, ep_lo;          // node_feature_extra
  size_t xp_hi[2], xp_lo[2];    // layer activations, ping-pong
  size_t ap_hi, ap_lo;          // aggr
  size_t mp_hi, mp_lo;          // mlp hidden
  size_t sb_hi, sb_lo;          // sin basis [N, KSh] planes (A operand of emb_score on the tensor-core path)
  size_t xs_hi[3], xs_lo[3];    // fast projection: [x | score_emb] planes [N, KS] (0: H_in, 1/2: layer activations, ping-pong)
  size_t score;   // [E', H]  raw logits / exp scratch (by-source order)
  size_t alpha;   // [E', H]  out-degree-scaled softmax (by-source order; general CSR path)
  size_t alpha2;  // [H, E'] x 2 words  tiled path: {row offsets, a'} per edge and head in by-target order
  size_t total;   // floats
};
WorkLayout make_work_layout(const qagnn_shape& s);

// ---- kernels' host launchers (each returns a status) ------------------------------------------
enum Act { ACT_NONE = 0, ACT_RELU = 1, ACT_GELU = 2 };

// Optional output remap of the projection GEMM for the shared-memory-tiled message passing:
// logical column c of the [M, 3D] result (Q | Kx | Mx) is stored head-major and padded,
//   C[ ((c / D) * H + (c % D) / d) * M * DP  +  r * DP  +  (c % D) % d ]        (pads are never written)
struct HeadMajorOut {
  int enabled, D, d, DP, H;
};

// C[M,N] (ldc) = act( [A1 | A2] @ W^T + bias ),  A1 [M,K1] (lda1), A2 [M,K2] (lda2) or null,
// W [N, K1+K2] row-major (ldw).  bias may be null.
int32_t sgemm_tn(const float* A1, int lda1, int K1, const float* A2, int lda2, int K2, const float* W, int ldw,
                 const float* bias, float* C, int ldc, int64_t M, int N, Act act, cudaStream_t st,
                 HeadMajorOut hm = HeadMajorOut{0, 0, 0, 0, 0});

// ---- tensor-core GEMM on split-bf16 planes (gemm_tc.cu) ---------------------------------------------
// An operand is a pair of bf16 planes [rows, K] (ld elements each): value = hi + lo.
struct TcOperand {
  const void* hi;
  const void* lo;
  int ld, K;
};
// Any subset of: fp32 row-major C, fp32 head-major padded (projection for the tiled MP), split-bf16 planes.
struct TcOutput {
  float* f32; int ldc;
  float* hm_buf; HeadMajorOut hm;
  void* hi; void* lo; int ldp;
  // optional per-row bias tables: bias becomes bias[row_class[r] * class_stride + column], classes clamped to [0, n_class)
  const int64_t* row_class; int class_stride; int n_class;
};
bool gemm_tc_available();
bool gemm_tc_shape_ok(int K1, int K2, int lda1, int lda2, int ldw, int N);
int32_t split_bf16(const float* a, int lda, long long M, int K, void* hi, void* lo, int ldp, cudaStream_t st);
int32_t gemm_tc(const TcOperand& A1, const TcOperand& A2, const TcOperand& W, const float* bias, long long M, int N,
                Act act, const TcOutput& out, cudaStream_t st);

// ---- shared-memory-tiled message passing (mp_headtile.cu) ----------------------------------------------
inline int head_dim_padded(int d) { return (d + 3) / 4 * 4; }
inline int round_up8(int k) { return (k + 7) / 8 * 8; }
// true when the per-head persistent kernel can run this shape on this device
bool headtile_supported(const qagnn_shape& s);
int32_t launch_message_passing_headtile(const qagnn_shape& s, const int32_t* prep_base, const qagnn_prep_layout& pl,
                                        const float* qkmh, const float* keh, const float* meh, float* score,
                                        float* alpha2, float* aggr, float* alpha_out, void* aggr_hi, void* aggr_lo,
                                        cudaStream_t st);
int32_t zero_head_pads(const qagnn_shape& s, float* qkmh, cudaStream_t st);

// the general CSR kernels (message_passing.cu) and their backward (mp_backward.cu) are instantiated for these shapes:
// D % 4 == 0 (float4 columns), D <= 1024 (8 chunks per lane), H in {1, 2, 4, 8, 16}
bool basic_mp_supported(const qagnn_shape& s);
int32_t launch_message_passing(const qagnn_shape& s, const int32_t* prep_base, const qagnn_prep_layout& pl,
                               const float* qkm, const float* ke, const float* me, float* score, float* alpha,
                               float* aggr, float* alpha_out, cudaStream_t st);

// column-sliced kernels with the edge tables in shared memory, for graphs too large for the per-graph tiles (mp_slice.cu)
bool slice_supported(const qagnn_shape& s);
int32_t launch_message_passing_slice(const qagnn_shape& s, const int32_t* prep_base, const qagnn_prep_layout& pl,
                                     const float* qkm, const float* ke, const float* me, float* score, float* aggr,
                                     float* alpha_out, cudaStream_t st);

int32_t launch_message_passing_backward(const qagnn_shape& s, const int32_t* prep_base, const qagnn_prep_layout& pl,
                                        const int32_t* combo_order, const float* qkm, const float* ke, const float* me,
                                        const float* alpha_s, const float* d_aggr, float* ds, float* d_qkm, float* d_ke,
                                        float* d_me, cudaStream_t st);

__device__ __forceinline__ float gelu_tanh(float x) {
  // utils/layers.py:10-14
  const float k0 = 0.7978845608028654f;  // sqrt(2/pi)
  return 0.5f * x * (1.0f + tanhf(k0 * (x + 0.044715f * x * x * x)));
}

}  // namespace qagnn
