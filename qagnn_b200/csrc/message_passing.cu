// Message passing of one GATConvE layer (modeling/modeling_qagnn.py:442,455-484 + the
// torch_geometric propagate/softmax and torch_scatter scatter it calls), on node-level projections:
//
//   s[e,h]   = sum_j Q[src,h,j] * (Kx[tgt,h,j] + Ke[combo,h,j])          (:464,:466,:469-470)
//   a[e,h]   = softmax over the edges that share SRC                       (:471-472)
//   a'[e,h]  = a[e,h] * outdeg(src)                                        (:476-481)
//   aggr[v]  = sum_{e: tgt=v} a'[e,h] * (Mx[src,h,:] + Me[combo,h,:])      (:465,:483-484, aggr="add")
//
// General path (any graph size): two kernels over the CSR orders built by graph_prep.
//   mp_scores_kernel     one warp per SOURCE node  : logits, segment softmax, rescale
//   mp_aggregate_kernel  one warp per TARGET node  : weighted sum of messages
// No atomics, no global max/sum scratch passes; every summation runs in edge-id order, so results
// are deterministic and follow the reference's CPU summation order.
#include "common.cuh"

namespace qagnn {

namespace {

struct HeadMap {
  // heads of the 4 elements of float4 chunk `c` (d = dim per head)
  int first, last;
  int hid[4];
};

__device__ __forceinline__ HeadMap head_map(int c, int d) {
  HeadMap m;
#pragma unroll
  for (int t = 0; t < 4; ++t) m.hid[t] = (4 * c + t) / d;
  m.first = m.hid[0];
  m.last = m.hid[3];
  return m;
}

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }

template <int H, int CH>
__global__ void __launch_bounds__(256) mp_scores_kernel(int64_t N, int D, const int32_t* __restrict__ rowptr_src,
                                                        const int32_t* __restrict__ csr_src_tgt,
                                                        const int32_t* __restrict__ csr_src_combo,
                                                        const int32_t* __restrict__ perm_src,
                                                        const float* __restrict__ qkm, const float* __restrict__ ke,
                                                        float* __restrict__ score, float* __restrict__ alpha,
                                                        float* __restrict__ alpha_out) {
  const int lane = threadIdx.x & 31;
  const int64_t v = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (v >= N) return;
  const int d = D / H;
  const int ld = 3 * D;

  float4 q[CH];
  HeadMap hm[CH];
  bool valid[CH];
#pragma unroll
  for (int i = 0; i < CH; ++i) {
    const int c = lane + 32 * i;
    valid[i] = 4 * c < D;
    hm[i] = head_map(c, d);
    q[i] = valid[i] ? ld4(qkm + v * ld + 4 * c) : make_float4(0.f, 0.f, 0.f, 0.f);
  }

  const int beg = rowptr_src[v], end = rowptr_src[v + 1];
  float mx[H];
#pragma unroll
  for (int h = 0; h < H; ++h) mx[h] = -INFINITY;

  // pass 1: logits
  for (int p = beg; p < end; ++p) {
    const int t = csr_src_tgt[p];
    const int cb = csr_src_combo[p];
    float part[H];
#pragma unroll
    for (int h = 0; h < H; ++h) part[h] = 0.f;
#pragma unroll
    for (int i = 0; i < CH; ++i) {
      if (!valid[i]) continue;
      const int c = lane + 32 * i;
      const float4 kx = ld4(qkm + (int64_t)t * ld + D + 4 * c);
      const float4 kt = ld4(ke + (int64_t)cb * D + 4 * c);
      const float p0 = q[i].x * (kx.x + kt.x), p1 = q[i].y * (kx.y + kt.y);
      const float p2 = q[i].z * (kx.z + kt.z), p3 = q[i].w * (kx.w + kt.w);
      if (hm[i].first == hm[i].last) {
        const float s4 = (p0 + p1) + (p2 + p3);
#pragma unroll
        for (int h = 0; h < H; ++h) part[h] += (hm[i].first == h) ? s4 : 0.f;
      } else {
#pragma unroll
        for (int h = 0; h < H; ++h) {
          part[h] += (hm[i].hid[0] == h) ? p0 : 0.f;
          part[h] += (hm[i].hid[1] == h) ? p1 : 0.f;
          part[h] += (hm[i].hid[2] == h) ? p2 : 0.f;
          part[h] += (hm[i].hid[3] == h) ? p3 : 0.f;
        }
      }
    }
    float mine = 0.f;
#pragma unroll
    for (int h = 0; h < H; ++h) {
      float s = part[h];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      mx[h] = fmaxf(mx[h], s);
      if (lane == h) mine = s;
    }
    if (lane < H) score[(int64_t)p * H + lane] = mine;
  }
  __syncwarp();

  // pass 2: exp(s - max) and the per-head sum.  Lane l owns head l % H (32 % H == 0).
  const int deg = end - beg;
  const int myh = lane % H;
  float mymax = 0.f;
#pragma unroll
  for (int h = 0; h < H; ++h)
    if (myh == h) mymax = mx[h];
  float sum = 0.f;
  float* sc = score + (int64_t)beg * H;
  for (int j = lane; j < deg * H; j += 32) {
    const float ex = expf(sc[j] - mymax);
    sc[j] = ex;
    sum += ex;
  }
#pragma unroll
  for (int o = 16; o >= H; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  // pass 3: normalise (denominator + 1e-16 as torch_geometric.utils.softmax), rescale by out-degree
  const float degf = (float)deg;
  float* al = alpha + (int64_t)beg * H;
  for (int j = lane; j < deg * H; j += 32) {
    const float a = sc[j] / (sum + 1e-16f);
    al[j] = a * degf;
    if (alpha_out != nullptr) alpha_out[(int64_t)perm_src[beg + j / H] * H + myh] = a;
  }
}

template <int H, int CH>
__global__ void __launch_bounds__(256) mp_aggregate_kernel(int64_t N, int D, const int32_t* __restrict__ rowptr_tgt,
                                                           const int32_t* __restrict__ csr_tgt_src,
                                                           const int32_t* __restrict__ csr_tgt_combo,
                                                           const int32_t* __restrict__ csr_tgt_apos,
                                                           const float* __restrict__ qkm, const float* __restrict__ me,
                                                           const float* __restrict__ alpha, float* __restrict__ aggr) {
  const int lane = threadIdx.x & 31;
  const int64_t v = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (v >= N) return;
  const int d = D / H;
  const int ld = 3 * D;
  float4 acc[CH];
  HeadMap hm[CH];
  bool valid[CH];
#pragma unroll
  for (int i = 0; i < CH; ++i) {
    const int c = lane + 32 * i;
    valid[i] = 4 * c < D;
    hm[i] = head_map(c, d);
    acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const int beg = rowptr_tgt[v], end = rowptr_tgt[v + 1];
  for (int p = beg; p < end; ++p) {
    const int s = csr_tgt_src[p];
    const int cb = csr_tgt_combo[p];
    const float* ap = alpha + (int64_t)csr_tgt_apos[p] * H;
#pragma unroll
    for (int i = 0; i < CH; ++i) {
      if (!valid[i]) continue;
      const int c = lane + 32 * i;
      const float4 mxv = ld4(qkm + (int64_t)s * ld + 2 * D + 4 * c);
      const float4 mt = ld4(me + (int64_t)cb * D + 4 * c);
      float w0, w1, w2, w3;
      if (hm[i].first == hm[i].last) {
        w0 = w1 = w2 = w3 = ap[hm[i].first];
      } else {
        w0 = ap[hm[i].hid[0]]; w1 = ap[hm[i].hid[1]]; w2 = ap[hm[i].hid[2]]; w3 = ap[hm[i].hid[3]];
      }
      acc[i].x += (mxv.x + mt.x) * w0;
      acc[i].y += (mxv.y + mt.y) * w1;
      acc[i].z += (mxv.z + mt.z) * w2;
      acc[i].w += (mxv.w + mt.w) * w3;
    }
  }
#pragma unroll
  for (int i = 0; i < CH; ++i) {
    if (!valid[i]) continue;
    *reinterpret_cast<float4*>(aggr + v * D + 4 * (lane + 32 * i)) = acc[i];
  }
}

template <int H, int CH>
int32_t launch_hc(const qagnn_shape& s, const int32_t* base, const qagnn_prep_layout& pl, const float* qkm,
                  const float* ke, const float* me, float* score, float* alpha, float* aggr, float* alpha_out,
                  cudaStream_t st) {
  auto I = [&](size_t off) { return (const int32_t*)((const char*)base + off); };
  const int block = 256;
  const unsigned grid = (unsigned)((s.N * 32 + block - 1) / block);
  mp_scores_kernel<H, CH><<<grid, block, 0, st>>>(s.N, s.D, I(pl.rowptr_src), I(pl.csr_src_tgt), I(pl.csr_src_combo),
                                                  I(pl.perm_src), qkm, ke, score, alpha, alpha_out);
  QAGNN_CHECK_LAUNCH();
  mp_aggregate_kernel<H, CH><<<grid, block, 0, st>>>(s.N, s.D, I(pl.rowptr_tgt), I(pl.csr_tgt_src),
                                                     I(pl.csr_tgt_combo), I(pl.csr_tgt_apos), qkm, me, alpha, aggr);
  QAGNN_CHECK_LAUNCH();
  return QAGNN_OK;
}

template <int H>
int32_t launch_h(const qagnn_shape& s, const int32_t* base, const qagnn_prep_layout& pl, const float* qkm,
                 const float* ke, const float* me, float* score, float* alpha, float* aggr, float* alpha_out,
                 cudaStream_t st) {
  const int ch = (s.D + 127) / 128;
  if (ch <= 1) return launch_hc<H, 1>(s, base, pl, qkm, ke, me, score, alpha, aggr, alpha_out, st);
  if (ch <= 2) return launch_hc<H, 2>(s, base, pl, qkm, ke, me, score, alpha, aggr, alpha_out, st);
  if (ch <= 4) return launch_hc<H, 4>(s, base, pl, qkm, ke, me, score, alpha, aggr, alpha_out, st);
  if (ch <= 8) return launch_hc<H, 8>(s, base, pl, qkm, ke, me, score, alpha, aggr, alpha_out, st);
  return QAGNN_ERR_UNSUPPORTED;
}

}  // namespace

bool basic_mp_supported(const qagnn_shape& s) {
  return s.D % 4 == 0 && s.D <= 1024 && (s.H == 1 || s.H == 2 || s.H == 4 || s.H == 8 || s.H == 16);
}

int32_t launch_message_passing(const qagnn_shape& s, const int32_t* prep_base, const qagnn_prep_layout& pl,
                               const float* qkm, const float* ke, const float* me, float* score, float* alpha,
                               float* aggr, float* alpha_out, cudaStream_t st) {
  if (!basic_mp_supported(s)) return QAGNN_ERR_UNSUPPORTED;
  switch (s.H) {
    case 1: return launch_h<1>(s, prep_base, pl, qkm, ke, me, score, alpha, aggr, alpha_out, st);
    case 2: return launch_h<2>(s, prep_base, pl, qkm, ke, me, score, alpha, aggr, alpha_out, st);
    case 4: return launch_h<4>(s, prep_base, pl, qkm, ke, me, score, alpha, aggr, alpha_out, st);
    case 8: return launch_h<8>(s, prep_base, pl, qkm, ke, me, score, alpha, aggr, alpha_out, st);
    case 16: return launch_h<16>(s, prep_base, pl, qkm, ke, me, score, alpha, aggr, alpha_out, st);
    default: return QAGNN_ERR_UNSUPPORTED;
  }
}

}  // namespace qagnn
