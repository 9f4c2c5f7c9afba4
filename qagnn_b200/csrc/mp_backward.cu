// Backward of the message passing of one GATConvE layer (the gradient of modeling/modeling_qagnn.py:442,455-484
// with torch_geometric's propagate / softmax and torch_scatter's scatter, on the node-level factorisation):
//
//   forward   s[e,h]  = Q[src] . (Kx[tgt] + Ke[c])        a = softmax over edges sharing SRC        a' = a * outdeg(src)
//             aggr[v] = sum_{e: tgt = v} a'[e,h] (Mx[src] + Me[c])
//   backward  da'[e,h] = dAggr[tgt,h,:] . (Mx[src,h,:] + Me[c,h,:])            da = outdeg(src) * da'
//             ds[e,h]  = a[e,h] (da[e,h] - sum_{e' in out(src)} a[e',h] da[e',h])                  (softmax)
//             dQ[u]  = sum_{e: src = u} ds (Kx[tgt] + Ke[c])      dMx[u] = sum_{e: src = u} a' dAggr[tgt]
//             dKx[v] = sum_{e: tgt = v} ds Q[src]
//             dKe[c] = sum_{e: combo = c} ds Q[src]                dMe[c] = sum_{e: combo = c} a' dAggr[tgt]
//
// Three kernels over the CSR orders of graph prep (general path: any graph):
//   mp_bwd_source_kernel   one warp per SOURCE node: da', softmax backward, ds (kept by-source), dQ, dMx     no atomics
//   mp_bwd_target_kernel   one warp per TARGET node: dKx                                                    no atomics
//   mp_bwd_table_kernel    one warp per run of 64 edges in COMBO order: register partial sums, one vector
//                          atomic add per (run, combo change) into dKe / dMe — the only atomics, a few thousand adds
#include "common.cuh"

namespace qagnn {

namespace {

struct HeadMap4 {
  int first, last;
  int hid[4];
};
__device__ __forceinline__ HeadMap4 head_map4(int c, int d) {
  HeadMap4 m;
#pragma unroll
  for (int t = 0; t < 4; ++t) m.hid[t] = (4 * c + t) / d;
  m.first = m.hid[0];
  m.last = m.hid[3];
  return m;
}
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }

// per-head partial sums of the 4 products of one float4 chunk
template <int H>
__device__ __forceinline__ void add_parts(float (&part)[H], const HeadMap4& hm, float p0, float p1, float p2, float p3) {
  if (hm.first == hm.last) {
    const float s4 = (p0 + p1) + (p2 + p3);
#pragma unroll
    for (int h = 0; h < H; ++h) part[h] += (hm.first == h) ? s4 : 0.f;
  } else {
#pragma unroll
    for (int h = 0; h < H; ++h) {
      part[h] += (hm.hid[0] == h) ? p0 : 0.f;
      part[h] += (hm.hid[1] == h) ? p1 : 0.f;
      part[h] += (hm.hid[2] == h) ? p2 : 0.f;
      part[h] += (hm.hid[3] == h) ? p3 : 0.f;
    }
  }
}
template <int H>
__device__ __forceinline__ float pick(const float (&w)[H], int h) {
  float r = 0.f;
#pragma unroll
  for (int i = 0; i < H; ++i) r = (h == i) ? w[i] : r;
  return r;
}

template <int H, int CH>
__global__ void __launch_bounds__(256) mp_bwd_source_kernel(int64_t N, int D, const int32_t* __restrict__ rowptr_src,
                                                            const int32_t* __restrict__ csr_src_tgt,
                                                            const int32_t* __restrict__ csr_src_combo,
                                                            const float* __restrict__ qkm, const float* __restrict__ ke,
                                                            const float* __restrict__ me, const float* __restrict__ alpha_s,
                                                            const float* __restrict__ d_aggr, float* __restrict__ ds,
                                                            float* __restrict__ d_qkm) {
  const int lane = threadIdx.x & 31;
  const int64_t u = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (u >= N) return;
  const int d = D / H, ld = 3 * D;
  HeadMap4 hm[CH];
  bool valid[CH];
  float4 mx[CH], dq[CH], dmx[CH];
#pragma unroll
  for (int i = 0; i < CH; ++i) {
    const int c = lane + 32 * i;
    valid[i] = 4 * c < D;
    hm[i] = head_map4(c, d);
    mx[i] = valid[i] ? ld4(qkm + u * ld + 2 * D + 4 * c) : make_float4(0.f, 0.f, 0.f, 0.f);
    dq[i] = dmx[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const int beg = rowptr_src[u], end = rowptr_src[u + 1];
  const float degf = (float)(end - beg), rdeg = 1.f / degf;
  float dot[H];
#pragma unroll
  for (int h = 0; h < H; ++h) dot[h] = 0.f;
  // pass A: da = outdeg * dAggr[tgt] . (Mx[u] + Me[c]) per head, sum_e a da, and dMx[u] += a' dAggr[tgt]
  for (int p = beg; p < end; ++p) {
    const int t = csr_src_tgt[p], cb = csr_src_combo[p];
    float as[H];  // a' of this edge
#pragma unroll
    for (int h = 0; h < H; ++h) as[h] = alpha_s[(int64_t)p * H + h];
    float part[H];
#pragma unroll
    for (int h = 0; h < H; ++h) part[h] = 0.f;
#pragma unroll
    for (int i = 0; i < CH; ++i) {
      if (!valid[i]) continue;
      const int c = lane + 32 * i;
      const float4 g = ld4(d_aggr + (int64_t)t * D + 4 * c);
      const float4 mt = ld4(me + (int64_t)cb * D + 4 * c);
      add_parts<H>(part, hm[i], g.x * (mx[i].x + mt.x), g.y * (mx[i].y + mt.y), g.z * (mx[i].z + mt.z), g.w * (mx[i].w + mt.w));
      dmx[i].x += pick<H>(as, hm[i].hid[0]) * g.x;
      dmx[i].y += pick<H>(as, hm[i].hid[1]) * g.y;
      dmx[i].z += pick<H>(as, hm[i].hid[2]) * g.z;
      dmx[i].w += pick<H>(as, hm[i].hid[3]) * g.w;
    }
    float mine = 0.f;
#pragma unroll
    for (int h = 0; h < H; ++h) {
      float s = part[h];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      const float da = s * degf;
      dot[h] += (as[h] * rdeg) * da;
      if (lane == h) mine = da;
    }
    if (lane < H) ds[(int64_t)p * H + lane] = mine;  // da for now
  }
  __syncwarp();
  // pass B: ds = a (da - dot), dQ[u] += ds (Kx[tgt] + Ke[c])
  for (int p = beg; p < end; ++p) {
    const int t = csr_src_tgt[p], cb = csr_src_combo[p];
    float dsv[H];
#pragma unroll
    for (int h = 0; h < H; ++h) dsv[h] = (alpha_s[(int64_t)p * H + h] * rdeg) * (ds[(int64_t)p * H + h] - dot[h]);
#pragma unroll
    for (int i = 0; i < CH; ++i) {
      if (!valid[i]) continue;
      const int c = lane + 32 * i;
      const float4 kx = ld4(qkm + (int64_t)t * ld + D + 4 * c);
      const float4 kt = ld4(ke + (int64_t)cb * D + 4 * c);
      dq[i].x += pick<H>(dsv, hm[i].hid[0]) * (kx.x + kt.x);
      dq[i].y += pick<H>(dsv, hm[i].hid[1]) * (kx.y + kt.y);
      dq[i].z += pick<H>(dsv, hm[i].hid[2]) * (kx.z + kt.z);
      dq[i].w += pick<H>(dsv, hm[i].hid[3]) * (kx.w + kt.w);
    }
    __syncwarp();  // every lane has read da[p] before it is overwritten
    if (lane < H) {
      float mine = 0.f;
#pragma unroll
      for (int h = 0; h < H; ++h) mine = (lane == h) ? dsv[h] : mine;
      ds[(int64_t)p * H + lane] = mine;
    }
  }
#pragma unroll
  for (int i = 0; i < CH; ++i) {
    if (!valid[i]) continue;
    const int c = lane + 32 * i;
    *reinterpret_cast<float4*>(d_qkm + u * ld + 4 * c) = dq[i];
    *reinterpret_cast<float4*>(d_qkm + u * ld + 2 * D + 4 * c) = dmx[i];
  }
}

template <int H, int CH>
__global__ void __launch_bounds__(256) mp_bwd_target_kernel(int64_t N, int D, const int32_t* __restrict__ rowptr_tgt,
                                                            const int32_t* __restrict__ csr_tgt_src,
                                                            const int32_t* __restrict__ csr_tgt_apos,
                                                            const float* __restrict__ qkm, const float* __restrict__ ds,
                                                            float* __restrict__ d_qkm) {
  const int lane = threadIdx.x & 31;
  const int64_t v = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (v >= N) return;
  const int d = D / H, ld = 3 * D;
  HeadMap4 hm[CH];
  bool valid[CH];
  float4 acc[CH];
#pragma unroll
  for (int i = 0; i < CH; ++i) {
    const int c = lane + 32 * i;
    valid[i] = 4 * c < D;
    hm[i] = head_map4(c, d);
    acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const int beg = rowptr_tgt[v], end = rowptr_tgt[v + 1];
  for (int p = beg; p < end; ++p) {
    const int s = csr_tgt_src[p];
    const float* dp = ds + (int64_t)csr_tgt_apos[p] * H;
    float dsv[H];
#pragma unroll
    for (int h = 0; h < H; ++h) dsv[h] = dp[h];
#pragma unroll
    for (int i = 0; i < CH; ++i) {
      if (!valid[i]) continue;
      const int c = lane + 32 * i;
      const float4 q = ld4(qkm + (int64_t)s * ld + 4 * c);
      acc[i].x += pick<H>(dsv, hm[i].hid[0]) * q.x;
      acc[i].y += pick<H>(dsv, hm[i].hid[1]) * q.y;
      acc[i].z += pick<H>(dsv, hm[i].hid[2]) * q.z;
      acc[i].w += pick<H>(dsv, hm[i].hid[3]) * q.w;
    }
  }
#pragma unroll
  for (int i = 0; i < CH; ++i) {
    if (!valid[i]) continue;
    *reinterpret_cast<float4*>(d_qkm + v * ld + D + 4 * (lane + 32 * i)) = acc[i];
  }
}

constexpr int kTableRun = 64;  // edges per warp in combo order

__device__ __forceinline__ void atomic_add4(float* p, const float4& v) {
  atomicAdd(p, v.x); atomicAdd(p + 1, v.y); atomicAdd(p + 2, v.z); atomicAdd(p + 3, v.w);
}

template <int H, int CH>
__global__ void __launch_bounds__(256) mp_bwd_table_kernel(int64_t Ep, int D, const int32_t* __restrict__ combo_order,
                                                           const int32_t* __restrict__ csr_src_tgt,
                                                           const int32_t* __restrict__ csr_src_combo,
                                                           const int32_t* __restrict__ perm_src,
                                                           const int32_t* __restrict__ src, const float* __restrict__ qkm,
                                                           const float* __restrict__ alpha_s, const float* __restrict__ ds,
                                                           const float* __restrict__ d_aggr, float* __restrict__ d_ke,
                                                           float* __restrict__ d_me) {
  const int lane = threadIdx.x & 31;
  const int64_t w = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t i0 = w * kTableRun;
  if (i0 >= Ep) return;
  const int64_t i1 = min(i0 + (int64_t)kTableRun, Ep);
  const int d = D / H, ld = 3 * D;
  HeadMap4 hm[CH];
  bool valid[CH];
  float4 ak[CH], am[CH];
#pragma unroll
  for (int i = 0; i < CH; ++i) {
    const int c = lane + 32 * i;
    valid[i] = 4 * c < D;
    hm[i] = head_map4(c, d);
    ak[i] = am[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  auto flush = [&](int cb) {
#pragma unroll
    for (int i = 0; i < CH; ++i) {
      if (!valid[i]) continue;
      const int c = lane + 32 * i;
      atomic_add4(d_ke + (int64_t)cb * D + 4 * c, ak[i]);
      atomic_add4(d_me + (int64_t)cb * D + 4 * c, am[i]);
      ak[i] = am[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  int cur = -1;
  for (int64_t i = i0; i < i1; ++i) {
    const int p = combo_order[i];  // by-source position of the i-th edge in combo order
    const int cb = csr_src_combo[p];
    if (cb != cur) {
      if (cur >= 0) flush(cur);
      cur = cb;
    }
    const int t = csr_src_tgt[p], s = src[perm_src[p]];
    float dsv[H], as[H];
#pragma unroll
    for (int h = 0; h < H; ++h) {
      dsv[h] = ds[(int64_t)p * H + h];
      as[h] = alpha_s[(int64_t)p * H + h];
    }
#pragma unroll
    for (int k = 0; k < CH; ++k) {
      if (!valid[k]) continue;
      const int c = lane + 32 * k;
      const float4 q = ld4(qkm + (int64_t)s * ld + 4 * c);
      const float4 g = ld4(d_aggr + (int64_t)t * D + 4 * c);
      ak[k].x += pick<H>(dsv, hm[k].hid[0]) * q.x; am[k].x += pick<H>(as, hm[k].hid[0]) * g.x;
      ak[k].y += pick<H>(dsv, hm[k].hid[1]) * q.y; am[k].y += pick<H>(as, hm[k].hid[1]) * g.y;
      ak[k].z += pick<H>(dsv, hm[k].hid[2]) * q.z; am[k].z += pick<H>(as, hm[k].hid[2]) * g.z;
      ak[k].w += pick<H>(dsv, hm[k].hid[3]) * q.w; am[k].w += pick<H>(as, hm[k].hid[3]) * g.w;
    }
  }
  if (cur >= 0) flush(cur);
}

template <int H, int CH>
int32_t launch_bwd_hc(const qagnn_shape& s, const int32_t* base, const qagnn_prep_layout& pl, const int32_t* combo_order,
                      const float* qkm, const float* ke, const float* me, const float* alpha_s, const float* d_aggr,
                      float* ds, float* d_qkm, float* d_ke, float* d_me, cudaStream_t st) {
  auto I = [&](size_t off) { return (const int32_t*)((const char*)base + off); };
  const int block = 256;
  const unsigned grid = (unsigned)((s.N * 32 + block - 1) / block);
  const int64_t Ep = s.N + s.E;
  const int C = s.R * s.T * s.T + s.T;
  QAGNN_CHECK_CUDA(cudaMemsetAsync(d_ke, 0, (size_t)C * s.D * sizeof(float), st));
  QAGNN_CHECK_CUDA(cudaMemsetAsync(d_me, 0, (size_t)C * s.D * sizeof(float), st));
  mp_bwd_source_kernel<H, CH><<<grid, block, 0, st>>>(s.N, s.D, I(pl.rowptr_src), I(pl.csr_src_tgt), I(pl.csr_src_combo), qkm,
                                                      ke, me, alpha_s, d_aggr, ds, d_qkm);
  QAGNN_CHECK_LAUNCH();
  mp_bwd_target_kernel<H, CH><<<grid, block, 0, st>>>(s.N, s.D, I(pl.rowptr_tgt), I(pl.csr_tgt_src), I(pl.csr_tgt_apos), qkm, ds,
                                                      d_qkm);
  QAGNN_CHECK_LAUNCH();
  const int64_t runs = (Ep + kTableRun - 1) / kTableRun;
  mp_bwd_table_kernel<H, CH><<<(unsigned)((runs * 32 + block - 1) / block), block, 0, st>>>(
      Ep, s.D, combo_order, I(pl.csr_src_tgt), I(pl.csr_src_combo), I(pl.perm_src), I(pl.src), qkm, alpha_s, ds, d_aggr, d_ke,
      d_me);
  QAGNN_CHECK_LAUNCH();
  return QAGNN_OK;
}

template <int H>
int32_t launch_bwd_h(const qagnn_shape& s, const int32_t* base, const qagnn_prep_layout& pl, const int32_t* combo_order,
                     const float* qkm, const float* ke, const float* me, const float* alpha_s, const float* d_aggr, float* ds,
                     float* d_qkm, float* d_ke, float* d_me, cudaStream_t st) {
  const int ch = (s.D + 127) / 128;
  if (ch <= 1) return launch_bwd_hc<H, 1>(s, base, pl, combo_order, qkm, ke, me, alpha_s, d_aggr, ds, d_qkm, d_ke, d_me, st);
  if (ch <= 2) return launch_bwd_hc<H, 2>(s, base, pl, combo_order, qkm, ke, me, alpha_s, d_aggr, ds, d_qkm, d_ke, d_me, st);
  if (ch <= 4) return launch_bwd_hc<H, 4>(s, base, pl, combo_order, qkm, ke, me, alpha_s, d_aggr, ds, d_qkm, d_ke, d_me, st);
  if (ch <= 8) return launch_bwd_hc<H, 8>(s, base, pl, combo_order, qkm, ke, me, alpha_s, d_aggr, ds, d_qkm, d_ke, d_me, st);
  return QAGNN_ERR_UNSUPPORTED;
}

}  // namespace

int32_t launch_message_passing_backward(const qagnn_shape& s, const int32_t* prep_base, const qagnn_prep_layout& pl,
                                        const int32_t* combo_order, const float* qkm, const float* ke, const float* me,
                                        const float* alpha_s, const float* d_aggr, float* ds, float* d_qkm, float* d_ke,
                                        float* d_me, cudaStream_t st) {
  if (!basic_mp_supported(s)) return QAGNN_ERR_UNSUPPORTED;
  switch (s.H) {
    case 1: return launch_bwd_h<1>(s, prep_base, pl, combo_order, qkm, ke, me, alpha_s, d_aggr, ds, d_qkm, d_ke, d_me, st);
    case 2: return launch_bwd_h<2>(s, prep_base, pl, combo_order, qkm, ke, me, alpha_s, d_aggr, ds, d_qkm, d_ke, d_me, st);
    case 4: return launch_bwd_h<4>(s, prep_base, pl, combo_order, qkm, ke, me, alpha_s, d_aggr, ds, d_qkm, d_ke, d_me, st);
    case 8: return launch_bwd_h<8>(s, prep_base, pl, combo_order, qkm, ke, me, alpha_s, d_aggr, ds, d_qkm, d_ke, d_me, st);
    case 16: return launch_bwd_h<16>(s, prep_base, pl, combo_order, qkm, ke, me, alpha_s, d_aggr, ds, d_qkm, d_ke, d_me, st);
    default: return QAGNN_ERR_UNSUPPORTED;
  }
}

}  // namespace qagnn
