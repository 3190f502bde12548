// Classification pretext heads: global average pooling of the backbone output (forward and backward), the K-hot
// cross entropy of the multi-label objective and the row top-k of its eval predictions.  Reference semantics:
// virtex/modules/textual_heads.py:46-95 (LinearTextualHead: mean over h*w, then nn.Linear) and
// virtex/models/classification.py:12-102 (log_softmax, the mean log-probability over the unique, non-ignored labels
// of each image, top-10).  The linear layer itself is a vtx_gemm.
#include "select.cuh"
#include "vtx_common.cuh"
#include "../../include/virtex_b200.h"

namespace vtx {

constexpr int kPoolLanes = 8;         // row lanes of the pooling block (one per warp)
constexpr int kKhotMaxV = 65536;      // label bitmap: 2048 words = 8 KB of shared memory
constexpr int kKhotMaxL = 1024;
constexpr int kKhotThreads = 256;
constexpr int kTopkMaxK = 16;
constexpr int kTopkThreads = 256;

// pooled[b, c] = bf16(sum_s feat[b * S + s, c] / S), fp32 accumulation.  Block (32 channel groups of 8) x (8 row
// lanes): one image, 256 channels; each lane walks every eighth row with 16-byte loads, the lanes are summed in
// shared memory in a fixed order.
__global__ void __launch_bounds__(32 * kPoolLanes) avgpool_fwd_kernel(const __nv_bfloat16* __restrict__ feat,
                                                                     __nv_bfloat16* __restrict__ pooled, int S, int C) {
  VTX_PDL_TRIGGER();
  __shared__ float red[kPoolLanes][32 * 8];
  const int cg = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int g = blockIdx.x * 32 + cg;  // 8-channel group
  const int b = blockIdx.y;
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  if (g * 8 < C) {
    const __nv_bfloat16* xp = feat + (long long)b * S * C + g * 8;
    int s = rl;
    for (; s + 3 * kPoolLanes < S; s += 4 * kPoolLanes) {  // four independent 16-byte loads in flight
      bf16x8 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = *reinterpret_cast<const bf16x8*>(xp + (long long)(s + u * kPoolLanes) * C);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        float f[8];
        unpack8(v[u], f);
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] += f[j];
      }
    }
    for (; s < S; s += kPoolLanes) {
      float f[8];
      unpack8(*reinterpret_cast<const bf16x8*>(xp + (long long)s * C), f);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += f[j];
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) red[rl][cg * 8 + j] = acc[j];
  __syncthreads();
  if (rl == 0 && g * 8 < C) {
    float t[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float a = 0.f;
#pragma unroll
      for (int l = 0; l < kPoolLanes; ++l) a += red[l][cg * 8 + j];
      t[j] = a / (float)S;
    }
    *reinterpret_cast<bf16x8*>(pooled + (long long)b * C + g * 8) = pack8(t);
  }
}

// dfeat[b * S + s, c] = bf16(dpooled[b, c] / S): one 16-byte store of 8 channels per thread.
__global__ void avgpool_bwd_kernel(const float* __restrict__ dpooled, __nv_bfloat16* __restrict__ dfeat, int S, int C,
                                   long long total8) {
  VTX_PDL_TRIGGER();
  const int G = C / 8;
  const float fs = (float)S;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < total8) {
    const long long row = i / G;
    const int g = (int)(i - row * G);
    const long long b = row / S;
    const float4* src = reinterpret_cast<const float4*>(dpooled + b * C + g * 8);
    const float4 a = __ldg(src), c = __ldg(src + 1);
    const float f[8] = {a.x / fs, a.y / fs, a.z / fs, a.w / fs, c.x / fs, c.y / fs, c.z / fs, c.w / fs};
    *reinterpret_cast<bf16x8*>(dfeat + row * C + g * 8) = pack8(f);
  }
}

// Block sum / max with a fixed reduction order (the same result in every thread).
__device__ __forceinline__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float t = 0.f;
  for (int w = 0; w < nw; ++w) t += red[w];
  return t;
}
__device__ __forceinline__ float block_max(float v, float* red) {
  v = warp_max(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float t = -INFINITY;
  for (int w = 0; w < nw; ++w) t = fmaxf(t, red[w]);
  return t;
}

// One block per image b of fp32 logits [B, ldl].  The label set is a V-bit bitmap in shared memory: every id of
// labels[b, :L] inside [0, V) sets its bit (a duplicate sets it again), then every id of the ignore list clears it;
// ids outside [0, V) are never used as an address.  K = |set|,
//     loss += (lse - (1/K) sum_{v in set} z_v) / B        (K = 0: NaN, the mean of nothing in the reference)
//     dlogits[b, v] = bf16((softmax_v - [v in set] / K) / B)     (K = 0: a zero row, what autograd gives there)
__global__ void __launch_bounds__(kKhotThreads) khot_xent_kernel(const float* __restrict__ logits, long long ldl,
                                                                 const long long* __restrict__ labels, int L,
                                                                 const long long* __restrict__ ignore, int n_ignore,
                                                                 int B, int V, float* __restrict__ loss,
                                                                 __nv_bfloat16* __restrict__ dlogits, long long lddl) {
  VTX_PDL_TRIGGER();
  __shared__ uint32_t bits[kKhotMaxV / 32];
  __shared__ float red[32];
  const int b = blockIdx.x;
  const int nwords = (V + 31) >> 5;
  for (int w = threadIdx.x; w < nwords; w += blockDim.x) bits[w] = 0u;
  __syncthreads();
  for (int t = threadIdx.x; t < L; t += blockDim.x) {
    const long long id = labels[(long long)b * L + t];
    if (id >= 0 && id < V) atomicOr(&bits[id >> 5], 1u << (id & 31));
  }
  __syncthreads();
  for (int t = threadIdx.x; t < n_ignore; t += blockDim.x) {
    const long long id = ignore[t];
    if (id >= 0 && id < V) atomicAnd(&bits[id >> 5], ~(1u << (id & 31)));
  }
  __syncthreads();
  const float* x = logits + (long long)b * ldl;
  // K and the sum of the set's logits
  float kf = 0.f, zs = 0.f;
  for (int w = threadIdx.x; w < nwords; w += blockDim.x) {
    uint32_t m = bits[w];
    kf += (float)__popc(m);
    while (m) {
      const int j = __ffs(m) - 1;
      m &= m - 1;
      zs += x[w * 32 + j];
    }
  }
  const float K = block_sum(kf, red);
  const float zsum = block_sum(zs, red);
  // log-sum-exp over the row (16-byte loads: ldl % 4 == 0)
  const int V4 = V >> 2;
  const float4* x4 = reinterpret_cast<const float4*>(x);
  float mx = -INFINITY;
  for (int i = threadIdx.x; i < V4; i += blockDim.x) {
    const float4 q = x4[i];
    mx = fmaxf(mx, fmaxf(fmaxf(q.x, q.y), fmaxf(q.z, q.w)));
  }
  for (int i = 4 * V4 + threadIdx.x; i < V; i += blockDim.x) mx = fmaxf(mx, x[i]);
  mx = block_max(mx, red);
  float s = 0.f;
  for (int i = threadIdx.x; i < V4; i += blockDim.x) {
    const float4 q = x4[i];
    s += expf(q.x - mx) + expf(q.y - mx) + expf(q.z - mx) + expf(q.w - mx);
  }
  for (int i = 4 * V4 + threadIdx.x; i < V; i += blockDim.x) s += expf(x[i] - mx);
  s = block_sum(s, red);
  const float lse = mx + logf(s);
  if (threadIdx.x == 0) {
    const float lb = K > 0.f ? lse - zsum / K : __int_as_float(0x7fffffff);
    atomicAdd(loss, lb / (float)B);
  }
  if (dlogits == nullptr) return;
  __nv_bfloat16* d = dlogits + (long long)b * lddl;
  const float inv_s = 1.f / s, inv_k = K > 0.f ? 1.f / K : 0.f, inv_b = 1.f / (float)B;
  const bool live = K > 0.f;
  auto grad = [&](int v) -> float {
    if (!live) return 0.f;
    const float ind = (bits[v >> 5] >> (v & 31)) & 1u ? inv_k : 0.f;
    return (expf(x[v] - mx) * inv_s - ind) * inv_b;
  };
  const int V8 = V >> 3;
  for (int i = threadIdx.x; i < V8; i += blockDim.x) {
    float f[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = grad(8 * i + j);
    *reinterpret_cast<bf16x8*>(d + 8 * i) = pack8(f);
  }
  for (int v = 8 * V8 + threadIdx.x; v < V; v += blockDim.x) d[v] = f2bf(grad(v));
}

// Top k (k <= 16) of each fp32 row, in rank_better order.  One block per row: each thread keeps a sorted list of the
// best k of its strided slice, then k block-wide rounds pop the overall best head.
__global__ void __launch_bounds__(kTopkThreads) topk_rows_kernel(const float* __restrict__ X, long long ld, int N, int k,
                                                                 long long* __restrict__ out) {
  VTX_PDL_TRIGGER();
  __shared__ float red_v[32];
  __shared__ int red_i[32];
  const float* x = X + (long long)blockIdx.x * ld;
  float tv[kTopkMaxK];
  int ti[kTopkMaxK];
#pragma unroll
  for (int r = 0; r < kTopkMaxK; ++r) { tv[r] = -INFINITY; ti[r] = 0x7fffffff; }
  float thr_v = -INFINITY;  // tv[k - 1], kept apart so that the lists are never indexed dynamically
  int thr_i = 0x7fffffff;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const float v = x[i];
    if (!rank_better(v, i, thr_v, thr_i)) continue;
    float cv = v;
    int ci = i;
#pragma unroll
    for (int r = 0; r < kTopkMaxK; ++r) {
      if (r < k && rank_better(cv, ci, tv[r], ti[r])) {
        const float sv = tv[r]; const int si = ti[r];
        tv[r] = cv; ti[r] = ci; cv = sv; ci = si;
      }
      if (r == k - 1) { thr_v = tv[r]; thr_i = ti[r]; }
    }
  }
  for (int r = 0; r < k; ++r) {
    float bv = tv[0];
    int bi = ti[0];
    block_best(bv, bi, red_v, red_i);
    if (ti[0] == bi && bi != 0x7fffffff) {
#pragma unroll
      for (int q = 0; q + 1 < kTopkMaxK; ++q) { tv[q] = tv[q + 1]; ti[q] = ti[q + 1]; }
      tv[kTopkMaxK - 1] = -INFINITY; ti[kTopkMaxK - 1] = 0x7fffffff;
    }
    if (threadIdx.x == 0) out[(long long)blockIdx.x * k + r] = bi;
  }
}

}  // namespace vtx

using namespace vtx;
#define STREAM reinterpret_cast<cudaStream_t>(stream)
#define REQ(cond, msg) \
  if (!(cond)) return set_error(VTX_EINVAL, "%s: %s", __func__, msg)
#define ALIGNED16(p) ((reinterpret_cast<uintptr_t>(p) & 15) == 0)

extern "C" int vtx_avgpool_fwd(const void* feat, void* pooled, int B, int S, int C, void* stream) {
  REQ(feat && pooled && B >= 0, "bad arguments");
  REQ(S >= 1 && C > 0 && C % 8 == 0, "need S >= 1 and C % 8 == 0");
  REQ(ALIGNED16(feat) && ALIGNED16(pooled), "pointers must be 16-byte aligned");
  if (B == 0) return VTX_OK;
  const dim3 grid((unsigned)((C / 8 + 31) / 32), (unsigned)B);
  avgpool_fwd_kernel<<<grid, 32 * kPoolLanes, 0, STREAM>>>((const __nv_bfloat16*)feat, (__nv_bfloat16*)pooled, S, C);
  return check_launch("avgpool_fwd");
}

extern "C" int vtx_avgpool_bwd(const float* dpooled, void* dfeat, int B, int S, int C, void* stream) {
  REQ(dpooled && dfeat && B >= 0, "bad arguments");
  REQ(S >= 1 && C > 0 && C % 8 == 0, "need S >= 1 and C % 8 == 0");
  REQ(ALIGNED16(dpooled) && ALIGNED16(dfeat), "pointers must be 16-byte aligned");
  if (B == 0) return VTX_OK;
  const long long total8 = (long long)B * S * (C / 8);
  REQ(total8 <= (long long)(1u << 31) * 256, "dfeat too large");
  avgpool_bwd_kernel<<<(unsigned)((total8 + 255) / 256), 256, 0, STREAM>>>(dpooled, (__nv_bfloat16*)dfeat, S, C, total8);
  return check_launch("avgpool_bwd");
}

extern "C" int vtx_khot_xent(const float* logits, int64_t ldl, const int64_t* labels, int L, const int64_t* ignore,
                             int n_ignore, int B, int V, float* loss, void* dlogits, int64_t lddl, void* stream) {
  REQ(logits && labels && loss && B >= 0 && n_ignore >= 0 && (n_ignore == 0 || ignore), "bad arguments");
  REQ(V >= 1 && V <= kKhotMaxV, "need 1 <= V <= 65536 (the label bitmap is 8 KB of shared memory)");
  REQ(L >= 0 && L <= kKhotMaxL, "need 0 <= L <= 1024 labels per image");
  REQ(ldl >= V && ldl % 4 == 0 && ALIGNED16(logits), "fp32 logits need ldl >= V, ldl % 4 == 0 (16-byte rows)");
  REQ(!dlogits || (lddl >= V && lddl % 8 == 0 && ALIGNED16(dlogits)),
      "bf16 dlogits need lddl >= V, lddl % 8 == 0 (16-byte rows)");
  if (B == 0) return VTX_OK;
  khot_xent_kernel<<<B, kKhotThreads, 0, STREAM>>>(logits, ldl, (const long long*)labels, L, (const long long*)ignore,
                                                   n_ignore, B, V, loss, (__nv_bfloat16*)dlogits, lddl);
  return check_launch("khot_xent");
}

extern "C" int vtx_topk_rows(const float* X, int64_t ld, int M, int N, int k, int64_t* out, void* stream) {
  REQ(X && out && M >= 0 && N >= 1 && ld >= N, "bad arguments");
  REQ(k >= 1 && k <= kTopkMaxK && k <= N, "need 1 <= k <= min(16, N)");
  if (M == 0) return VTX_OK;
  topk_rows_kernel<<<M, kTopkThreads, 0, STREAM>>>(X, ld, N, k, (long long*)out);
  return check_launch("topk_rows");
}
