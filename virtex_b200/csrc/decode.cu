// Autoregressive beam-search decoding: single-query attention over a KV cache, the fused beam-selection step and the
// history / cache-index reorder.  Reference semantics: virtex/models/captioning.py:144-213 (decoding_step) and
// virtex/utils/beam_search.py (AutoRegressiveBeamSearch.search); the reference recomputes the whole prefix every step,
// here each step embeds only the newest token and attends over cached keys / values.
#include <cooperative_groups.h>

#include "select.cuh"
#include "vtx_common.cuh"
#include "../../include/virtex_b200.h"

namespace vtx {

constexpr int kDecAttnWarps = 8;   // one warp per (row, head)
constexpr int kDecMaxKeys = 64;    // two keys per lane
constexpr int kBeamThreads = 256;  // one block per row
constexpr int kBeamMaxK = 16;      // per-row candidates (per_node, or beam at the first step)
constexpr int kBeamMaxIn = 8;      // beams per image = blocks per cluster (the portable cluster size)
static_assert(kBeamMaxIn * kBeamMaxK <= 4 * 32, "the image merge holds 4 candidates per lane");

// One warp per (row, head), head_dim 64.  Key j of row r lives at k + phys * row_stride + j * pos_stride (v alike),
// phys = r / group for j < Tk - 1 when table is NULL, table[r * ldt + j] otherwise; the newest key (j = Tk - 1) of a
// table-indexed row is always the row's own slot.  Lane l scores keys l and l + 32 with the full 64-dim q; the output
// pass gives each lane two dims and broadcasts the probabilities through shuffles.  fp32 softmax, bf16 output.
__global__ void __launch_bounds__(32 * kDecAttnWarps)
decode_attn_kernel(const __nv_bfloat16* __restrict__ q, long long ldq, const __nv_bfloat16* __restrict__ k,
                   const __nv_bfloat16* __restrict__ v, long long row_stride, long long pos_stride,
                   const int* __restrict__ table, int ldt, int group, __nv_bfloat16* __restrict__ out, long long ldo,
                   int rows, int heads, int Tk) {
  VTX_PDL_TRIGGER();
  const int lane = threadIdx.x & 31;
  const long long unit = (long long)blockIdx.x * kDecAttnWarps + (threadIdx.x >> 5);
  if (unit >= (long long)rows * heads) return;
  const int r = (int)(unit / heads), h = (int)(unit % heads);
  float qf[64];
  const bf16x8* qp = reinterpret_cast<const bf16x8*>(q + (long long)r * ldq + h * 64);
#pragma unroll
  for (int c = 0; c < 8; ++c) unpack8(qp[c], qf + 8 * c);
  auto key_base = [&](int j) -> long long {
    int phys;
    if (table == nullptr) phys = r / group;
    else phys = (j == Tk - 1) ? r : table[(long long)r * ldt + j];
    return (long long)phys * row_stride + (long long)j * pos_stride + h * 64;
  };
  float s[2];
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int j = lane + 32 * i;
    s[i] = -INFINITY;
    if (j < Tk) {
      const bf16x8* kp = reinterpret_cast<const bf16x8*>(k + key_base(j));
      float acc = 0.f;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        float kf[8];
        unpack8(kp[c], kf);
#pragma unroll
        for (int e = 0; e < 8; ++e) acc = fmaf(qf[8 * c + e], kf[e], acc);
      }
      s[i] = acc * 0.125f;  // 1/sqrt(64)
    }
  }
  const float m = warp_max(fmaxf(s[0], s[1]));
  float pexp[2];
#pragma unroll
  for (int i = 0; i < 2; ++i) pexp[i] = (lane + 32 * i < Tk) ? expf(s[i] - m) : 0.f;
  const float inv = 1.f / warp_sum(pexp[0] + pexp[1]);
  float o0 = 0.f, o1 = 0.f;
#pragma unroll 8
  for (int j = 0; j < Tk; ++j) {  // unrolled: eight value rows in flight per lane
    const float pj = __shfl_sync(0xffffffffu, j < 32 ? pexp[0] : pexp[1], j & 31);
    const __nv_bfloat162 vv = *reinterpret_cast<const __nv_bfloat162*>(v + key_base(j) + 2 * lane);
    const float2 vf = __bfloat1622float2(vv);
    o0 = fmaf(pj, vf.x, o0);
    o1 = fmaf(pj, vf.y, o1);
  }
  *reinterpret_cast<__nv_bfloat162*>(out + (long long)r * ldo + h * 64 + 2 * lane) =
      __floats2bfloat162_rn(o0 * inv, o1 * inv);
}

// One block per row, one thread-block cluster per image (cluster size beam_in).  Each block: log_softmax of its row
// (lp = (x - max) - log(sum exp(x - max))), the repetition penalty (lp of the row's last token := -10000), EOS forcing
// (a row whose last token is EOS scores 0 at EOS and -inf elsewhere, its logits are not read) and the row's top
// per_node, each plus the row's running score, into its shared memory.  Block 0 of the cluster then reads the
// beam_in * per_node candidates of the image through distributed shared memory (candidate index = beam * per_node +
// rank) and keeps the top beam_out.  last == NULL (first step): no penalty, no forcing, running scores 0.
__global__ void __launch_bounds__(kBeamThreads)
beam_step_kernel(const float* __restrict__ logits, long long ldl, int V, int beam_in, int per_node, int beam_out,
                 int eos, const long long* __restrict__ last, const float* __restrict__ scores_in,
                 long long* __restrict__ tokens, long long* __restrict__ parents, float* __restrict__ scores_out,
                 int* __restrict__ ended) {
  VTX_PDL_TRIGGER();
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  __shared__ float red_v[32];
  __shared__ int red_i[32];
  __shared__ float cv[kBeamMaxK];
  __shared__ int ct[kBeamMaxK];
  const long long row = blockIdx.x;
  const int img = (int)(row / beam_in);
  const long long lt = last ? last[row] : -1;
  const float base = scores_in ? scores_in[row] : 0.f;
  if (lt == eos) {  // ended beam: EOS at 0, then the lowest non-EOS ids at -inf (the tie order of -inf)
    if (threadIdx.x == 0) {
      int tok = 0;
      for (int r = 0; r < per_node; ++r) {
        if (r == 0) { cv[0] = 0.f + base; ct[0] = eos; continue; }
        if (tok == eos) ++tok;
        cv[r] = -INFINITY + base; ct[r] = tok++;
      }
    }
  } else {
    const float* x = logits + row * ldl;
    float m = -INFINITY;
    for (int i = threadIdx.x; i < V; i += blockDim.x) m = fmaxf(m, x[i]);
    int dummy = 0;
    block_best(m, dummy, red_v, red_i);  // a NaN logit makes the sum, hence every lp, NaN, as in torch's log_softmax
    float s = 0.f;
    for (int i = threadIdx.x; i < V; i += blockDim.x) s += expf(x[i] - m);
    s = warp_sum(s);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red_v[threadIdx.x >> 5] = s;
    __syncthreads();
    s = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red_v[w];  // same order in every thread
    const float ls = logf(s);
    // per-thread sorted top-per_node of its strided slice
    float tv[kBeamMaxK];
    int ti[kBeamMaxK];
#pragma unroll
    for (int r = 0; r < kBeamMaxK; ++r) { tv[r] = -INFINITY; ti[r] = 0x7fffffff; }
    float thr_v = -INFINITY;  // tv[per_node - 1], kept apart so that the lists are never indexed dynamically
    int thr_i = 0x7fffffff;
    for (int i = threadIdx.x; i < V; i += blockDim.x) {
      float lp = (x[i] - m) - ls;
      if (i == lt) lp = -10000.f;
      if (!rank_better(lp, i, thr_v, thr_i)) continue;
      // insert, keeping the list sorted (unrolled so the arrays stay in registers)
      float cvv = lp;
      int cii = i;
#pragma unroll
      for (int r = 0; r < kBeamMaxK; ++r) {
        if (r < per_node && rank_better(cvv, cii, tv[r], ti[r])) {
          const float sv = tv[r]; const int si = ti[r];
          tv[r] = cvv; ti[r] = cii; cvv = sv; cii = si;
        }
        if (r == per_node - 1) { thr_v = tv[r]; thr_i = ti[r]; }
      }
    }
    // block merge: per_node rounds, the winning thread pops its head
    for (int r = 0; r < per_node; ++r) {
      float bv = tv[0];
      int bi = ti[0];
      block_best(bv, bi, red_v, red_i);
      if (ti[0] == bi && bi != 0x7fffffff) {
#pragma unroll
        for (int q = 0; q + 1 < kBeamMaxK; ++q) { tv[q] = tv[q + 1]; ti[q] = ti[q + 1]; }
        tv[kBeamMaxK - 1] = -INFINITY; ti[kBeamMaxK - 1] = 0x7fffffff;
      }
      if (threadIdx.x == 0) { cv[r] = bv + base; ct[r] = bi; }
    }
  }
  cluster.sync();  // every row's candidates are in its block's shared memory
  // image merge by one warp of block 0 (beam_in * per_node <= 8 * 16 candidates, beam_out rounds)
  if (cluster.block_rank() == 0 && threadIdx.x < 32) {
    const int nc = beam_in * per_node;
    float mv[4];
    int mt[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {  // lane l holds candidates l, l + 32, l + 64, l + 96
      const int c = threadIdx.x + 32 * k;
      mv[k] = -INFINITY; mt[k] = -1;
      if (c < nc) {
        const int b = c / per_node, r = c % per_node;
        mv[k] = cluster.map_shared_rank(cv, b)[r];
        mt[k] = cluster.map_shared_rank(ct, b)[r];
      }
    }
    bool live = false;
    for (int r = 0; r < beam_out; ++r) {
      float bv = -INFINITY;
      int bi = 0x7fffffff;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int c = threadIdx.x + 32 * k;
        if (mt[k] >= 0 && rank_better(mv[k], c, bv, bi)) { bv = mv[k]; bi = c; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (rank_better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
      }
      int tok = -1;
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (threadIdx.x + 32 * k == bi) { tok = mt[k]; mt[k] = -1; }  // the owner lane hands out and retires it
      tok = __reduce_max_sync(0xffffffffu, tok);
      if (threadIdx.x == 0) {
        const long long orow = (long long)img * beam_out + r;
        tokens[orow] = tok;
        parents[orow] = (long long)img * beam_in + bi / per_node;
        scores_out[orow] = bv;
      }
      live |= tok != eos;
    }
    if (threadIdx.x == 0 && live && ended) *ended = 0;
  }
  cluster.sync();  // keep every block's shared memory alive until block 0 has read it
}

// out_hist[r, :n_hist] = in_hist[parent[r], :n_hist], out_hist[r, n_hist] = tokens[r];
// out_table[r, j] = in_table[parent[r], j] for j < n_tab - 1, out_table[r, n_tab - 1] = parent[r].
__global__ void beam_reorder_kernel(const long long* __restrict__ parents, const long long* __restrict__ tokens,
                                    const long long* __restrict__ in_hist, long long* __restrict__ out_hist, int ldh,
                                    int n_hist, const int* __restrict__ in_table, int* __restrict__ out_table, int ldt,
                                    int n_tab, int rows) {
  VTX_PDL_TRIGGER();
  const int r = blockIdx.x * blockDim.y + threadIdx.y;
  if (r >= rows) return;
  const long long p = parents[r];
  for (int j = threadIdx.x; j <= n_hist; j += blockDim.x)
    out_hist[(long long)r * ldh + j] = j < n_hist ? in_hist[p * ldh + j] : tokens[r];
  if (out_table)
    for (int j = threadIdx.x; j < n_tab; j += blockDim.x)
      out_table[(long long)r * ldt + j] = j + 1 < n_tab ? in_table[p * ldt + j] : (int)p;
}

}  // namespace vtx

using namespace vtx;
#define STREAM reinterpret_cast<cudaStream_t>(stream)
#define REQ(cond, msg) \
  if (!(cond)) return set_error(VTX_EINVAL, "%s: %s", __func__, msg)

extern "C" int vtx_decode_attn(const void* q, int64_t ldq, const void* k, const void* v, int64_t row_stride,
                               int64_t pos_stride, const int32_t* table, int ldt, int group, void* out, int64_t ldo,
                               int rows, int heads, int Tk, int cache_len, void* stream) {
  REQ(q && k && v && out && rows >= 0 && heads > 0 && group > 0, "bad arguments");
  REQ((heads * 64) % 128 == 0, "H = heads * 64 must be a multiple of 128");
  REQ(Tk >= 1 && Tk <= cache_len && cache_len <= kDecMaxKeys, "need 1 <= Tk <= cache_len <= 64");
  REQ(!table || ldt >= Tk - 1, "table narrower than the cache");
  REQ(ldq % 8 == 0 && row_stride % 8 == 0 && pos_stride % 8 == 0 && ldo % 2 == 0, "misaligned strides");
  if (rows == 0) return VTX_OK;
  const long long units = (long long)rows * heads;
  decode_attn_kernel<<<(unsigned)((units + kDecAttnWarps - 1) / kDecAttnWarps), 32 * kDecAttnWarps, 0, STREAM>>>(
      (const __nv_bfloat16*)q, ldq, (const __nv_bfloat16*)k, (const __nv_bfloat16*)v, row_stride, pos_stride, table, ldt,
      group, (__nv_bfloat16*)out, ldo, rows, heads, Tk);
  return check_launch("decode_attn");
}

extern "C" int vtx_beam_step(const float* logits, int64_t ldl, int V, int images, int beam_in, int per_node,
                             int beam_out, int eos, const int64_t* last, const float* scores_in, int64_t* tokens,
                             int64_t* parents, float* scores_out, int32_t* ended, void* stream) {
  REQ(logits && tokens && parents && scores_out && images >= 0, "bad arguments");
  REQ(V >= 1 && ldl >= V, "need 1 <= V <= ldl");
  REQ(per_node >= 1 && per_node <= kBeamMaxK && per_node <= V, "need 1 <= per_node <= min(16, V)");
  REQ(beam_in >= 1 && beam_out >= 1 && beam_out <= beam_in * per_node, "need 1 <= beam_out <= beam_in * per_node");
  REQ(beam_in <= kBeamMaxIn, "beam_in exceeds the 8 blocks of one cluster");
  REQ(eos >= 0 && eos < V, "eos outside the vocabulary");
  // nonzero ("every beam ended") until a block finds a live beam and stores 0
  if (ended && cudaMemsetAsync(ended, 1, sizeof(int32_t), STREAM) != cudaSuccess)
    return set_error(VTX_ECUDA, "beam_step: cannot reset the ended flag");
  if (images == 0) return VTX_OK;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(images * beam_in));
  cfg.blockDim = dim3(kBeamThreads);
  cfg.stream = STREAM;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)beam_in;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  const cudaError_t err = cudaLaunchKernelEx(&cfg, beam_step_kernel, (const float*)logits, (long long)ldl, V, beam_in,
                                             per_node, beam_out, eos, (const long long*)last, scores_in,
                                             (long long*)tokens, (long long*)parents, scores_out, (int*)ended);
  if (err != cudaSuccess) return set_error(VTX_ECUDA, "beam_step: %s", cudaGetErrorString(err));
  return check_launch("beam_step");
}

extern "C" int vtx_beam_reorder(const int64_t* parents, const int64_t* tokens, const int64_t* in_hist,
                                int64_t* out_hist, int ldh, int n_hist, const int32_t* in_table, int32_t* out_table,
                                int ldt, int n_tab, int rows, void* stream) {
  REQ(parents && tokens && out_hist && rows >= 0 && n_hist >= 0 && ldh > n_hist && (n_hist == 0 || in_hist),
      "bad history arguments");
  REQ(!out_table || ((in_table || n_tab <= 1) && n_tab >= 1 && n_tab <= ldt), "bad table arguments");
  REQ(in_hist != out_hist && (!out_table || in_table != out_table), "in-place reorder is not supported");
  if (rows == 0) return VTX_OK;
  const dim3 block(32, 8);
  beam_reorder_kernel<<<(rows + 7) / 8, block, 0, STREAM>>>((const long long*)parents, (const long long*)tokens,
                                                            (const long long*)in_hist, (long long*)out_hist, ldh,
                                                            n_hist, in_table, out_table, ldt, n_tab, rows);
  return check_launch("beam_reorder");
}
