// Memory/latency-bound kernels of the TransformerDecoder textual head (everything that is not a GEMM):
// fused embedding (gather + LayerNorm(1e-8) + dropout + pad mask), residual-add + dropout + LayerNorm, multi-head
// attention cores for T<=32 queries / S<=64 keys with the causal + key-padding mask generated from caption_lengths
// (never materialised), exact-erf GELU + dropout, token cross-entropy (fwd + dlogits in place), bias-gradient column
// sums and argmax.  Reference semantics: virtex/modules/embedding.py:46-74, torch/nn/modules/transformer.py:1144-1199,
// torch/nn/functional.py:6244-6690, virtex/models/captioning.py:111-114 (SURVEY.md Appendix C.5-C.11).
// The decoder residual stream is fp32; GEMM operands/outputs are bf16 (the bf16-autocast placement of the reference).
#include "vtx_common.cuh"
#include "../../include/virtex_b200.h"

namespace vtx {

constexpr int kWarpsPerBlock = 4;

// ------------------------------------------------------------------------------------------------ LayerNorm helpers
// one warp per row; two-pass statistics (mean, then centred variance) in fp32
__device__ __forceinline__ void warp_row_stats(const float* row, int H, int lane, float eps, float& mean, float& rstd) {
  float s = 0.f;
  for (int i = lane * 4; i < H; i += 128) {
    const float4 v = *reinterpret_cast<const float4*>(row + i);
    s += v.x + v.y + v.z + v.w;
  }
  mean = warp_sum(s) / H;
  float q = 0.f;
  for (int i = lane * 4; i < H; i += 128) {
    const float4 v = *reinterpret_cast<const float4*>(row + i);
    const float a = v.x - mean, b = v.y - mean, c = v.z - mean, d = v.w - mean;
    q += a * a + b * b + c * c + d * d;
  }
  rstd = rsqrtf(warp_sum(q) / H + eps);
}

// ------------------------------------------------------------------------------------------------ embedding
// z = words[tok] + positions[t];  out = LN_eps(z) -> dropout -> * [tok != pad]
__global__ void embed_fwd_kernel(const long long* __restrict__ tokens, const float* __restrict__ words,
                                 const float* __restrict__ positions, const float* __restrict__ gamma,
                                 const float* __restrict__ beta, float* __restrict__ z, float* __restrict__ stats,
                                 float* __restrict__ out, __nv_bfloat16* __restrict__ out_bf, int M, int T, int H,
                                 int pad, float eps, float p, const uint64_t* seed_ptr, uint32_t site) {
  VTX_PDL_TRIGGER();
  const uint64_t seed = seed_ptr ? *seed_ptr : 0ull;
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (row >= M) return;
  const long long tok = tokens[row];
  const int t = row % T;
  float* zr = z + (long long)row * H;
  for (int i = lane * 4; i < H; i += 128) {
    const float4 a = *reinterpret_cast<const float4*>(words + tok * H + i);
    const float4 b = *reinterpret_cast<const float4*>(positions + (long long)t * H + i);
    *reinterpret_cast<float4*>(zr + i) = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
  }
  __syncwarp();
  float mean, rstd;
  warp_row_stats(zr, H, lane, eps, mean, rstd);
  if (lane == 0) {
    stats[2 * row] = mean;
    stats[2 * row + 1] = rstd;
  }
  const float keep = (tok != pad) ? 1.f : 0.f;
  const float inv_keep = p > 0.f ? 1.f / (1.f - p) : 1.f;
  for (int i = lane * 4; i < H; i += 128) {
    const float4 v = *reinterpret_cast<const float4*>(zr + i);
    const float4 g = *reinterpret_cast<const float4*>(gamma + i);
    const float4 b = *reinterpret_cast<const float4*>(beta + i);
    float o[4] = {(v.x - mean) * rstd * g.x + b.x, (v.y - mean) * rstd * g.y + b.y, (v.z - mean) * rstd * g.z + b.z,
                  (v.w - mean) * rstd * g.w + b.w};
    const Drop4 dr = drop4(p, inv_keep, seed, site, ((uint64_t)row * H + i) >> 2);
#pragma unroll
    for (int j = 0; j < 4; ++j) o[j] *= keep * dr.scale(j);
    *reinterpret_cast<float4*>(out + (long long)row * H + i) = make_float4(o[0], o[1], o[2], o[3]);
    __nv_bfloat162 h0 = __floats2bfloat162_rn(o[0], o[1]), h1 = __floats2bfloat162_rn(o[2], o[3]);
    uint2 u;
    u.x = *reinterpret_cast<uint32_t*>(&h0);
    u.y = *reinterpret_cast<uint32_t*>(&h1);
    *reinterpret_cast<uint2*>(out_bf + (long long)row * H + i) = u;
  }
}

// upstream g = (dy_a + dy_b) * [tok != pad] * dropmask -> LN backward -> scatter-add into d_words[tok], d_positions[t]
__global__ void embed_bwd_kernel(const float* __restrict__ dy_a, const __nv_bfloat16* __restrict__ dy_b,
                                 const long long* __restrict__ tokens, const float* __restrict__ z,
                                 const float* __restrict__ stats, const float* __restrict__ gamma,
                                 float* __restrict__ d_words, float* __restrict__ d_pos, float* __restrict__ d_gamma,
                                 float* __restrict__ d_beta, int M, int T, int H, int pad, float p, const uint64_t* seed_ptr,
                                 uint32_t site) {
  VTX_PDL_TRIGGER();
  const uint64_t seed = seed_ptr ? *seed_ptr : 0ull;
  extern __shared__ float acc[];  // [2][H] : dgamma, dbeta partials of this CTA
  for (int i = threadIdx.x; i < 2 * H; i += blockDim.x) acc[i] = 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const float inv_keep = p > 0.f ? 1.f / (1.f - p) : 1.f;
  for (int row = blockIdx.x * kWarpsPerBlock + warp; row < M; row += gridDim.x * kWarpsPerBlock) {
    const long long tok = tokens[row];
    if (tok == pad) continue;  // zero upstream gradient: contributes nothing anywhere
    const int t = row % T;
    const float mean = stats[2 * row], rstd = stats[2 * row + 1];
    const float* zr = z + (long long)row * H;
    float s1 = 0.f, s2 = 0.f;
    for (int i = lane; i < H; i += 32) {
      float g = dy_a ? dy_a[(long long)row * H + i] : 0.f;
      if (dy_b) g += bf2f(dy_b[(long long)row * H + i]);
      g *= dropout_scale(p, inv_keep, seed, site, (uint64_t)row * H + i);
      const float xh = (zr[i] - mean) * rstd;
      atomicAdd(&acc[i], g * xh);
      atomicAdd(&acc[H + i], g);
      const float dxh = g * gamma[i];
      s1 += dxh;
      s2 += dxh * xh;
    }
    s1 = warp_sum(s1) / H;
    s2 = warp_sum(s2) / H;
    for (int i = lane; i < H; i += 32) {
      float g = dy_a ? dy_a[(long long)row * H + i] : 0.f;
      if (dy_b) g += bf2f(dy_b[(long long)row * H + i]);
      g *= dropout_scale(p, inv_keep, seed, site, (uint64_t)row * H + i);
      const float xh = (zr[i] - mean) * rstd;
      const float dz = rstd * (g * gamma[i] - s1 - xh * s2);
      atomicAdd(d_words + tok * H + i, dz);
      atomicAdd(d_pos + (long long)t * H + i, dz);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < H; i += blockDim.x) {
    atomicAdd(d_gamma + i, acc[i]);
    atomicAdd(d_beta + i, acc[H + i]);
  }
}

// ------------------------------------------------------------------------------------------------ add + dropout + LN
// z = res + dropout(branch);  out = LN(z)*gamma + beta     (ln == 0: out = z, the pre-norm residual update)
__global__ void add_ln_fwd_kernel(const float* __restrict__ res, const __nv_bfloat16* __restrict__ branch,
                                  const float* __restrict__ gamma, const float* __restrict__ beta,
                                  float* __restrict__ z, float* __restrict__ stats, float* __restrict__ out,
                                  __nv_bfloat16* __restrict__ out_bf, int M, int H, float eps, float p, const uint64_t* seed_ptr,
                                  uint32_t site, int ln) {
  VTX_PDL_TRIGGER();
  const uint64_t seed = seed_ptr ? *seed_ptr : 0ull;
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (row >= M) return;
  const float inv_keep = p > 0.f ? 1.f / (1.f - p) : 1.f;
  float* zr = z + (long long)row * H;
  for (int i = lane * 4; i < H; i += 128) {
    float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
    if (res) r = *reinterpret_cast<const float4*>(res + (long long)row * H + i);
    if (branch) {
      const uint2 u = *reinterpret_cast<const uint2*>(branch + (long long)row * H + i);
      const float2 b0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
      const float2 b1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
      const Drop4 dr = drop4(p, inv_keep, seed, site, ((uint64_t)row * H + i) >> 2);
      r.x += b0.x * dr.scale(0);
      r.y += b0.y * dr.scale(1);
      r.z += b1.x * dr.scale(2);
      r.w += b1.y * dr.scale(3);
    }
    *reinterpret_cast<float4*>(zr + i) = r;
  }
  __syncwarp();
  float mean = 0.f, rstd = 1.f;
  if (ln) {
    warp_row_stats(zr, H, lane, eps, mean, rstd);
    if (lane == 0) {
      stats[2 * row] = mean;
      stats[2 * row + 1] = rstd;
    }
  }
  for (int i = lane * 4; i < H; i += 128) {
    const float4 v = *reinterpret_cast<const float4*>(zr + i);
    float o[4] = {v.x, v.y, v.z, v.w};
    if (ln) {
      const float4 g = *reinterpret_cast<const float4*>(gamma + i);
      const float4 b = *reinterpret_cast<const float4*>(beta + i);
      o[0] = (v.x - mean) * rstd * g.x + b.x;
      o[1] = (v.y - mean) * rstd * g.y + b.y;
      o[2] = (v.z - mean) * rstd * g.z + b.z;
      o[3] = (v.w - mean) * rstd * g.w + b.w;
    }
    if (out) *reinterpret_cast<float4*>(out + (long long)row * H + i) = make_float4(o[0], o[1], o[2], o[3]);
    if (out_bf) {
      __nv_bfloat162 h0 = __floats2bfloat162_rn(o[0], o[1]), h1 = __floats2bfloat162_rn(o[2], o[3]);
      uint2 u;
      u.x = *reinterpret_cast<uint32_t*>(&h0);
      u.y = *reinterpret_cast<uint32_t*>(&h1);
      *reinterpret_cast<uint2*>(out_bf + (long long)row * H + i) = u;
    }
  }
}

// g = dy_a + dy_b;  LN backward -> dz;  d_res = dz (+ d_skip);  d_branch = dz * dropmask (bf16);  dgamma/dbeta +=
// ln == 0: dz = g (plain residual split).
__global__ void ln_bwd_kernel(const float* __restrict__ dy_a, const __nv_bfloat16* __restrict__ dy_b,
                              const float* __restrict__ z, const float* __restrict__ stats,
                              const float* __restrict__ gamma, const float* __restrict__ d_skip,
                              float* __restrict__ d_res, __nv_bfloat16* __restrict__ d_branch,
                              float* __restrict__ d_gamma, float* __restrict__ d_beta, int M, int H, float p,
                              const uint64_t* seed_ptr, uint32_t site, int ln) {
  VTX_PDL_TRIGGER();
  const uint64_t seed = seed_ptr ? *seed_ptr : 0ull;
  extern __shared__ float acc[];  // [warps][2][H] per-warp partial dgamma / dbeta (no atomics in the row loop)
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  float* my = acc + (size_t)warp * 2 * H;
  if (ln) {
    for (int i = lane; i < 2 * H; i += 32) my[i] = 0.f;
    __syncwarp();
  }
  const float inv_keep = p > 0.f ? 1.f / (1.f - p) : 1.f;
  for (int row = blockIdx.x * kWarpsPerBlock + warp; row < M; row += gridDim.x * kWarpsPerBlock) {
    const long long base = (long long)row * H;
    float mean = 0.f, rstd = 1.f, s1 = 0.f, s2 = 0.f;
    if (ln) {
      mean = stats[2 * row];
      rstd = stats[2 * row + 1];
      for (int i = lane * 4; i < H; i += 128) {
        float g[4] = {0.f, 0.f, 0.f, 0.f};
        if (dy_a) {
          const float4 t = *reinterpret_cast<const float4*>(dy_a + base + i);
          g[0] = t.x; g[1] = t.y; g[2] = t.z; g[3] = t.w;
        }
        if (dy_b) {
          const uint2 u = *reinterpret_cast<const uint2*>(dy_b + base + i);
          const float2 b0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
          const float2 b1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
          g[0] += b0.x; g[1] += b0.y; g[2] += b1.x; g[3] += b1.y;
        }
        const float4 zz = *reinterpret_cast<const float4*>(z + base + i);
        const float4 gm = *reinterpret_cast<const float4*>(gamma + i);
        const float xh[4] = {(zz.x - mean) * rstd, (zz.y - mean) * rstd, (zz.z - mean) * rstd, (zz.w - mean) * rstd};
        const float gw[4] = {gm.x, gm.y, gm.z, gm.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          my[i + j] += g[j] * xh[j];
          my[H + i + j] += g[j];
          const float dxh = g[j] * gw[j];
          s1 += dxh;
          s2 += dxh * xh[j];
        }
      }
      s1 = warp_sum(s1) / H;
      s2 = warp_sum(s2) / H;
    }
    for (int i = lane * 4; i < H; i += 128) {
      float g[4] = {0.f, 0.f, 0.f, 0.f};
      if (dy_a) {
        const float4 t = *reinterpret_cast<const float4*>(dy_a + base + i);
        g[0] = t.x; g[1] = t.y; g[2] = t.z; g[3] = t.w;
      }
      if (dy_b) {
        const uint2 u = *reinterpret_cast<const uint2*>(dy_b + base + i);
        const float2 b0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
        const float2 b1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
        g[0] += b0.x; g[1] += b0.y; g[2] += b1.x; g[3] += b1.y;
      }
      float dz[4] = {g[0], g[1], g[2], g[3]};
      if (ln) {
        const float4 zz = *reinterpret_cast<const float4*>(z + base + i);
        const float4 gm = *reinterpret_cast<const float4*>(gamma + i);
        dz[0] = rstd * (g[0] * gm.x - s1 - (zz.x - mean) * rstd * s2);
        dz[1] = rstd * (g[1] * gm.y - s1 - (zz.y - mean) * rstd * s2);
        dz[2] = rstd * (g[2] * gm.z - s1 - (zz.z - mean) * rstd * s2);
        dz[3] = rstd * (g[3] * gm.w - s1 - (zz.w - mean) * rstd * s2);
      }
      if (d_branch) {
        float t[4];
        const Drop4 dr = drop4(p, inv_keep, seed, site, ((uint64_t)base + i) >> 2);
#pragma unroll
        for (int j = 0; j < 4; ++j) t[j] = dz[j] * dr.scale(j);
        __nv_bfloat162 h0 = __floats2bfloat162_rn(t[0], t[1]), h1 = __floats2bfloat162_rn(t[2], t[3]);
        uint2 u;
        u.x = *reinterpret_cast<uint32_t*>(&h0);
        u.y = *reinterpret_cast<uint32_t*>(&h1);
        *reinterpret_cast<uint2*>(d_branch + base + i) = u;
      }
      if (d_res) {
        float4 o = make_float4(dz[0], dz[1], dz[2], dz[3]);
        if (d_skip) {
          const float4 k = *reinterpret_cast<const float4*>(d_skip + base + i);
          o.x += k.x; o.y += k.y; o.z += k.z; o.w += k.w;
        }
        *reinterpret_cast<float4*>(d_res + base + i) = o;
      }
    }
  }
  if (ln) {
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * H; i += blockDim.x) {
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < kWarpsPerBlock; ++w) t += acc[(size_t)w * 2 * H + i];
      atomicAdd((i < H ? d_gamma + i : d_beta + (i - H)), t);
    }
  }
}

// ------------------------------------------------------------------------------- register-accumulating variants
// Used for H in {128, 256, 512, 1024} (the generic kernels above serve every other width, e.g. H = 2048).  Same
// arithmetic as ln_bwd_kernel / embed_bwd_kernel, different data movement (validated on B200 in round 2: -1.1 ms/step):
//   * every lane owns the columns {lane*4 + 128*k}: the upstream gradient and z are read ONCE per row (they were read
//     twice) and the dgamma / dbeta (/ dposition) partial sums of all rows of a warp stay in REGISTERS; the validated
//     kernels do two shared-memory read-modify-writes per element, 4-way bank conflicted (ln_bwd) or shared-memory
//     atomics (embed_bwd);
//   * embed_bwd: a warp only handles rows of ONE position t, so d_positions gets one atomic per column per warp instead
//     of one per element (7.8 M atomics on 30 x 1024 addresses), and the word-table scatter uses red.global.add.v4.f32.
__device__ __forceinline__ void red_add_v4_head(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// loads the 4 upstream-gradient values of columns [i, i+4) of one row: g = dy_a (fp32, optional) + dy_b (bf16, optional)
__device__ __forceinline__ void load_g4(const float* dy_a, const __nv_bfloat16* dy_b, long long off, float* g) {
  g[0] = g[1] = g[2] = g[3] = 0.f;
  if (dy_a) {
    const float4 t = *reinterpret_cast<const float4*>(dy_a + off);
    g[0] = t.x; g[1] = t.y; g[2] = t.z; g[3] = t.w;
  }
  if (dy_b) {
    const uint2 u = *reinterpret_cast<const uint2*>(dy_b + off);
    const float2 b0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
    const float2 b1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
    g[0] += b0.x; g[1] += b0.y; g[2] += b1.x; g[3] += b1.y;
  }
}

// cross-warp reduction of per-lane column partials through shared memory, then one atomic per column per CTA
template <int KB>
__device__ __forceinline__ void flush_columns(float* smem, const float* part, float* dst, int H) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
#pragma unroll
  for (int k = 0; k < KB; ++k)
    *reinterpret_cast<float4*>(smem + warp * H + lane * 4 + 128 * k) =
        make_float4(part[4 * k], part[4 * k + 1], part[4 * k + 2], part[4 * k + 3]);
  __syncthreads();
  for (int i = threadIdx.x; i < H; i += blockDim.x) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kWarpsPerBlock; ++w) t += smem[w * H + i];
    atomicAdd(dst + i, t);
  }
}

template <int KB>
__global__ void __launch_bounds__(32 * kWarpsPerBlock)
ln_bwd_reg_kernel(const float* __restrict__ dy_a, const __nv_bfloat16* __restrict__ dy_b, const float* __restrict__ z,
                  const float* __restrict__ stats, const float* __restrict__ gamma, const float* __restrict__ d_skip,
                  float* __restrict__ d_res, __nv_bfloat16* __restrict__ d_branch, float* __restrict__ d_gamma,
                  float* __restrict__ d_beta, int M, float p, const uint64_t* seed_ptr, uint32_t site) {
  VTX_PDL_TRIGGER();
  constexpr int H = KB * 128;
  extern __shared__ float acc[];  // [warps][H] scratch of the final cross-warp reduction
  const uint64_t seed = seed_ptr ? *seed_ptr : 0ull;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float inv_keep = p > 0.f ? 1.f / (1.f - p) : 1.f;
  float dg[KB * 4], db[KB * 4];
#pragma unroll
  for (int j = 0; j < KB * 4; ++j) dg[j] = db[j] = 0.f;
  for (int row = blockIdx.x * kWarpsPerBlock + warp; row < M; row += gridDim.x * kWarpsPerBlock) {
    const long long base = (long long)row * H;
    const float mean = stats[2 * row], rstd = stats[2 * row + 1];
    float g[KB * 4], xh[KB * 4];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int k = 0; k < KB; ++k) {
      const int i = lane * 4 + 128 * k;
      load_g4(dy_a, dy_b, base + i, g + 4 * k);
      const float4 zz = *reinterpret_cast<const float4*>(z + base + i);
      const float4 gm = *reinterpret_cast<const float4*>(gamma + i);
      xh[4 * k] = (zz.x - mean) * rstd; xh[4 * k + 1] = (zz.y - mean) * rstd;
      xh[4 * k + 2] = (zz.z - mean) * rstd; xh[4 * k + 3] = (zz.w - mean) * rstd;
      const float gw[4] = {gm.x, gm.y, gm.z, gm.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        dg[4 * k + j] += g[4 * k + j] * xh[4 * k + j];
        db[4 * k + j] += g[4 * k + j];
        const float dxh = g[4 * k + j] * gw[j];
        s1 += dxh;
        s2 += dxh * xh[4 * k + j];
      }
    }
    s1 = warp_sum(s1) / H;
    s2 = warp_sum(s2) / H;
#pragma unroll
    for (int k = 0; k < KB; ++k) {
      const int i = lane * 4 + 128 * k;
      const float4 gm = *reinterpret_cast<const float4*>(gamma + i);  // L1 hit: same addresses as above
      const float gw[4] = {gm.x, gm.y, gm.z, gm.w};
      float dz[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) dz[j] = rstd * (g[4 * k + j] * gw[j] - s1 - xh[4 * k + j] * s2);
      if (d_branch) {
        float t[4];
        const Drop4 dr = drop4(p, inv_keep, seed, site, ((uint64_t)base + i) >> 2);
#pragma unroll
        for (int j = 0; j < 4; ++j) t[j] = dz[j] * dr.scale(j);
        __nv_bfloat162 h0 = __floats2bfloat162_rn(t[0], t[1]), h1 = __floats2bfloat162_rn(t[2], t[3]);
        uint2 u;
        u.x = *reinterpret_cast<uint32_t*>(&h0);
        u.y = *reinterpret_cast<uint32_t*>(&h1);
        *reinterpret_cast<uint2*>(d_branch + base + i) = u;
      }
      if (d_res) {
        float4 o = make_float4(dz[0], dz[1], dz[2], dz[3]);
        if (d_skip) {
          const float4 sk = *reinterpret_cast<const float4*>(d_skip + base + i);
          o.x += sk.x; o.y += sk.y; o.z += sk.z; o.w += sk.w;
        }
        *reinterpret_cast<float4*>(d_res + base + i) = o;
      }
    }
  }
  flush_columns<KB>(acc, dg, d_gamma, H);
  flush_columns<KB>(acc, db, d_beta, H);
}

// warp w handles position t = w % T and the batch entries {w / T, w / T + NC, ...}: rows b*T + t
template <int KB>
__global__ void __launch_bounds__(32 * kWarpsPerBlock)
embed_bwd_reg_kernel(const float* __restrict__ dy_a, const __nv_bfloat16* __restrict__ dy_b,
                     const long long* __restrict__ tokens, const float* __restrict__ z, const float* __restrict__ stats,
                     const float* __restrict__ gamma, float* __restrict__ d_words, float* __restrict__ d_pos,
                     float* __restrict__ d_gamma, float* __restrict__ d_beta, int M, int T, int pad, float p,
                     const uint64_t* seed_ptr, uint32_t site) {
  VTX_PDL_TRIGGER();
  constexpr int H = KB * 128;
  extern __shared__ float acc[];  // [warps][H]
  const uint64_t seed = seed_ptr ? *seed_ptr : 0ull;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float inv_keep = p > 0.f ? 1.f / (1.f - p) : 1.f;
  const int gw_id = blockIdx.x * kWarpsPerBlock + warp;
  const int nc = (gridDim.x * kWarpsPerBlock) / T;  // batch chunks (host guarantees >= 1)
  const int t = gw_id % T, chunk = gw_id / T;
  const int B = M / T;
  float dg[KB * 4], db[KB * 4], dp[KB * 4];
#pragma unroll
  for (int j = 0; j < KB * 4; ++j) dg[j] = db[j] = dp[j] = 0.f;
  if (chunk < nc) {
    for (int b = chunk; b < B; b += nc) {
      const int row = b * T + t;
      const long long tok = tokens[row];
      if (tok == pad) continue;  // zero upstream gradient: contributes nothing anywhere
      const long long base = (long long)row * H;
      const float mean = stats[2 * row], rstd = stats[2 * row + 1];
      float g[KB * 4], xh[KB * 4];
      float s1 = 0.f, s2 = 0.f;
#pragma unroll
      for (int k = 0; k < KB; ++k) {
        const int i = lane * 4 + 128 * k;
        load_g4(dy_a, dy_b, base + i, g + 4 * k);
        const float4 zz = *reinterpret_cast<const float4*>(z + base + i);
        const float4 gm = *reinterpret_cast<const float4*>(gamma + i);
        const float zv[4] = {zz.x, zz.y, zz.z, zz.w};
        const float gwv[4] = {gm.x, gm.y, gm.z, gm.w};
        const Drop4 dr = drop4(p, inv_keep, seed, site, ((uint64_t)base + i) >> 2);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float gj = g[4 * k + j] * dr.scale(j);
          const float x = (zv[j] - mean) * rstd;
          g[4 * k + j] = gj;
          xh[4 * k + j] = x;
          dg[4 * k + j] += gj * x;
          db[4 * k + j] += gj;
          const float dxh = gj * gwv[j];
          s1 += dxh;
          s2 += dxh * x;
        }
      }
      s1 = warp_sum(s1) / H;
      s2 = warp_sum(s2) / H;
#pragma unroll
      for (int k = 0; k < KB; ++k) {
        const int i = lane * 4 + 128 * k;
        const float4 gm = *reinterpret_cast<const float4*>(gamma + i);
        const float gwv[4] = {gm.x, gm.y, gm.z, gm.w};
        float dz[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          dz[j] = rstd * (g[4 * k + j] * gwv[j] - s1 - xh[4 * k + j] * s2);
          dp[4 * k + j] += dz[j];
        }
        red_add_v4_head(d_words + tok * H + i, dz[0], dz[1], dz[2], dz[3]);
      }
    }
#pragma unroll
    for (int k = 0; k < KB; ++k)
      red_add_v4_head(d_pos + (long long)t * H + lane * 4 + 128 * k, dp[4 * k], dp[4 * k + 1], dp[4 * k + 2],
                      dp[4 * k + 3]);
  }
  flush_columns<KB>(acc, dg, d_gamma, H);
  flush_columns<KB>(acc, db, d_beta, H);
}

// ------------------------------------------------------------------------------------------------ attention
// One warp per (batch b, head h); head_dim = 64; Tq <= 32 queries, Tk <= 64 keys.  The five small matrix products
// (S = Q K^T, O = P V; backward: dP = dO V^T, dQ = dS K, dK = dS^T Q, dV = P^T dO) run on mma.sync.m16n8k16 bf16
// tiles with fp32 accumulation -- the tiles are 30x30 / 30x49, far below a tcgen05 instruction shape, and the kernel
// is bound by its q/k/v/o bytes, not by math.  Operands are staged once in shared memory (row stride 72 halves:
// conflict-free ldmatrix); the causal + key-padding mask comes from caption_lengths and is never materialised.
// causal == 1: key j allowed for query i iff j <= i and j < lengths[b] (captioning: future + key-padding mask);
// causal == 2: iff j < lengths[b] (masked language modelling: key-padding mask only, textual_heads.py:255-262 with
// mask_future_positions = False); causal == 0: all Tk keys (cross-attention over the visual grid).
constexpr int kD = 64;
constexpr int kLd = 72;  // smem row stride in bf16 elements (144 B)

struct AttnArgs {
  const __nv_bfloat16 *q, *k, *v;
  long long ldq, ldk, ldv;
  int B, heads, Tq, Tk;
  const long long* lengths;
  int causal;
  float scale, p;
  const uint64_t* seed_ptr;
  uint32_t site;
};

__device__ __forceinline__ void mma16816(float* c, const uint32_t* a, const uint32_t* b) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
__device__ __forceinline__ void ldsm_x4(uint32_t* r, const __nv_bfloat16* p) {
  const uint32_t a = static_cast<uint32_t>(__cvta_generic_to_shared(p));
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t* r, const __nv_bfloat16* p) {
  const uint32_t a = static_cast<uint32_t>(__cvta_generic_to_shared(p));
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ void ldsm_x2(uint32_t* r, const __nv_bfloat16* p) {
  const uint32_t a = static_cast<uint32_t>(__cvta_generic_to_shared(p));
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(a));
}
__device__ __forceinline__ void ldsm_x2_t(uint32_t* r, const __nv_bfloat16* p) {
  const uint32_t a = static_cast<uint32_t>(__cvta_generic_to_shared(p));
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(a));
}
__device__ __forceinline__ uint32_t pack_bf2(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

// A fragment (m16 x k16) of a row-major [m][k] smem tile at (m0, k0)
__device__ __forceinline__ void frag_a(uint32_t* a, const __nv_bfloat16* t, int m0, int k0, int lane) {
  ldsm_x4(a, t + (m0 + (lane & 7) + ((lane >> 3) & 1) * 8) * kLd + k0 + (lane >> 4) * 8);
}
// A fragment of the TRANSPOSE of a row-major [k][m] smem tile: A[m][k] = X[k][m]
__device__ __forceinline__ void frag_a_t(uint32_t* a, const __nv_bfloat16* x, int m0, int k0, int lane) {
  ldsm_x4_t(a, x + (k0 + (lane & 7) + (lane >> 4) * 8) * kLd + m0 + ((lane >> 3) & 1) * 8);
}
// B fragment (k16 x n8) where the smem tile is [n][k] row-major (k contiguous)
__device__ __forceinline__ void frag_b(uint32_t* b, const __nv_bfloat16* t, int n0, int k0, int lane) {
  ldsm_x2(b, t + (n0 + (lane & 7)) * kLd + k0 + ((lane >> 3) & 1) * 8);
}
// B fragment where the smem tile is [k][n] row-major (n contiguous)
__device__ __forceinline__ void frag_b_t(uint32_t* b, const __nv_bfloat16* t, int k0, int n0, int lane) {
  ldsm_x2_t(b, t + (k0 + (lane & 7) + ((lane >> 3) & 1) * 8) * kLd + n0);
}

// rows x 64 bf16 global -> smem [rows_pad][kLd], zero filling rows >= rows.  Asynchronous 16-byte copies
// (cp.async.cg, bypassing L1): a warp issues ALL chunks of Q, K and V (and dO) before waiting once, so the unit costs
// one memory latency instead of one per loop iteration (the synchronous load -> store loop made the kernel latency
// bound at ~10x its byte roofline).  Rows past `rows` use src-size 0: the hardware writes zeros, the (clamped) source
// address is never dereferenced.
__device__ __forceinline__ void stage_rows_async(__nv_bfloat16* dst, const __nv_bfloat16* src, long long ld, int rows,
                                                 int rows_pad, int lane) {
  for (int e = lane; e < rows_pad * 8; e += 32) {
    const int r = e >> 3, c = (e & 7) * 8;
    const bool ok = r < rows;
    const __nv_bfloat16* gp = src + (long long)(ok ? r : 0) * ld + c;
    const uint32_t sa = static_cast<uint32_t>(__cvta_generic_to_shared(dst + r * kLd + c));
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(sa), "l"(gp), "r"(ok ? 16 : 0) : "memory");
  }
}
__device__ __forceinline__ void stage_wait_all() {
  asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
  __syncwarp();
}

constexpr int kAttnFwdWarps = 4;
// shared memory per warp: Q [32] + K [Tk16] + V [Tk16] rows of kLd bf16 (self-attention: Tk16 = 32 -> 13.5 KB, twice the
// resident warps of the cross-attention case Tk16 = 64)
__host__ __device__ constexpr int attn_fwd_smem_per_warp(int Tk16) { return (32 + 2 * Tk16) * kLd * 2; }

__global__ void __launch_bounds__(32 * kAttnFwdWarps) attn_fwd_kernel(const AttnArgs a, __nv_bfloat16* __restrict__ out,
                                                                        long long ldo, float* __restrict__ lse) {
  VTX_PDL_TRIGGER();
  const uint64_t seed = a.seed_ptr ? *a.seed_ptr : 0ull;
  extern __shared__ __align__(16) uint8_t sm_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int unit = blockIdx.x * kAttnFwdWarps + warp;
  if (unit >= a.B * a.heads) return;
  const int b = unit / a.heads, h = unit % a.heads;
  const int Tk16 = (a.Tk + 15) & ~15;
  __nv_bfloat16* sQ = reinterpret_cast<__nv_bfloat16*>(sm_raw + (size_t)warp * attn_fwd_smem_per_warp(Tk16));
  __nv_bfloat16* sK = sQ + 32 * kLd;
  __nv_bfloat16* sV = sK + Tk16 * kLd;
  stage_rows_async(sQ, a.q + (long long)b * a.Tq * a.ldq + h * kD, a.ldq, a.Tq, 32, lane);
  stage_rows_async(sK, a.k + (long long)b * a.Tk * a.ldk + h * kD, a.ldk, a.Tk, Tk16, lane);
  stage_rows_async(sV, a.v + (long long)b * a.Tk * a.ldv + h * kD, a.ldv, a.Tk, Tk16, lane);
  stage_wait_all();
  const int g = lane >> 2, tq = lane & 3;
  const int len = a.causal ? (int)a.lengths[b] : a.Tk;
  const int nkt = Tk16 >> 3;  // 8-key tiles
  float s[2][8][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) s[mt][nt][e] = 0.f;
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    uint32_t af[2][4];
    frag_a(af[0], sQ, 0, ks * 16, lane);
    frag_a(af[1], sQ, 16, ks * 16, lane);
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      if (nt < nkt) {
        uint32_t bf[2];
        frag_b(bf, sK, nt * 8, ks * 16, lane);
        mma16816(s[0][nt], af[0], bf);
        mma16816(s[1][nt], af[1], bf);
      }
    }
  }
  // masked softmax over keys; rows live in quads (4 lanes x 2 elements x 8 key tiles)
  const float inv_keep = a.p > 0.f ? 1.f / (1.f - a.p) : 1.f;
  float rsum[2][2];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
      const int i = mt * 16 + g + hh * 8;
      float mx = -INFINITY;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int j = nt * 8 + 2 * tq + e;
          const bool ok = (j < a.Tk) && (a.causal == 1 ? (j <= i && j < len) : a.causal == 2 ? (j < len) : true);
          const float v = ok ? s[mt][nt][hh * 2 + e] * a.scale : -INFINITY;
          s[mt][nt][hh * 2 + e] = v;
          mx = fmaxf(mx, v);
        }
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
      float sum = 0.f;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        // keys (j, j + 1) of this lane share one hash: element index ((unit*32 + i)*64 + j), j even
        const Drop4 dr = drop4(a.p, inv_keep, seed, a.site, (((uint64_t)unit * 32 + i) * 64 + nt * 8 + 2 * tq) >> 2);
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const float v = s[mt][nt][hh * 2 + e];
          float pr = (v == -INFINITY) ? 0.f : __expf(v - mx);
          sum += pr;
          pr *= dr.scale(((2 * tq) & 3) + e);
          s[mt][nt][hh * 2 + e] = pr;
        }
      }
      sum += __shfl_xor_sync(0xffffffffu, sum, 1);
      sum += __shfl_xor_sync(0xffffffffu, sum, 2);
      rsum[mt][hh] = sum;
      if (tq == 0 && i < a.Tq && lse) lse[(long long)unit * 32 + i] = mx + __logf(sum);
    }
  // O = P V
  float o[2][8][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) o[mt][nt][e] = 0.f;
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    if (ks * 16 < Tk16) {
      uint32_t pf[2][4];
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) {
        pf[mt][0] = pack_bf2(s[mt][2 * ks][0], s[mt][2 * ks][1]);
        pf[mt][1] = pack_bf2(s[mt][2 * ks][2], s[mt][2 * ks][3]);
        pf[mt][2] = pack_bf2(s[mt][2 * ks + 1][0], s[mt][2 * ks + 1][1]);
        pf[mt][3] = pack_bf2(s[mt][2 * ks + 1][2], s[mt][2 * ks + 1][3]);
      }
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        uint32_t bf[2];
        frag_b_t(bf, sV, ks * 16, nt * 8, lane);
        mma16816(o[0][nt], pf[0], bf);
        mma16816(o[1][nt], pf[1], bf);
      }
    }
  }
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
      const int i = mt * 16 + g + hh * 8;
      if (i >= a.Tq) continue;
      const float inv = 1.f / rsum[mt][hh];
      __nv_bfloat16* op = out + ((long long)b * a.Tq + i) * ldo + h * kD + 2 * tq;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt)
        *reinterpret_cast<uint32_t*>(op + nt * 8) = pack_bf2(o[mt][nt][hh * 2] * inv, o[mt][nt][hh * 2 + 1] * inv);
    }
}

constexpr int kAttnBwdWarps = 3;
// Q, dO, Pd, dS [32 rows each] + K, V [Tk16 rows each]
__host__ __device__ constexpr int attn_bwd_smem_per_warp(int Tk16) { return (4 * 32 + 2 * Tk16) * kLd * 2; }

__global__ void __launch_bounds__(32 * kAttnBwdWarps) attn_bwd_kernel(const AttnArgs a, const __nv_bfloat16* __restrict__ dout,
                                                                        long long ldo, const float* __restrict__ lse,
                                                                        __nv_bfloat16* __restrict__ dq, long long lddq,
                                                                        __nv_bfloat16* __restrict__ dk, long long lddk,
                                                                        __nv_bfloat16* __restrict__ dv, long long lddv) {
  VTX_PDL_TRIGGER();
  const uint64_t seed = a.seed_ptr ? *a.seed_ptr : 0ull;
  extern __shared__ __align__(16) uint8_t sm_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int unit = blockIdx.x * kAttnBwdWarps + warp;
  if (unit >= a.B * a.heads) return;
  const int b = unit / a.heads, h = unit % a.heads;
  const int Tk16 = (a.Tk + 15) & ~15;
  __nv_bfloat16* sQ = reinterpret_cast<__nv_bfloat16*>(sm_raw + (size_t)warp * attn_bwd_smem_per_warp(Tk16));
  __nv_bfloat16* sdO = sQ + 32 * kLd;
  __nv_bfloat16* sK = sdO + 32 * kLd;
  __nv_bfloat16* sV = sK + Tk16 * kLd;
  __nv_bfloat16* sP = sV + Tk16 * kLd;  // dropped probabilities Pd [query][key]
  __nv_bfloat16* sdS = sP + 32 * kLd;   // dS [query][key]
  stage_rows_async(sQ, a.q + (long long)b * a.Tq * a.ldq + h * kD, a.ldq, a.Tq, 32, lane);
  stage_rows_async(sdO, dout + (long long)b * a.Tq * ldo + h * kD, ldo, a.Tq, 32, lane);
  stage_rows_async(sK, a.k + (long long)b * a.Tk * a.ldk + h * kD, a.ldk, a.Tk, Tk16, lane);
  stage_rows_async(sV, a.v + (long long)b * a.Tk * a.ldv + h * kD, a.ldv, a.Tk, Tk16, lane);
  stage_wait_all();
  const int g = lane >> 2, tq = lane & 3;
  const int len = a.causal ? (int)a.lengths[b] : a.Tk;
  const int nkt = Tk16 >> 3;
  const float inv_keep = a.p > 0.f ? 1.f / (1.f - a.p) : 1.f;
  // ---- S = Q K^T and dPd = dO V^T
  float s[2][8][4], dp[2][8][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) s[mt][nt][e] = dp[mt][nt][e] = 0.f;
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    uint32_t aq[2][4], ao[2][4];
    frag_a(aq[0], sQ, 0, ks * 16, lane);
    frag_a(aq[1], sQ, 16, ks * 16, lane);
    frag_a(ao[0], sdO, 0, ks * 16, lane);
    frag_a(ao[1], sdO, 16, ks * 16, lane);
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      if (nt < nkt) {
        uint32_t bk[2], bv[2];
        frag_b(bk, sK, nt * 8, ks * 16, lane);
        frag_b(bv, sV, nt * 8, ks * 16, lane);
        mma16816(s[0][nt], aq[0], bk);
        mma16816(s[1][nt], aq[1], bk);
        mma16816(dp[0][nt], ao[0], bv);
        mma16816(dp[1][nt], ao[1], bv);
      }
    }
  }
  // ---- P, dP, D_i, dS; stage Pd and dS (bf16) as [query][key]
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
      const int i = mt * 16 + g + hh * 8;
      const bool row_ok = i < a.Tq;
      const float L = row_ok ? lse[(long long)unit * 32 + i] : 0.f;
      float Di = 0.f;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        const Drop4 dr = drop4(a.p, inv_keep, seed, a.site, (((uint64_t)unit * 32 + i) * 64 + nt * 8 + 2 * tq) >> 2);
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int j = nt * 8 + 2 * tq + e;
          const bool ok = row_ok && (j < a.Tk) && (a.causal == 1 ? (j <= i && j < len) : a.causal == 2 ? (j < len) : true);
          const float pr = ok ? __expf(s[mt][nt][hh * 2 + e] * a.scale - L) : 0.f;
          const float mk = dr.scale(((2 * tq) & 3) + e);
          const float dpr = dp[mt][nt][hh * 2 + e] * mk;  // dP = dPd * mask
          Di += pr * dpr;
          s[mt][nt][hh * 2 + e] = pr;
          dp[mt][nt][hh * 2 + e] = dpr;
          // Pd is consumed by dV only
          sP[i * kLd + j] = f2bf(pr * mk);
        }
      }
      Di += __shfl_xor_sync(0xffffffffu, Di, 1);
      Di += __shfl_xor_sync(0xffffffffu, Di, 2);
#pragma unroll
      for (int nt = 0; nt < 8; ++nt)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int j = nt * 8 + 2 * tq + e;
          const float ds = s[mt][nt][hh * 2 + e] * (dp[mt][nt][hh * 2 + e] - Di) * a.scale;
          s[mt][nt][hh * 2 + e] = ds;
          sdS[i * kLd + j] = f2bf(ds);
        }
    }
  __syncwarp();
  // ---- dQ = dS K   (A = dS from registers, B = K [key][d] -> transposed fragments)
  {
    float acc[2][8][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < 8; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[mt][nt][e] = 0.f;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      if (ks * 16 < Tk16) {
        uint32_t pf[2][4];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          pf[mt][0] = pack_bf2(s[mt][2 * ks][0], s[mt][2 * ks][1]);
          pf[mt][1] = pack_bf2(s[mt][2 * ks][2], s[mt][2 * ks][3]);
          pf[mt][2] = pack_bf2(s[mt][2 * ks + 1][0], s[mt][2 * ks + 1][1]);
          pf[mt][3] = pack_bf2(s[mt][2 * ks + 1][2], s[mt][2 * ks + 1][3]);
        }
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          uint32_t bf[2];
          frag_b_t(bf, sK, ks * 16, nt * 8, lane);
          mma16816(acc[0][nt], pf[0], bf);
          mma16816(acc[1][nt], pf[1], bf);
        }
      }
    }
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        const int i = mt * 16 + g + hh * 8;
        if (i >= a.Tq) continue;
        __nv_bfloat16* op = dq + ((long long)b * a.Tq + i) * lddq + h * kD + 2 * tq;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
          *reinterpret_cast<uint32_t*>(op + nt * 8) = pack_bf2(acc[mt][nt][hh * 2], acc[mt][nt][hh * 2 + 1]);
      }
  }
  // ---- dV = Pd^T dO and dK = dS^T Q, one 16-key tile at a time (reduction over the 32 queries)
  for (int kt = 0; kt * 16 < Tk16; ++kt) {
    float av[8][4], ak[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) av[nt][e] = ak[nt][e] = 0.f;
#pragma unroll
    for (int ks = 0; ks < 2; ++ks) {
      uint32_t ap[4], as_[4];
      frag_a_t(ap, sP, kt * 16, ks * 16, lane);
      frag_a_t(as_, sdS, kt * 16, ks * 16, lane);
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        uint32_t bo[2], bq[2];
        frag_b_t(bo, sdO, ks * 16, nt * 8, lane);
        frag_b_t(bq, sQ, ks * 16, nt * 8, lane);
        mma16816(av[nt], ap, bo);
        mma16816(ak[nt], as_, bq);
      }
    }
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
      const int j = kt * 16 + g + hh * 8;
      if (j >= a.Tk) continue;
      __nv_bfloat16* pk = dk + ((long long)b * a.Tk + j) * lddk + h * kD + 2 * tq;
      __nv_bfloat16* pv = dv + ((long long)b * a.Tk + j) * lddv + h * kD + 2 * tq;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        *reinterpret_cast<uint32_t*>(pk + nt * 8) = pack_bf2(ak[nt][hh * 2], ak[nt][hh * 2 + 1]);
        *reinterpret_cast<uint32_t*>(pv + nt * 8) = pack_bf2(av[nt][hh * 2], av[nt][hh * 2 + 1]);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ GELU + dropout
__global__ void gelu_dropout_fwd_kernel(const __nv_bfloat16* __restrict__ u, __nv_bfloat16* __restrict__ h,
                                        long long n8, float p, const uint64_t* seed_ptr, uint32_t site) {
  VTX_PDL_TRIGGER();
  const uint64_t seed = seed_ptr ? *seed_ptr : 0ull;
  const float inv_keep = p > 0.f ? 1.f / (1.f - p) : 1.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    float f[8];
    unpack8(*reinterpret_cast<const bf16x8*>(u + i * 8), f);
    const Drop4 d0 = drop4(p, inv_keep, seed, site, (uint64_t)i * 2), d1 = drop4(p, inv_keep, seed, site, (uint64_t)i * 2 + 1);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      // the reference evaluates GELU on the bf16 tensor and rounds the result to bf16 before dropout
      const float g = bf2f(f2bf(0.5f * f[j] * (1.0f + erff(f[j] * 0.70710678118654752f))));
      f[j] = g * (j < 4 ? d0.scale(j) : d1.scale(j - 4));
    }
    *reinterpret_cast<bf16x8*>(h + i * 8) = pack8(f);
  }
}
// du = dh * dropmask * gelu'(u)     (in place over dh allowed)
__global__ void gelu_dropout_bwd_kernel(const __nv_bfloat16* __restrict__ dh, const __nv_bfloat16* __restrict__ u,
                                        __nv_bfloat16* __restrict__ du, long long n8, float p, const uint64_t* seed_ptr,
                                        uint32_t site) {
  VTX_PDL_TRIGGER();
  const uint64_t seed = seed_ptr ? *seed_ptr : 0ull;
  const float inv_keep = p > 0.f ? 1.f / (1.f - p) : 1.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    float d[8], x[8];
    unpack8(*reinterpret_cast<const bf16x8*>(dh + i * 8), d);
    unpack8(*reinterpret_cast<const bf16x8*>(u + i * 8), x);
    const Drop4 d0 = drop4(p, inv_keep, seed, site, (uint64_t)i * 2), d1 = drop4(p, inv_keep, seed, site, (uint64_t)i * 2 + 1);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float cdf = 0.5f * (1.0f + erff(x[j] * 0.70710678118654752f));
      const float pdf = 0.3989422804014327f * __expf(-0.5f * x[j] * x[j]);
      d[j] = d[j] * (j < 4 ? d0.scale(j) : d1.scale(j - 4)) * (cdf + x[j] * pdf);
    }
    *reinterpret_cast<bf16x8*>(du + i * 8) = pack8(d);
  }
}

// ------------------------------------------------------------------------------------------------ cross entropy
// counts[0] = number of targets != pad: tokens[b, t>=1] (shift = 1: next-token targets) or tokens[b, t] (shift = 0: the
// tensor already holds one label per position, e.g. masked_labels of virtex/models/masked_lm.py:68-72)
__global__ void count_valid_kernel(const long long* __restrict__ tokens, int B, int T, int pad, int shift,
                                   float* __restrict__ count) {
  VTX_PDL_TRIGGER();
  float c = 0.f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < B * T; i += gridDim.x * blockDim.x)
    if ((i % T) >= shift && tokens[i] != pad) c += 1.f;
  c = warp_sum(c);
  if ((threadIdx.x & 31) == 0 && c != 0.f) atomicAdd(count, c);
}

// One CTA per row (b,t) of bf16 logits [B*T, ldl].  Target = tokens[b,t+1] for t < T-1 (else ignored) when shift = 1,
// tokens[b,t] when shift = 0; ignored when
// == pad.  loss += nll / count;  if write_grad: logits row overwritten by dlogits = (softmax - onehot)/count (or 0).
__global__ void ce_kernel(__nv_bfloat16* __restrict__ logits, long long ldl, const long long* __restrict__ tokens, int T,
                          int V, int pad, int shift, const float* __restrict__ count, float* __restrict__ loss,
                          int write_grad) {
  VTX_PDL_TRIGGER();
  __shared__ float red[32];
  __shared__ float bcast;
  const int row = blockIdx.x;
  const int t = row % T;
  __nv_bfloat16* z = logits + (long long)row * ldl;
  const long long target = !shift ? tokens[row] : (t < T - 1) ? tokens[row + 1] : (long long)pad;
  const bool valid = target != pad;
  const int nv = V / 8;
  if (!valid) {
    if (write_grad)
      for (int i = threadIdx.x; i < nv; i += blockDim.x) *reinterpret_cast<uint4*>(z + i * 8) = make_uint4(0, 0, 0, 0);
    return;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  float mx = -INFINITY;
  for (int i = threadIdx.x; i < nv; i += blockDim.x) {
    float f[8];
    unpack8(*reinterpret_cast<const bf16x8*>(z + i * 8), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) mx = fmaxf(mx, f[j]);
  }
  mx = warp_max(mx);
  if (lane == 0) red[warp] = mx;
  __syncthreads();
  if (warp == 0) {
    float v = lane < nwarps ? red[lane] : -INFINITY;
    v = warp_max(v);
    if (lane == 0) bcast = v;
  }
  __syncthreads();
  mx = bcast;
  float s = 0.f;
  for (int i = threadIdx.x; i < nv; i += blockDim.x) {
    float f[8];
    unpack8(*reinterpret_cast<const bf16x8*>(z + i * 8), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) s += __expf(f[j] - mx);
  }
  s = warp_sum(s);
  __syncthreads();
  if (lane == 0) red[warp] = s;
  __syncthreads();
  if (warp == 0) {
    float v = lane < nwarps ? red[lane] : 0.f;
    v = warp_sum(v);
    if (lane == 0) bcast = v;
  }
  __syncthreads();
  s = bcast;
  const float inv_n = 1.f / fmaxf(*count, 1.f);
  if (threadIdx.x == 0) {
    const float zt = bf2f(z[target]);
    atomicAdd(loss, (mx + __logf(s) - zt) * inv_n);
  }
  if (write_grad) {
    const float inv_s = 1.f / s;
    __syncthreads();  // everyone (incl. thread 0's read of z[target]) is done with the original logits
    for (int i = threadIdx.x; i < nv; i += blockDim.x) {
      float f[8];
      unpack8(*reinterpret_cast<const bf16x8*>(z + i * 8), f);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float pr = __expf(f[j] - mx) * inv_s;
        f[j] = (pr - ((long long)(i * 8 + j) == target ? 1.f : 0.f)) * inv_n;
      }
      *reinterpret_cast<bf16x8*>(z + i * 8) = pack8(f);
    }
  }
}

// Same arithmetic as ce_kernel with the row held in registers -- one global read pass with all
// of a thread's loads in flight (the validated kernel walks the row three times with one dependent load at a time,
// ~3 x 5 x memory latency per CTA) and exp() evaluated once.  Rows of up to 256 * 8 * IT logits.
template <int IT>
__global__ void __launch_bounds__(256) ce_reg_kernel(__nv_bfloat16* __restrict__ logits, long long ldl,
                                                    const long long* __restrict__ tokens, int T, int V, int pad,
                                                    int shift, const float* __restrict__ count,
                                                    float* __restrict__ loss, int write_grad) {
  VTX_PDL_TRIGGER();
  __shared__ float red[32];
  __shared__ float bcast;
  const int row = blockIdx.x;
  const int t = row % T;
  __nv_bfloat16* z = logits + (long long)row * ldl;
  const long long target = !shift ? tokens[row] : (t < T - 1) ? tokens[row + 1] : (long long)pad;
  const bool valid = target != pad;
  const int nv = V / 8;
  if (!valid) {
    if (write_grad)
      for (int i = threadIdx.x; i < nv; i += blockDim.x) *reinterpret_cast<uint4*>(z + i * 8) = make_uint4(0, 0, 0, 0);
    return;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  float f[IT][8];
#pragma unroll
  for (int k = 0; k < IT; ++k) {
    const int i = threadIdx.x + k * 256;
    if (i < nv) {
      unpack8(*reinterpret_cast<const bf16x8*>(z + i * 8), f[k]);
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) f[k][j] = -INFINITY;
    }
  }
  const float zt = threadIdx.x == 0 ? bf2f(z[target]) : 0.f;  // read before anybody overwrites the row
  float mx = -INFINITY;
#pragma unroll
  for (int k = 0; k < IT; ++k)
#pragma unroll
    for (int j = 0; j < 8; ++j) mx = fmaxf(mx, f[k][j]);
  mx = warp_max(mx);
  if (lane == 0) red[warp] = mx;
  __syncthreads();
  if (warp == 0) {
    float v = lane < nwarps ? red[lane] : -INFINITY;
    v = warp_max(v);
    if (lane == 0) bcast = v;
  }
  __syncthreads();
  mx = bcast;
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < IT; ++k) {
    if (threadIdx.x + k * 256 < nv) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        f[k][j] = __expf(f[k][j] - mx);
        s += f[k][j];
      }
    }
  }
  s = warp_sum(s);
  __syncthreads();
  if (lane == 0) red[warp] = s;
  __syncthreads();
  if (warp == 0) {
    float v = lane < nwarps ? red[lane] : 0.f;
    v = warp_sum(v);
    if (lane == 0) bcast = v;
  }
  __syncthreads();
  s = bcast;
  const float inv_n = 1.f / fmaxf(*count, 1.f);
  if (threadIdx.x == 0) atomicAdd(loss, (mx + __logf(s) - zt) * inv_n);
  if (write_grad) {
    const float inv_s = 1.f / s;
#pragma unroll
    for (int k = 0; k < IT; ++k) {
      const int i = threadIdx.x + k * 256;
      if (i < nv) {
        float g[8];
#pragma unroll
        for (int j = 0; j < 8; ++j)
          g[j] = (f[k][j] * inv_s - ((long long)(i * 8 + j) == target ? 1.f : 0.f)) * inv_n;
        *reinterpret_cast<bf16x8*>(z + i * 8) = pack8(g);
      }
    }
  }
}

// out[n] += sum_m X[m,n]    X bf16 [M, ld]
__global__ void colsum_kernel(const __nv_bfloat16* __restrict__ X, long long ld, int M, int N, float* __restrict__ out,
                              int rows_per_block) {
  VTX_PDL_TRIGGER();
  const int g = blockIdx.y * blockDim.x + threadIdx.x;  // 8-column group
  if (g * 8 >= N) return;
  const int m0 = blockIdx.x * rows_per_block;
  const int m1 = min(M, m0 + rows_per_block);
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  int m = m0;
  for (; m + 4 <= m1; m += 4) {  // four independent 16-byte loads in flight per thread
    bf16x8 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = *reinterpret_cast<const bf16x8*>(X + (long long)(m + u) * ld + g * 8);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      float f[8];
      unpack8(v[u], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += f[j];
    }
  }
  for (; m < m1; ++m) {
    float f[8];
    unpack8(*reinterpret_cast<const bf16x8*>(X + (long long)m * ld + g * 8), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] += f[j];
  }
#pragma unroll
  for (int j = 0; j < 8; ++j)
    if (g * 8 + j < N) atomicAdd(out + g * 8 + j, acc[j]);
}

// Row-lane variant (M >= 64): a CTA covers 256 columns x a row slice with 8 row lanes (one per warp) and reduces the lanes in
// shared memory, so the number of atomics per output column drops from (row blocks) = 296 to 296 / (N / 256) -- the
// validated kernel is bound by those atomics (31 us for a 15.7 MB input).
__global__ void __launch_bounds__(256) colsum_lanes_kernel(const __nv_bfloat16* __restrict__ X, long long ld, int M, int N,
                                                          float* __restrict__ out, int rows_per_block) {
  VTX_PDL_TRIGGER();
  __shared__ float red[8][256];
  const int cgrp = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int col0 = blockIdx.y * 256 + cgrp * 8;
  const int m0 = blockIdx.x * rows_per_block;
  const int m1 = min(M, m0 + rows_per_block);
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  if (col0 < N) {
    const __nv_bfloat16* xp = X + col0;
    int m = m0 + rl;
    for (; m + 24 < m1; m += 32) {  // four independent 16-byte loads in flight per thread
      bf16x8 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = *reinterpret_cast<const bf16x8*>(xp + (long long)(m + 8 * u) * ld);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        float f[8];
        unpack8(v[u], f);
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] += f[j];
      }
    }
    for (; m < m1; m += 8) {
      float f[8];
      unpack8(*reinterpret_cast<const bf16x8*>(xp + (long long)m * ld), f);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += f[j];
    }
  }
  *reinterpret_cast<float4*>(&red[rl][cgrp * 8]) = make_float4(acc[0], acc[1], acc[2], acc[3]);
  *reinterpret_cast<float4*>(&red[rl][cgrp * 8 + 4]) = make_float4(acc[4], acc[5], acc[6], acc[7]);
  __syncthreads();
  const int c = blockIdx.y * 256 + threadIdx.x;
  if (c < N) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += red[w][threadIdx.x];
    atomicAdd(out + c, t);
  }
}

// first-index argmax of each fp32 row.  NaN compares greater than every number and the first NaN wins, as in
// torch.argmax: a row with a NaN logit must not return the largest finite index, nor an all-NaN row a sentinel index.
__device__ __forceinline__ bool argmax_better(float v, int i, float best, int idx) {
  const bool vn = isnan(v), bn = isnan(best);
  if (vn != bn) return vn;
  return v > best || ((v == best || vn) && i < idx);
}
__global__ void argmax_rows_kernel(const float* __restrict__ X, long long ld, int N, long long* __restrict__ out) {
  VTX_PDL_TRIGGER();
  __shared__ float bv[32];
  __shared__ int bi[32];
  const float* x = X + (long long)blockIdx.x * ld;
  float best = -INFINITY;
  int idx = 0x7fffffff;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const float v = x[i];
    if (argmax_better(v, i, best, idx)) { best = v; idx = i; }
  }
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
    if (argmax_better(ov, oi, best, idx)) { best = ov; idx = oi; }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { bv[warp] = best; bi[warp] = idx; }
  __syncthreads();
  if (warp == 0) {
    best = lane < (blockDim.x >> 5) ? bv[lane] : -INFINITY;
    idx = lane < (blockDim.x >> 5) ? bi[lane] : 0x7fffffff;
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, best, o);
      const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
      if (argmax_better(ov, oi, best, idx)) { best = ov; idx = oi; }
    }
    if (lane == 0) out[blockIdx.x] = idx;
  }
}

}  // namespace vtx

using namespace vtx;
#define STREAM reinterpret_cast<cudaStream_t>(stream)
#define REQ(cond, msg) \
  if (!(cond)) return set_error(VTX_EINVAL, "%s: %s", __func__, msg)

extern "C" int vtx_embed_fwd(const int64_t* tokens, const float* words, const float* positions, const float* gamma,
                             const float* beta, float* z, float* stats, float* out, void* out_bf, int M, int T, int H,
                             int pad, float eps, float p, const uint64_t* seed_ptr, uint32_t site, void* stream) {
  REQ(tokens && words && positions && gamma && beta && z && stats && out && out_bf && H % 128 == 0, "bad arguments");
  embed_fwd_kernel<<<(M + kWarpsPerBlock - 1) / kWarpsPerBlock, 32 * kWarpsPerBlock, 0, STREAM>>>(
      (const long long*)tokens, words, positions, gamma, beta, z, stats, out, (__nv_bfloat16*)out_bf, M, T, H, pad, eps,
      p, seed_ptr, site);
  return check_launch("embed_fwd");
}
extern "C" int vtx_embed_bwd(const float* dy_a, const void* dy_b, const int64_t* tokens, const float* z,
                             const float* stats, const float* gamma, float* d_words, float* d_pos, float* d_gamma,
                             float* d_beta, int M, int T, int H, int pad, float p, const uint64_t* seed_ptr, uint32_t site,
                             void* stream) {
  REQ(tokens && z && stats && gamma && d_words && d_pos && d_gamma && d_beta && (dy_a || dy_b), "bad arguments");
  int blocks = (M + kWarpsPerBlock - 1) / kWarpsPerBlock;
  const int cap = vtx_num_sms() * 2;
  if (blocks > cap) blocks = cap;
  if (H % 128 == 0 && H <= 1024 && (H / 128 == 1 || H / 128 == 2 || H / 128 == 4 || H / 128 == 8) && T > 0 && M % T == 0) {
    int xb = cap;
    if (xb * kWarpsPerBlock < T) xb = (T + kWarpsPerBlock - 1) / kWarpsPerBlock;
    const size_t xs = (size_t)kWarpsPerBlock * H * sizeof(float);
#define VTX_EMB_X(KB)                                                                                                  \
  embed_bwd_reg_kernel<KB><<<xb, 32 * kWarpsPerBlock, xs, STREAM>>>(dy_a, (const __nv_bfloat16*)dy_b,                   \
                                                                      (const long long*)tokens, z, stats, gamma, d_words, \
                                                                      d_pos, d_gamma, d_beta, M, T, pad, p, seed_ptr, site)
    switch (H / 128) {
      case 1: VTX_EMB_X(1); break;
      case 2: VTX_EMB_X(2); break;
      case 4: VTX_EMB_X(4); break;
      default: VTX_EMB_X(8); break;
    }
#undef VTX_EMB_X
    return check_launch("embed_bwd_reg");
  }
  embed_bwd_kernel<<<blocks, 32 * kWarpsPerBlock, 2 * H * sizeof(float), STREAM>>>(
      dy_a, (const __nv_bfloat16*)dy_b, (const long long*)tokens, z, stats, gamma, d_words, d_pos, d_gamma, d_beta, M, T,
      H, pad, p, seed_ptr, site);
  return check_launch("embed_bwd");
}
extern "C" int vtx_add_ln_fwd(const float* res, const void* branch, const float* gamma, const float* beta, float* z,
                              float* stats, float* out, void* out_bf, int M, int H, float eps, float p, const uint64_t* seed_ptr,
                              uint32_t site, int ln, void* stream) {
  REQ(z && (res || branch) && H % 128 == 0 && (!ln || (gamma && beta && stats)), "bad arguments");
  add_ln_fwd_kernel<<<(M + kWarpsPerBlock - 1) / kWarpsPerBlock, 32 * kWarpsPerBlock, 0, STREAM>>>(
      res, (const __nv_bfloat16*)branch, gamma, beta, z, stats, out, (__nv_bfloat16*)out_bf, M, H, eps, p, seed_ptr, site,
      ln);
  return check_launch("add_ln_fwd");
}
extern "C" int vtx_ln_bwd(const float* dy_a, const void* dy_b, const float* z, const float* stats, const float* gamma,
                          const float* d_skip, float* d_res, void* d_branch, float* d_gamma, float* d_beta, int M,
                          int H, float p, const uint64_t* seed_ptr, uint32_t site, int ln, void* stream) {
  REQ((dy_a || dy_b) && H % 128 == 0 && (!ln || (z && stats && gamma && d_gamma && d_beta)), "bad arguments");
  int blocks = (M + kWarpsPerBlock - 1) / kWarpsPerBlock;
  const int cap = vtx_num_sms() * 2;
  if (blocks > cap) blocks = cap;
  if (ln && H % 128 == 0 && (H / 128 == 1 || H / 128 == 2 || H / 128 == 4 || H / 128 == 8)) {
    const size_t xs = (size_t)kWarpsPerBlock * H * sizeof(float);
#define VTX_LN_X(KB)                                                                                                   \
  ln_bwd_reg_kernel<KB><<<blocks, 32 * kWarpsPerBlock, xs, STREAM>>>(dy_a, (const __nv_bfloat16*)dy_b, z, stats, gamma,  \
                                                                     d_skip, d_res, (__nv_bfloat16*)d_branch, d_gamma,   \
                                                                     d_beta, M, p, seed_ptr, site)
    switch (H / 128) {
      case 1: VTX_LN_X(1); break;
      case 2: VTX_LN_X(2); break;
      case 4: VTX_LN_X(4); break;
      default: VTX_LN_X(8); break;
    }
#undef VTX_LN_X
    return check_launch("ln_bwd_reg");
  }
  const size_t ln_smem = ln ? (size_t)kWarpsPerBlock * 2 * H * sizeof(float) : 0;
  static size_t ln_attr = 0;
  if (ln_smem > 48 * 1024 && ln_smem > ln_attr) {
    cudaFuncSetAttribute(ln_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ln_smem);
    ln_attr = ln_smem;
  }
  ln_bwd_kernel<<<blocks, 32 * kWarpsPerBlock, ln_smem, STREAM>>>(
      dy_a, (const __nv_bfloat16*)dy_b, z, stats, gamma, d_skip, d_res, (__nv_bfloat16*)d_branch, d_gamma, d_beta, M, H,
      p, seed_ptr, site, ln);
  return check_launch("ln_bwd");
}

static int fill_attn(AttnArgs* a, const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                     int B, int heads, int Tq, int Tk, const int64_t* lengths, int causal, float p, const uint64_t* seed_ptr,
                     uint32_t site) {
  if (!q || !k || !v || Tq < 1 || Tq > 32 || Tk < 1 || Tk > 64 || causal < 0 || causal > 2 || (causal && !lengths))
    return set_error(VTX_EINVAL, "attention: unsupported shape (Tq<=32, Tk<=64, head_dim 64)");
  if (ldq % 8 || ldk % 8 || ldv % 8) return set_error(VTX_EINVAL, "attention: leading dims must be multiples of 8");
  a->q = (const __nv_bfloat16*)q; a->k = (const __nv_bfloat16*)k; a->v = (const __nv_bfloat16*)v;
  a->ldq = ldq; a->ldk = ldk; a->ldv = ldv;
  a->B = B; a->heads = heads; a->Tq = Tq; a->Tk = Tk;
  a->lengths = (const long long*)lengths; a->causal = causal;
  a->scale = 0.125f;  // 1/sqrt(64)
  a->p = p; a->seed_ptr = seed_ptr; a->site = site;
  return VTX_OK;
}

extern "C" int vtx_attn_fwd(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                            void* out, int64_t ldo, float* lse, int B, int heads, int Tq, int Tk,
                            const int64_t* lengths, int causal, float p, const uint64_t* seed_ptr, uint32_t site, void* stream) {
  AttnArgs a;
  int rc = fill_attn(&a, q, ldq, k, ldk, v, ldv, B, heads, Tq, Tk, lengths, causal, p, seed_ptr, site);
  if (rc) return rc;
  REQ(out && ldo % 8 == 0, "bad output");
  const size_t smem = (size_t)kAttnFwdWarps * attn_fwd_smem_per_warp((Tk + 15) & ~15);
  // per device and cheap: set unconditionally (a process may drive several devices through the module-level API)
  cudaFuncSetAttribute(attn_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       kAttnFwdWarps * attn_fwd_smem_per_warp(64));
  const int units = B * heads;
  attn_fwd_kernel<<<(units + kAttnFwdWarps - 1) / kAttnFwdWarps, 32 * kAttnFwdWarps, smem, STREAM>>>(
      a, (__nv_bfloat16*)out, ldo, lse);
  return check_launch("attn_fwd");
}
extern "C" int vtx_attn_bwd(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                            const void* dout, int64_t ldo, const float* lse, void* dq, int64_t lddq, void* dk,
                            int64_t lddk, void* dv, int64_t lddv, int B, int heads, int Tq, int Tk,
                            const int64_t* lengths, int causal, float p, const uint64_t* seed_ptr, uint32_t site, void* stream) {
  AttnArgs a;
  int rc = fill_attn(&a, q, ldq, k, ldk, v, ldv, B, heads, Tq, Tk, lengths, causal, p, seed_ptr, site);
  if (rc) return rc;
  REQ(dout && lse && dq && dk && dv && ldo % 8 == 0 && lddq % 8 == 0 && lddk % 8 == 0 && lddv % 8 == 0, "bad arguments");
  const size_t smem = (size_t)kAttnBwdWarps * attn_bwd_smem_per_warp((Tk + 15) & ~15);
  cudaFuncSetAttribute(attn_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       kAttnBwdWarps * attn_bwd_smem_per_warp(64));
  const int units = B * heads;
  attn_bwd_kernel<<<(units + kAttnBwdWarps - 1) / kAttnBwdWarps, 32 * kAttnBwdWarps, smem, STREAM>>>(
      a, (const __nv_bfloat16*)dout, ldo, lse, (__nv_bfloat16*)dq, lddq, (__nv_bfloat16*)dk, lddk, (__nv_bfloat16*)dv,
      lddv);
  return check_launch("attn_bwd");
}
extern "C" int vtx_gelu_dropout_fwd(const void* u, void* h, int64_t n, float p, const uint64_t* seed_ptr, uint32_t site,
                                    void* stream) {
  REQ(u && h && n % 8 == 0, "bad arguments");
  const long long n8 = n / 8;
  long long blocks = (n8 + 255) / 256;
  const long long cap = (long long)vtx_num_sms() * 8;
  if (blocks > cap) blocks = cap;
  gelu_dropout_fwd_kernel<<<(int)blocks, 256, 0, STREAM>>>((const __nv_bfloat16*)u, (__nv_bfloat16*)h, n8, p, seed_ptr, site);
  return check_launch("gelu_dropout_fwd");
}
extern "C" int vtx_gelu_dropout_bwd(const void* dh, const void* u, void* du, int64_t n, float p, const uint64_t* seed_ptr,
                                    uint32_t site, void* stream) {
  REQ(dh && u && du && n % 8 == 0, "bad arguments");
  const long long n8 = n / 8;
  long long blocks = (n8 + 255) / 256;
  const long long cap = (long long)vtx_num_sms() * 8;
  if (blocks > cap) blocks = cap;
  gelu_dropout_bwd_kernel<<<(int)blocks, 256, 0, STREAM>>>((const __nv_bfloat16*)dh, (const __nv_bfloat16*)u,
                                                           (__nv_bfloat16*)du, n8, p, seed_ptr, site);
  return check_launch("gelu_dropout_bwd");
}
extern "C" int vtx_count_valid(const int64_t* tokens, int B, int T, int pad, int shift, float* count, void* stream) {
  REQ(tokens && count && (shift == 0 || shift == 1), "bad arguments");
  count_valid_kernel<<<32, 256, 0, STREAM>>>((const long long*)tokens, B, T, pad, shift, count);
  return check_launch("count_valid");
}
extern "C" int vtx_cross_entropy(void* logits, int64_t ldl, const int64_t* tokens, int B, int T, int V, int pad,
                                 int shift, const float* count, float* loss, int write_grad, void* stream) {
  REQ(logits && tokens && count && loss && V % 8 == 0 && ldl % 8 == 0 && (shift == 0 || shift == 1), "bad arguments");
  if (V / 8 <= 256 * 5) {
    ce_reg_kernel<5><<<B * T, 256, 0, STREAM>>>((__nv_bfloat16*)logits, ldl, (const long long*)tokens, T, V, pad, shift,
                                                count, loss, write_grad);
    return check_launch("cross_entropy_reg");
  }
  ce_kernel<<<B * T, 256, 0, STREAM>>>((__nv_bfloat16*)logits, ldl, (const long long*)tokens, T, V, pad, shift, count,
                                       loss, write_grad);
  return check_launch("cross_entropy");
}
extern "C" int vtx_colsum(const void* X, int64_t ld, int M, int N, float* out, void* stream) {
  REQ(X && out && ld % 8 == 0, "bad arguments");
  if (N % 8 == 0 && M >= 64) {
    const int by = (N + 255) / 256;
    int bx = (vtx_num_sms() * 2 + by - 1) / by;
    if (bx > M / 8) bx = M / 8;
    const int rpb = (M + bx - 1) / bx;
    bx = (M + rpb - 1) / rpb;
    colsum_lanes_kernel<<<dim3(bx, by), 256, 0, STREAM>>>((const __nv_bfloat16*)X, ld, M, N, out, rpb);
    return check_launch("colsum_lanes");
  }
  const int groups = (N + 7) / 8;
  const int threads = 128;
  const int gy = (groups + threads - 1) / threads;
  int gx = (vtx_num_sms() * 2 + gy - 1) / gy;  // few row blocks: every block ends with one atomic per column
  if (gx > M) gx = M;
  if (gx < 1) gx = 1;
  const int rows_per_block = (M + gx - 1) / gx;
  gx = (M + rows_per_block - 1) / rows_per_block;
  colsum_kernel<<<dim3(gx, gy), threads, 0, STREAM>>>((const __nv_bfloat16*)X, ld, M, N, out, rows_per_block);
  return check_launch("colsum");
}
extern "C" int vtx_argmax_rows(const float* X, int64_t ld, int M, int N, int64_t* out, void* stream) {
  REQ(X && out, "bad arguments");
  argmax_rows_kernel<<<M, 256, 0, STREAM>>>(X, ld, N, (long long*)out);
  return check_launch("argmax_rows");
}
