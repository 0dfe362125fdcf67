// Fine-tuning of the attention-pooling head with the backbone frozen (ClassificationLit.training_step / model_step +
// configure_optimizers of the reference, chimeralm/models/basic_module.py:87-104,200-223).  The backbone forward is the
// unchanged clm_forward; what it leaves in the context (XN, score, the per-tile softmax partials, pooled) is all the
// backward needs, so the backbone is never recomputed.
//
//   ht_fwd_kernel          the classifier again, with dropout (p, keep-masks from dropout_hash) and its pre-activations kept
//   ht_loss_kernel         mean cross-entropy over the batch and d loss / d logits (F.cross_entropy)
//   ht_bwd_x_kernel        d input of one Linear (+ skip gradient), times the dropout mask and GELU' of the layer below
//   ht_bwd_w_kernel        d weight / d bias of one Linear, reduced over the batch
//   ht_pool_prep_kernel    per read: softmax normaliser from the merged partials, g * dpooled, (beta - pooled) . dpooled
//   score_bwd_kernel       pooling + scorer backward on the tensor cores (see below)
//   score_bwd_reduce_kernel  per-CTA partials -> d attention.0.{weight,bias}, d attention.2.{weight,bias}
//   adamw_kernel           torch.optim.AdamW on fp32 master copies, written through to the tensors the forward reads
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

#include "ptx.cuh"

namespace clm {

// ---------------------------------------------------------------------------------------------
// Dropout keep-masks: a counter-based hash, so that the mask of (seed, step, site, read, unit) needs no state and a host
// mirror reproduces every bit (chimeralm_b200/train.py::dropout_keep).  mix32 is the "lowbias32" integer finaliser:
//   mix32(x): x ^= x >> 16; x *= 0x7feb352d; x ^= x >> 15; x *= 0x846ca68b; x ^= x >> 16     (uint32 arithmetic)
//   h = mix32(seed ^ 0x9e3779b9); h = mix32(h ^ step); h = mix32(h ^ site); h = mix32(h ^ read); h = mix32(h ^ unit)
//   keep  <=>  (h >> 8) >= round(p * 2^24)
// site 0 = classifier.2, 1 = classifier.5, 2 = classifier.6.layers.2; read = row in the batch; unit = feature index.
__host__ __device__ __forceinline__ uint32_t mix32(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
  return x;
}
__host__ __device__ __forceinline__ bool dropout_keep(uint32_t seed, uint32_t step, uint32_t site, uint32_t read, uint32_t unit,
                                                      uint32_t thr) {
  uint32_t h = mix32(seed ^ 0x9e3779b9u);
  h = mix32(h ^ step); h = mix32(h ^ site); h = mix32(h ^ read); h = mix32(h ^ unit);
  return (h >> 8) >= thr;
}

struct DropoutCfg {
  uint32_t seed, step, thr;   // thr = round(p * 2^24); 0 disables dropout
  float scale;                // 1 / (1 - p)
};

__device__ __forceinline__ float ht_gelu(float z) { return 0.5f * z * (1.0f + erff(z * 0.7071067811865476f)); }
__device__ __forceinline__ float ht_gelu_grad(float z) {   // d/dz z Phi(z) = Phi(z) + z phi(z)
  return 0.5f * (1.0f + erff(z * 0.7071067811865476f)) + z * 0.3989422804014327f * __expf(-0.5f * z * z);
}

// ---------------------------------------------------------------------------------------------
// Classifier forward of a training step: y[b,o] = W[o,:] . x[b,:] + bias[o], one warp per output neuron o, all reads
// (the shape of head_layer_kernel).  MODE 0: z = y kept, out = dropout(GELU(z)); MODE 1: out = y + skip; MODE 2: out = y.
template <int IN, int MODE>
__global__ void __launch_bounds__(256) ht_fwd_kernel(const float* __restrict__ W, const float* __restrict__ bias,
                                                     const float* __restrict__ x, const float* __restrict__ skip,
                                                     float* __restrict__ z, float* __restrict__ out, int B, int OUT,
                                                     DropoutCfg dc, int site) {
  const int o = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (o >= OUT) return;
  constexpr int V = IN / 128;
  float4 w[V];
#pragma unroll
  for (int v = 0; v < V; ++v) w[v] = __ldg(reinterpret_cast<const float4*>(W + (long long)o * IN) + lane + 32 * v);
  const float bo = __ldg(bias + o);
  const int b_lo = blockIdx.y * 32, b_hi = min(B, b_lo + 32);
  for (int b = b_lo; b < b_hi; ++b) {
    float a = 0.f;
#pragma unroll
    for (int v = 0; v < V; ++v) {
      const float4 xv = reinterpret_cast<const float4*>(x + (long long)b * IN)[lane + 32 * v];
      a += w[v].x * xv.x + w[v].y * xv.y + w[v].z * xv.z + w[v].w * xv.w;
    }
    for (int s = 16; s > 0; s >>= 1) a += __shfl_xor_sync(0xffffffffu, a, s);
    if (lane == 0) {
      a += bo;
      const long long i = (long long)b * OUT + o;
      if (MODE == 0) {
        z[i] = a;
        const bool keep = dc.thr == 0 || dropout_keep(dc.seed, dc.step, (uint32_t)site, (uint32_t)b, (uint32_t)o, dc.thr);
        out[i] = keep ? ht_gelu(a) * dc.scale : 0.f;
      } else if (MODE == 1) {
        out[i] = a + skip[i];
      } else {
        out[i] = a;
      }
    }
  }
}

// Mean cross-entropy over the batch (F.cross_entropy, reduction="mean") and its gradient d loss / d logits
// = (softmax(logits) - onehot(target)) / B.  One block; targets are 0 / 1.
__global__ void __launch_bounds__(256) ht_loss_kernel(const float* __restrict__ logits, const int64_t* __restrict__ target,
                                                      float* __restrict__ dlogits, float* __restrict__ loss_out, int B) {
  __shared__ float red[8];
  float acc = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    const float l0 = logits[2 * b], l1 = logits[2 * b + 1];
    const float m = fmaxf(l0, l1);
    const float e0 = expf(l0 - m), e1 = expf(l1 - m);
    const float lse = m + logf(e0 + e1);
    const int y = target[b] != 0 ? 1 : 0;
    acc += lse - (y ? l1 : l0);
    const float inv = 1.0f / (e0 + e1);
    dlogits[2 * b] = (e0 * inv - (y == 0 ? 1.f : 0.f)) / (float)B;
    dlogits[2 * b + 1] = (e1 * inv - (y == 1 ? 1.f : 0.f)) / (float)B;
  }
  for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += red[i];
    if (loss_out) *loss_out = t / (float)B;
  }
}

constexpr int HT_RB = 8;   // reads per block in ht_bwd_x_kernel

// dx[b,i] = sum_o W[o,i] dy[b,o] (+ add[b,i]); with z != null the result is the gradient of the pre-activation of the layer
// below: dx * keep(site, b, i) * scale * GELU'(z[b,i]).  grid (IN / 256, ceil(B / 8)); dy rows staged in shared memory.
__global__ void __launch_bounds__(256) ht_bwd_x_kernel(const float* __restrict__ W, const float* __restrict__ dy,
                                                       const float* __restrict__ add, const float* __restrict__ z,
                                                       float* __restrict__ dx, int B, int OUT, int IN, DropoutCfg dc, int site) {
  __shared__ float s_dy[HT_RB][512];
  const int i = blockIdx.x * 256 + threadIdx.x, b0 = blockIdx.y * HT_RB;
  const int nb = min(HT_RB, B - b0);
  for (int k = threadIdx.x; k < nb * OUT; k += 256) s_dy[k / OUT][k % OUT] = dy[(long long)(b0 + k / OUT) * OUT + k % OUT];
  __syncthreads();
  if (i >= IN) return;
  float acc[HT_RB];
#pragma unroll
  for (int r = 0; r < HT_RB; ++r) acc[r] = 0.f;
  for (int o = 0; o < OUT; ++o) {
    const float w = __ldg(W + (long long)o * IN + i);
#pragma unroll
    for (int r = 0; r < HT_RB; ++r) acc[r] = fmaf(w, s_dy[r][o], acc[r]);
  }
#pragma unroll
  for (int r = 0; r < HT_RB; ++r) {
    if (r >= nb) break;
    const int b = b0 + r;
    const long long j = (long long)b * IN + i;
    float g = acc[r] + (add ? add[j] : 0.f);
    if (z) {
      const bool keep = dc.thr == 0 || dropout_keep(dc.seed, dc.step, (uint32_t)site, (uint32_t)b, (uint32_t)i, dc.thr);
      g = keep ? g * dc.scale * ht_gelu_grad(z[j]) : 0.f;
    }
    dx[j] = g;
  }
}

// dW[o,i] = sum_b dy[b,o] x[b,i], db[o] = sum_b dy[b,o] (fixed summation order: deterministic).  grid (ceil(IN / 256), OUT).
__global__ void __launch_bounds__(256) ht_bwd_w_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                                       float* __restrict__ dW, float* __restrict__ db, int B, int OUT, int IN) {
  const int o = blockIdx.y, i = blockIdx.x * 256 + threadIdx.x;
  if (i < IN) {
    float a = 0.f;
    for (int b = 0; b < B; ++b) a = fmaf(dy[(long long)b * OUT + o], x[(long long)b * IN + i], a);
    dW[(long long)o * IN + i] = a;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    float s = 0.f;
    for (int b = 0; b < B; ++b) s += dy[(long long)b * OUT + o];
    db[o] = s;
  }
}

// ---------------------------------------------------------------------------------------------
// Pooling backward, per read (one block, thread = channel c):  pooled = sum_t w_t h_t with h_t = xn_t * g + beta, so
//   ds_t = w_t (h_t . dp - pooled . dp) = w_t (xn_t . (g * dp) + (beta - pooled) . dp)
// rd[b] = (M, 1 / L, (beta - pooled) . dp) with M, L the softmax max and normaliser merged from the forward's per-tile
// partials exactly as head_fused_kernel merges them; gdp[b] = g * dp.
__global__ void __launch_bounds__(256) ht_pool_prep_kernel(const float* __restrict__ part, int n_split,
                                                           const float* __restrict__ pooled, const float* __restrict__ dpooled,
                                                           const float* __restrict__ g, const float* __restrict__ beta,
                                                           float* __restrict__ rd, float* __restrict__ gdp) {
  constexpr int D = 256;
  __shared__ float red[8];
  const int b = blockIdx.x, c = threadIdx.x;
  const float* pp = part + (long long)b * n_split * (2 + D);
  float M = -INFINITY;
  for (int s = 0; s < n_split; ++s) M = fmaxf(M, pp[s * (2 + D)]);
  float L = 0.f;
  for (int s = 0; s < n_split; ++s) {
    const float ms = pp[s * (2 + D)];
    L += pp[s * (2 + D) + 1] * ((ms == -INFINITY) ? 0.f : __expf(ms - M));
  }
  const float dp = dpooled[(long long)b * D + c];
  gdp[(long long)b * D + c] = g[c] * dp;
  float t = (beta[c] - pooled[(long long)b * D + c]) * dp;
  for (int s = 16; s > 0; s >>= 1) t += __shfl_xor_sync(0xffffffffu, t, s);
  if ((c & 31) == 0) red[c >> 5] = t;
  __syncthreads();
  if (c == 0) {
    float cst = 0.f;
    for (int i = 0; i < 8; ++i) cst += red[i];
    rd[4 * b] = M; rd[4 * b + 1] = 1.0f / L; rd[4 * b + 2] = cst; rd[4 * b + 3] = 0.f;
  }
}

// ---------------------------------------------------------------------------------------------
// Scorer + pooling backward on the tensor cores.  With z_t = W0' xn_t + b0' (ln_f's affine folded in, the forward's
// att0_wf / att0_bf), a_t = GELU(z_t), s_t = w2 . a_t + b2:
//   dz_t[o] = ds_t w2[o] GELU'(z_t[o]);  dW2 = sum_t ds_t a_t;  db2 = sum_t ds_t;  db0 = sum_t dz_t
//   dW0 = sum_t dz_t (x) h_t = (sum_t dz_t (x) xn_t) diag(g) + db0 (x) beta
// CTA pairs split W0's 256 output rows into halves of 128 (blockIdx.x & 1) and walk the token tiles of the forward
// (128 tokens of one read; the rows past T are TMA zero fill and get ds = 0).  Per tile:
//   MMA1  Z[t][o]  = xn_tile (K-major, 128 x 256) * W0'_half^T (K-major, 128 x 256)      TMEM columns   0..127
//   epilogue (4 warps, thread = token row): ds_t from the score, the read's (M, 1/L) and xn_t . (g dp) taken from the
//         staged tile; dz_t (bf16, MN-major in shared memory), per-column sums of dz and ds a (warp reduce-scatter)
//   MMA2  G[o][c] += dz^T (MN-major, 128 o x 128 t) * xn (MN-major: the same swizzled tile, 256 c x 128 t)   128..383
// One tile at a time (load -> MMA1 -> epilogue -> MMA2): the backward runs once per training step, not per read.  At the
// end G and the column sums go to per-CTA partials that score_bwd_reduce_kernel adds up in a fixed order.
struct ScoreBwdParams {
  const float* b0f;    // [256] folded scorer bias
  const float* w2;     // [256] attention.2.weight
  const float* score;  // [B*T] scores of the forward
  const float* rd;     // [B][4] (M, 1/L, cst, -)
  const float* gdp;    // [B][256]
  float* part_dw;      // [grid][128][256]
  float* part_vec;     // [grid][3][128]: sum dz, sum ds a, (sum ds, 0, ...)
  int B, T, tiles_per_seq, num_tiles;
};

namespace sb {
constexpr int BM = 128, BK = 64, HALF = 128;
constexpr int KB_BYTES = BM * BK * 2;          // 16 KB: [128 rows x 64 bf16]
constexpr int OFF_W = 0;                       // W0' half: 4 k-blocks [128 o x 64 c]
constexpr int OFF_X = OFF_W + 4 * KB_BYTES;    // xn tile: 4 k-blocks [128 t x 64 c]
constexpr int OFF_DZ = OFF_X + 4 * KB_BYTES;   // dz: 2 atoms [128 t x 64 o]
constexpr int OFF_BAR = OFF_DZ + 2 * KB_BYTES;
constexpr int OFF_F = OFF_BAR + 128;           // b0[128] w2[128] gdp[256] red[4][3][128]
constexpr int SMEM_TOTAL = OFF_F + (128 + 128 + 256 + 4 * 3 * 128) * 4;
constexpr int THREADS = 192;                   // warp 0 TMA, warp 1 MMA, warps 2..5 epilogue
constexpr int TM_Z = 0, TM_G = 128;
}  // namespace sb

// kind::f16, bf16 x bf16 -> fp32, A and B both MN-major (bits 15 and 16)
__host__ __device__ constexpr uint32_t idesc_bf16_f32_mnmn(uint32_t M, uint32_t N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// 32 per-lane values v[j] -> lane j holds sum over the warp of v[j] (31 shuffles instead of 32 x 5)
__device__ __forceinline__ float warp_reduce_scatter32(float (&v)[32], int lane) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    const bool upper = (lane & off) != 0;
#pragma unroll
    for (int k = 0; k < off; ++k) {
      const float send = upper ? v[k] : v[k + off];
      const float keep = upper ? v[k + off] : v[k];
      v[k] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  return v[0];
}

__global__ void __launch_bounds__(sb::THREADS, 1)
score_bwd_kernel(const __grid_constant__ CUtensorMap tmXN, const __grid_constant__ CUtensorMap tmW, ScoreBwdParams p) {
  using namespace sb;
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((ptx::smem_u32(smem) & 1023u) != 0) __trap();
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
  uint64_t* w_full = bars;        // W0' half landed
  uint64_t* a_full = bars + 1;    // xn tile landed
  uint64_t* z_full = bars + 2;    // MMA1 complete
  uint64_t* dz_full = bars + 3;   // dz written (4 warp arrivals)
  uint64_t* g_done = bars + 4;    // MMA2 complete: xn tile and dz may be overwritten
  uint64_t* fin = bars + 5;       // every MMA of this CTA complete
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 6);
  float* s_b0 = reinterpret_cast<float*>(smem + OFF_F);
  float* s_w2 = s_b0 + 128;
  float* s_gdp = s_w2 + 128;
  float* s_red = s_gdp + 256;     // [4 warps][3][128]
  const int half = blockIdx.x & 1, pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  for (int i = threadIdx.x; i < 128; i += THREADS) {
    s_b0[i] = __ldg(p.b0f + half * HALF + i);
    s_w2[i] = __ldg(p.w2 + half * HALF + i);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmXN); ptx::prefetch_tmap(&tmW);
    ptx::mbar_init(w_full, 1); ptx::mbar_init(a_full, 1); ptx::mbar_init(z_full, 1);
    ptx::mbar_init(dz_full, 4); ptx::mbar_init(g_done, 1); ptx::mbar_init(fin, 1);
    ptx::fence_mbar_init();
  } else if (warp == 1) {
    ptx::tmem_alloc<512>(tmem_ptr);
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    if (lane == 0) {
      ptx::mbar_expect_tx(w_full, 4 * KB_BYTES);
      for (int kb = 0; kb < 4; ++kb) ptx::tma_load_2d(smem + OFF_W + kb * KB_BYTES, &tmW, w_full, kb * BK, half * HALF);
      uint32_t it = 0;
      for (int tile = pair; tile < p.num_tiles; tile += n_pairs, ++it) {
        const int b = tile / p.tiles_per_seq, t0 = (tile % p.tiles_per_seq) * BM;
        if (it > 0) ptx::mbar_wait(g_done, (it - 1) & 1);
        ptx::mbar_expect_tx(a_full, 4 * KB_BYTES);
        for (int kb = 0; kb < 4; ++kb) ptx::tma_load_3d(smem + OFF_X + kb * KB_BYTES, &tmXN, a_full, kb * BK, t0, b);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc1 = ptx::idesc_bf16_f32(BM, HALF);
      constexpr uint32_t idesc2 = idesc_bf16_f32_mnmn(HALF, 256);
      const uint32_t sW = ptx::smem_u32(smem + OFF_W), sX = ptx::smem_u32(smem + OFF_X), sDZ = ptx::smem_u32(smem + OFF_DZ);
      ptx::mbar_wait(w_full, 0);
      uint32_t it = 0;
      for (int tile = pair; tile < p.num_tiles; tile += n_pairs, ++it) {
        ptx::mbar_wait(a_full, it & 1);
        ptx::tc_fence_after_sync();
        for (int kb = 0; kb < 4; ++kb) {
          const uint64_t da = ptx::smem_desc_k_sw128(sX + kb * KB_BYTES), db = ptx::smem_desc_k_sw128(sW + kb * KB_BYTES);
#pragma unroll
          for (int k = 0; k < 4; ++k) ptx::umma_f16(tmem_base + TM_Z, da + 2 * k, db + 2 * k, idesc1, (kb | k) != 0);
        }
        ptx::umma_commit(z_full);
        ptx::mbar_wait(dz_full, it & 1);
        ptx::tc_fence_after_sync();
        // A = dz^T: M = o in 2 atoms of 64 (16 KB apart), K = tokens in rows of 128 B; B = xn: N = c in 4 atoms of 64
        // (the k-blocks of the tile, 16 KB apart), K = tokens.  16 K-rows (2 KB) per MMA.
        const uint64_t da = ptx::smem_desc_mn_sw128(sDZ, KB_BYTES, 1024), db = ptx::smem_desc_mn_sw128(sX, KB_BYTES, 1024);
#pragma unroll
        for (int ks = 0; ks < BM / 16; ++ks)
          ptx::umma_f16(tmem_base + TM_G, da + (2048 >> 4) * ks, db + (2048 >> 4) * ks, idesc2, (it | ks) != 0);
        ptx::umma_commit(g_done);
      }
      ptx::umma_commit(fin);
    }
  } else {
    const int q = warp & 3, e = warp - 2;   // TMEM lane quarter of this warp
    const int r = q * 32 + lane;            // token row of the tile; o row of G at the end
    const uint32_t lane_addr = tmem_base + (uint32_t(q * 32) << 16);
    float acc_dz[4] = {0.f, 0.f, 0.f, 0.f}, acc_da[4] = {0.f, 0.f, 0.f, 0.f}, acc_ds = 0.f;
    uint32_t it = 0;
    for (int tile = pair; tile < p.num_tiles; tile += n_pairs, ++it) {
      const int b = tile / p.tiles_per_seq, t0 = (tile % p.tiles_per_seq) * BM;
      const int valid = min(BM, p.T - t0);
      ptx::bar_sync(1, 128);   // the previous tile's gdp has been used by every thread
      s_gdp[e * 32 + lane] = p.gdp[(long long)b * 256 + e * 32 + lane];
      s_gdp[128 + e * 32 + lane] = p.gdp[(long long)b * 256 + 128 + e * 32 + lane];
      ptx::bar_sync(1, 128);
      ptx::mbar_wait(z_full, it & 1);   // implies the tile landed and the previous MMA2 finished (dz buffer free)
      ptx::tc_fence_after_sync();
      // ---- ds_t
      float ds = 0.f;
      if (r < valid) {
        float dot = 0.f;
        const uint8_t* row = smem + OFF_X + r * 128;
#pragma unroll
        for (int kb = 0; kb < 4; ++kb)
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const uint4 v = *reinterpret_cast<const uint4*>(row + kb * KB_BYTES + ((j ^ (r & 7)) << 4));
            const uint32_t w[4] = {v.x, v.y, v.z, v.w};
            const float* gg = s_gdp + kb * 64 + j * 8;
#pragma unroll
            for (int u = 0; u < 4; ++u)
              dot += __uint_as_float(w[u] << 16) * gg[2 * u] + __uint_as_float(w[u] & 0xffff0000u) * gg[2 * u + 1];
          }
        const float M = p.rd[4 * b], invL = p.rd[4 * b + 1], cst = p.rd[4 * b + 2];
        const float wt = __expf(p.score[(long long)b * p.T + t0 + r] - M) * invL;
        ds = wt * (dot + cst);
      }
      {
        float t = ds;
        for (int s = 16; s > 0; s >>= 1) t += __shfl_xor_sync(0xffffffffu, t, s);
        acc_ds += t;
      }
      // ---- dz, column sums
#pragma unroll 1
      for (int ci = 0; ci < 4; ++ci) {
        uint32_t a[32];
        ptx::tmem_ld_32x32b_x32(lane_addr + TM_Z + ci * 32, a);
        ptx::tmem_ld_wait();
        float vz[32], va[32];
        uint32_t pk[16];
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const int o = ci * 32 + j;
          const float zz = __uint_as_float(a[j]) + s_b0[o];
          const float dz = ds * s_w2[o] * ht_gelu_grad(zz);
          va[j] = ds * ht_gelu(zz);
          const __nv_bfloat16 h = __float2bfloat16(dz);
          vz[j] = dz;
          const uint32_t hb = *reinterpret_cast<const unsigned short*>(&h);
          if (j & 1) pk[j >> 1] |= hb << 16; else pk[j >> 1] = hb;
        }
        // dz[t = r][o]: atom o / 64, 16-byte chunk (o % 64) / 8 swizzled with the row
        uint8_t* dzrow = smem + OFF_DZ + (ci >> 1) * KB_BYTES + r * 128;
#pragma unroll
        for (int c8 = 0; c8 < 4; ++c8) {
          const int chunk = (ci & 1) * 4 + c8;
          *reinterpret_cast<uint4*>(dzrow + ((chunk ^ (r & 7)) << 4)) =
              make_uint4(pk[4 * c8], pk[4 * c8 + 1], pk[4 * c8 + 2], pk[4 * c8 + 3]);
        }
        acc_dz[ci] += warp_reduce_scatter32(vz, lane);
        acc_da[ci] += warp_reduce_scatter32(va, lane);
      }
      ptx::fence_proxy_async_smem();   // generic-proxy dz stores -> the MMA (async proxy) reads them
      ptx::tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(dz_full);
    }
    // ---- drain G (row o = r of this half, 256 columns c) and the column sums
    float* dst = p.part_dw + ((long long)blockIdx.x * HALF + r) * 256;
    if (it > 0) {
      ptx::mbar_wait(fin, 0);
      ptx::tc_fence_after_sync();
#pragma unroll 1
      for (int ci = 0; ci < 8; ++ci) {
        uint32_t a[32];
        ptx::tmem_ld_32x32b_x32(lane_addr + TM_G + ci * 32, a);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          *reinterpret_cast<float4*>(dst + ci * 32 + j) = make_float4(__uint_as_float(a[j]), __uint_as_float(a[j + 1]),
                                                                       __uint_as_float(a[j + 2]), __uint_as_float(a[j + 3]));
      }
    } else {
      for (int c = 0; c < 256; ++c) dst[c] = 0.f;
    }
#pragma unroll
    for (int ci = 0; ci < 4; ++ci) {
      s_red[(q * 3 + 0) * 128 + ci * 32 + lane] = acc_dz[ci];
      s_red[(q * 3 + 1) * 128 + ci * 32 + lane] = acc_da[ci];
    }
    s_red[(q * 3 + 2) * 128 + lane] = lane == 0 ? acc_ds : 0.f;
    ptx::bar_sync(1, 128);
    float* pv = p.part_vec + (long long)blockIdx.x * 3 * 128;
    for (int k = 0; k < 3; ++k) {
      float s = 0.f;
      for (int qq = 0; qq < 4; ++qq) s += s_red[(qq * 3 + k) * 128 + r];   // fixed order
      pv[k * 128 + r] = s;
    }
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after_sync();
    ptx::tmem_dealloc<512>(tmem_base);
  }
}

// Partials of the score_bwd_kernel CTAs -> gradients (grid 256 = o, thread = c):
//   dW0[o][c] = g[c] sum_cta G_cta[o][c] + beta[c] db0[o];  db0[o] = sum_cta sum dz;  dW2[o] = sum_cta sum ds a;  db2 = sum ds
__global__ void __launch_bounds__(256) score_bwd_reduce_kernel(const float* __restrict__ part_dw, const float* __restrict__ part_vec,
                                                               int n_cta, const float* __restrict__ g, const float* __restrict__ beta,
                                                               float* __restrict__ dW0, float* __restrict__ db0,
                                                               float* __restrict__ dW2, float* __restrict__ db2) {
  const int o = blockIdx.x, c = threadIdx.x, half = o >> 7, ol = o & 127;
  float s = 0.f, sdz = 0.f, sda = 0.f;
  for (int k = half; k < n_cta; k += 2) {
    s += part_dw[((long long)k * 128 + ol) * 256 + c];
    sdz += part_vec[(long long)k * 384 + ol];
    sda += part_vec[(long long)k * 384 + 128 + ol];
  }
  dW0[(long long)o * 256 + c] = g[c] * s + beta[c] * sdz;
  if (c == 0) { db0[o] = sdz; dW2[o] = sda; }
  if (o == 0 && c == 0) {
    float t = 0.f;
    for (int k = 0; k < n_cta; k += 2) t += part_vec[(long long)k * 384 + 256];
    *db2 = t;
  }
}

// ---------------------------------------------------------------------------------------------
// torch.optim.AdamW (single-tensor form):  p *= 1 - lr wd;  m = b1 m + (1 - b1) g;  v = b2 v + (1 - b2) g^2;
//   p -= (lr / (1 - b1^t)) m / (sqrt(v) / sqrt(1 - b2^t) + eps)
// over all head tensors at once (one flat buffer).  t is a device counter that adamw_step_kernel advances after the update,
// so the step number stays right without the host knowing whether a step was applied: when the forward of this step
// reported a bad status (a token id out of range, the fp16 convolution out of its range) nothing is updated.
struct AdamWParams {
  float* p; float* m; float* v; const float* g;
  long long n;
  float lr, beta1, beta2, eps, wd;
  int* step;               // device step counter (steps applied so far)
  const int* status;       // the forward's published status word (mapped host memory), low byte = error bits
};

__global__ void __launch_bounds__(256) adamw_kernel(AdamWParams a) {
  __shared__ float s_c[2];
  __shared__ int s_skip;
  if (threadIdx.x == 0) {
    const int st = *reinterpret_cast<const volatile int*>(a.status);
    s_skip = (st & 0xff) != 0;
    const int t = *a.step + 1;
    s_c[0] = (float)((double)a.lr / (1.0 - pow((double)a.beta1, (double)t)));   // step size
    s_c[1] = (float)sqrt(1.0 - pow((double)a.beta2, (double)t));                // sqrt of bias correction 2
  }
  __syncthreads();
  if (s_skip) return;
  const float step_size = s_c[0], bc2s = s_c[1];
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += (long long)gridDim.x * blockDim.x) {
    const float g = a.g[i];
    float p = a.p[i] * (1.0f - a.lr * a.wd);
    const float m = a.m[i] + (1.0f - a.beta1) * (g - a.m[i]);   // exp_avg.lerp_(grad, 1 - beta1)
    const float v = a.v[i] * a.beta2 + (1.0f - a.beta2) * g * g;
    p -= step_size * m / (sqrtf(v) / bc2s + a.eps);
    a.p[i] = p; a.m[i] = m; a.v[i] = v;
  }
}

// advances the device step counter once every block of adamw_kernel has read it (same condition as the update)
__global__ void adamw_step_kernel(int* step, const int* status) {
  if ((*reinterpret_cast<const volatile int*>(status) & 0xff) == 0) *step += 1;
}

}  // namespace clm
