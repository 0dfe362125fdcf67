// Fine-tuning of the last block's tail (out_proj, residual, norm2, fc1, GELU-tanh, fc2, residual) and ln_f together with
// the head (clm_tail_train_begin; DESIGN.md §4.8 "Training the last block's tail").  Everything upstream of the tail is
// frozen, so the forward leaves the tail's inputs in place: R holds block L's input residual r0 (the last block does not
// store its own, skip_dead_res) and Y its conv output y.  Per row t (all B*T rows, [PAD] rows included):
//   r1 = r0 + Wo y + bo;  n1 = (r1 - mu1) rho1;  x2 = g2 n1 + beta2;  h = W1 x2 + b1;  a = gelu_tanh(h)
//   r2 = r1 + W2 a + b2;  n2 = (r2 - mu2) rho2;  hid = gf n2 + betaf
// and backward from the head's dhid = w dp + W0^T dz:
//   dr2 = rho2 (dn2 - mean(dn2) - n2 mean(dn2 n2)), dn2 = gf dhid      (EPI_TAIL_DHID, on dz . W0)
//   dh  = (W2^T dr2) gelu_tanh'(h)                                      (EPI_TAIL_DH,   on dr2 . W2)
//   dr1 = dr2 + rho1 (dn1 - mean(dn1) - n1 mean(dn1 n1)), dn1 = g2 dx2, dx2 = W1^T dh   (EPI_TAIL_DR1, on dh . W1)
//   dW2 = sum dr2 a^T, dW1 = sum dh x2^T, dWo = sum dr1 y^T               (tail_wgrad_kernel)
//   dgf = sum dhid n2, dbetaf = sum dhid, db2 = sum dr2, db1 = sum dh, dg2 = sum dx2 n1, dbeta2 = sum dx2, dbo = sum dr1
// The column sums come from the dgrad epilogues as per-warp partials that colsum_reduce_kernel adds in a fixed order, and
// the weight gradients from split-K partials that wgrad_reduce_kernel adds in a fixed order: gradients are bit-reproducible.
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

#include "gemm_tcgen05.cuh"
#include "head_train.cuh"
#include "ptx.cuh"

namespace clm {

__device__ __forceinline__ float gelu_tanh_grad_f(float x) {
  const float k0 = 0.7978845608028654f, k1 = 0.044715f;
  const float t = tanhf(k0 * (x + k1 * x * x * x));
  return 0.5f * (1.0f + t) + 0.5f * x * (1.0f - t * t) * k0 * (1.0f + 3.0f * k1 * x * x);
}

// 8 bf16 (16 bytes) -> floats
__device__ __forceinline__ void bf16x8_to_f32(uint4 u, float* f) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    f[2 * i] = __uint_as_float(w[i] << 16);
    f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
}

// v[32] of this thread's row -> lane j adds the warp's column sum of v[j] into colsum[(group * nvec + k) * N + n + j]:
// one partial per (row tile, TMEM lane quarter), so that the reduction order is fixed
__device__ __forceinline__ void tail_colsum_store(float (&v)[32], int lane, float* colsum, long long slot, int N, int n) {
  const float s = warp_reduce_scatter32(v, lane);
  colsum[slot * N + n + lane] = s;
}

// The dgrad epilogues of gemm_bf16_tn_kernel (warps 2..5, thread = output row; TMEM holds the 128 x BN accumulator).
template <int BN, int EPI>
__device__ void gemm_tail_epilogue(const GemmParams& p, uint32_t tmem_base, int m0, int n0, int q, int lane) {
  const long long row = (long long)m0 + q * 32 + lane;
  const bool row_ok = row < p.M;
  const uint32_t taddr = tmem_base + (uint32_t(q * 32) << 16);
  const long long group = (long long)(m0 / GEMM_BM) * 4 + q;
  __nv_bfloat16* out = reinterpret_cast<__nv_bfloat16*>(p.out);
  if constexpr (EPI == EPI_TAIL_DH) {
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      uint32_t r[32];
      ptx::tmem_ld_32x32b_x32(taddr + c0, r);
      ptx::tmem_ld_wait();
      const int n = n0 + c0;
      float v[32];
      if (row_ok) {
        const uint4* hp = reinterpret_cast<const uint4*>(p.aux + row * p.ldo + n);
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
          float h[8];
          bf16x8_to_f32(hp[j / 8], h);
#pragma unroll
          for (int u = 0; u < 8; ++u) v[j + u] = __uint_as_float(r[j + u]) * gelu_tanh_grad_f(h[u]);
        }
        uint4* o = reinterpret_cast<uint4*>(out + row * p.ldo + n);
#pragma unroll
        for (int j = 0; j < 32; j += 8)
          o[j / 8] = make_uint4(pack_bf16(v[j], v[j + 1]), pack_bf16(v[j + 2], v[j + 3]), pack_bf16(v[j + 4], v[j + 5]),
                                pack_bf16(v[j + 6], v[j + 7]));
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = 0.f;
      }
      tail_colsum_store(v, lane, p.colsum, group, p.N, n);
    }
  } else {
    // EPI_TAIL_DHID / EPI_TAIL_DR1: a LayerNorm backward over the whole 256-column row (BN == N == 256), two sweeps of TMEM
    static_assert(BN == 256, "the LayerNorm backward epilogues own whole rows");
    constexpr bool DHID = EPI == EPI_TAIL_DHID;
    float wt = 0.f, rho = 0.f;
    const float* dp = nullptr;
    if (row_ok) {
      rho = p.rho[row];
      if constexpr (DHID) {   // softmax weight of the row in its read, as score_bwd_kernel forms it
        const long long b = row / p.T;
        wt = __expf(p.score_in[row] - p.rd[4 * b]) * p.rd[4 * b + 1];
        dp = p.dp + b * 256;
      }
    }
    const __nv_bfloat16* nrow = p.nrm + row * 256;
    float s1 = 0.f, s2 = 0.f;
#pragma unroll 1
    for (int c0 = 0; c0 < 256; c0 += 32) {
      uint32_t r[32];
      ptx::tmem_ld_32x32b_x32(taddr + c0, r);
      ptx::tmem_ld_wait();
      if (row_ok) {
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
          float nv[8];
          bf16x8_to_f32(*reinterpret_cast<const uint4*>(nrow + c0 + j), nv);
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int c = c0 + j + u;
            float d = __uint_as_float(r[j + u]);
            if constexpr (DHID) d = fmaf(wt, __ldg(dp + c), d);
            const float dn = __ldg(p.gam + c) * d;
            s1 += dn;
            s2 = fmaf(dn, nv[u], s2);
          }
        }
      }
    }
    const float m1 = s1 * (1.0f / 256.0f), m2 = s2 * (1.0f / 256.0f);
#pragma unroll 1
    for (int c0 = 0; c0 < 256; c0 += 32) {
      uint32_t r[32];
      ptx::tmem_ld_32x32b_x32(taddr + c0, r);
      ptx::tmem_ld_wait();
      float va[32], vb[32], vc[32];   // d (dhid / dx2) * n, d, the row's output gradient (dr2 / dr1)
      if (row_ok) {
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
          float nv[8], add[8];
          bf16x8_to_f32(*reinterpret_cast<const uint4*>(nrow + c0 + j), nv);
          if constexpr (!DHID) bf16x8_to_f32(*reinterpret_cast<const uint4*>(p.aux + row * 256 + c0 + j), add);   // dr2
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int c = c0 + j + u;
            float d = __uint_as_float(r[j + u]);
            if constexpr (DHID) d = fmaf(wt, __ldg(dp + c), d);
            const float dn = __ldg(p.gam + c) * d;
            float g = rho * (dn - m1 - nv[u] * m2);
            if constexpr (!DHID) g += add[u];
            va[j + u] = d * nv[u];
            vb[j + u] = d;
            vc[j + u] = g;
          }
        }
        uint4* o = reinterpret_cast<uint4*>(out + row * 256 + c0);
#pragma unroll
        for (int j = 0; j < 32; j += 8)
          o[j / 8] = make_uint4(pack_bf16(vc[j], vc[j + 1]), pack_bf16(vc[j + 2], vc[j + 3]), pack_bf16(vc[j + 4], vc[j + 5]),
                                pack_bf16(vc[j + 6], vc[j + 7]));
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) va[j] = vb[j] = vc[j] = 0.f;
      }
      tail_colsum_store(va, lane, p.colsum, group * 3 + 0, 256, c0);
      tail_colsum_store(vb, lane, p.colsum, group * 3 + 1, 256, c0);
      tail_colsum_store(vc, lane, p.colsum, group * 3 + 2, 256, c0);
    }
  }
}

// dst_k[c] = sum over groups g (in order, then a fixed tree) of part[(g * nvec + k) * N + c]; grid nvec * N, block 256
__global__ void __launch_bounds__(256) colsum_reduce_kernel(const float* __restrict__ part, int n_groups, int nvec, int N,
                                                            float* dst0, float* dst1, float* dst2) {
  __shared__ float red[256];
  const int k = blockIdx.x / N, c = blockIdx.x % N;
  float s = 0.f;
  for (int g = threadIdx.x; g < n_groups; g += 256) s += part[((long long)g * nvec + k) * N + c];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if ((int)threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) (k == 0 ? dst0 : k == 1 ? dst1 : dst2)[c] = red[0];
}

// LayerNorm statistics of the fp32 residual rows (R32 layout): n = (r - mu) rho as bf16 [M,256], rho [M], and with g != null
// also x = g n + beta as bf16.  One warp per row, biased variance (torch.nn.functional.layer_norm).
__global__ void __launch_bounds__(256) tail_ln_kernel(const float* __restrict__ R, const float* __restrict__ g,
                                                      const float* __restrict__ beta, __nv_bfloat16* __restrict__ n_out,
                                                      __nv_bfloat16* __restrict__ x_out, float* __restrict__ rho_out,
                                                      long long M, float eps) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= M) return;
  const int ca = 4 * lane, cb = 128 + 4 * lane;
  const float4 a = *reinterpret_cast<const float4*>(R + ptx::r32_off(row, ca));
  const float4 b = *reinterpret_cast<const float4*>(R + ptx::r32_off(row, cb));
  float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) s += v[i];
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mu = s * (1.0f / 256.0f);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) q += (v[i] - mu) * (v[i] - mu);
  for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  const float rho = rsqrtf(q * (1.0f / 256.0f) + eps);
  if (lane == 0) rho_out[row] = rho;
  float n[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) n[i] = (v[i] - mu) * rho;
  uint2* nr = reinterpret_cast<uint2*>(n_out + row * 256);
  nr[lane] = make_uint2(pack_bf16(n[0], n[1]), pack_bf16(n[2], n[3]));
  nr[32 + lane] = make_uint2(pack_bf16(n[4], n[5]), pack_bf16(n[6], n[7]));
  if (x_out) {
    float x[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int c = i < 4 ? ca + i : cb + i - 4;
      x[i] = fmaf(__ldg(g + c), n[i], __ldg(beta + c));
    }
    uint2* xr = reinterpret_cast<uint2*>(x_out + row * 256);
    xr[lane] = make_uint2(pack_bf16(x[0], x[1]), pack_bf16(x[2], x[3]));
    xr[32 + lane] = make_uint2(pack_bf16(x[4], x[5]), pack_bf16(x[6], x[7]));
  }
}

// dst[c][r] = bf16(src[r][c]): the per-step K-major copies of W0, W2, W1 that the dgrad GEMMs take as B.  grid (C/32, R/32)
__global__ void __launch_bounds__(256) transpose_f32_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst,
                                                                 int R, int C) {
  __shared__ float s[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32, tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int i = ty; i < 32; i += 8) s[i][tx] = src[(long long)(r0 + i) * C + c0 + tx];
  __syncthreads();
  for (int i = ty; i < 32; i += 8) dst[(long long)(c0 + i) * R + r0 + tx] = __float2bfloat16(s[tx][i]);
}

// ---------------------------------------------------------------------------------------------
// Weight gradient C[o][i] = sum_t A[t][o] B[t][i] over the M token rows (K = tokens), both operands token-major bf16, so
// both are MN-major UMMA operands (as score_bwd_kernel's second MMA).  One CTA per (128 o) x (256 i) output tile and split
// of the token chunks; per 128-token chunk TMA brings A as 2 atoms [128 t x 64 o] and B as 4 atoms [128 t x 64 i] (rows
// past M are zero fill), and 8 MMAs of 16 tokens accumulate into 256 TMEM columns.  The CTA's tile goes to
// part[split][O][I]; wgrad_reduce_kernel adds the splits in order.
struct WgradParams {
  float* part;        // [n_split][O][I]
  int O, I;
  int n_chunks;       // ceil(M / 128)
  int chunks_per_split;
};

namespace tw {
constexpr int KT = 128;
constexpr int ATOM = KT * 64 * 2;             // 16 KB
constexpr int A_BYTES = 2 * ATOM, B_BYTES = 4 * ATOM;
constexpr int STAGE = A_BYTES + B_BYTES;      // 96 KB
constexpr int STAGES = 2;
constexpr int OFF_BAR = STAGES * STAGE;
constexpr int SMEM_TOTAL = OFF_BAR + 128 + 1024;   // barriers + alignment slack
constexpr int THREADS = 192;                       // warp 0 TMA, warp 1 MMA, warps 2..5 epilogue
}  // namespace tw

__global__ void __launch_bounds__(tw::THREADS, 1)
tail_wgrad_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, WgradParams p) {
  using namespace tw;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
  uint64_t* empty = full + STAGES;
  uint64_t* done = empty + STAGES;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(done + 1);
  const int ib = blockIdx.x, ob = blockIdx.y, split = blockIdx.z;
  const int o0 = ob * 128, i0 = ib * 256;
  const int k_lo = split * p.chunks_per_split, k_hi = min(p.n_chunks, k_lo + p.chunks_per_split);
  const int nk = max(0, k_hi - k_lo);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmA); ptx::prefetch_tmap(&tmB);
    for (int s = 0; s < STAGES; ++s) { ptx::mbar_init(&full[s], 1); ptx::mbar_init(&empty[s], 1); }
    ptx::mbar_init(done, 1);
    ptx::fence_mbar_init();
  } else if (warp == 1) {
    ptx::tmem_alloc<256>(tmem_ptr);
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    if (lane == 0) {
      for (int it = 0; it < nk; ++it) {
        const int s = it % STAGES;
        ptx::mbar_wait(&empty[s], ((it / STAGES) & 1) ^ 1);
        uint8_t* sa = smem + s * STAGE;
        const int t0 = (k_lo + it) * KT;
        ptx::mbar_expect_tx(&full[s], STAGE);
        for (int a = 0; a < 2; ++a) ptx::tma_load_2d(sa + a * ATOM, &tmA, &full[s], o0 + 64 * a, t0);
        for (int a = 0; a < 4; ++a) ptx::tma_load_2d(sa + A_BYTES + a * ATOM, &tmB, &full[s], i0 + 64 * a, t0);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = idesc_bf16_f32_mnmn(128, 256);
      for (int it = 0; it < nk; ++it) {
        const int s = it % STAGES;
        ptx::mbar_wait(&full[s], (it / STAGES) & 1);
        ptx::tc_fence_after_sync();
        const uint32_t sa = ptx::smem_u32(smem + s * STAGE);
        const uint64_t da = ptx::smem_desc_mn_sw128(sa, ATOM, 1024), db = ptx::smem_desc_mn_sw128(sa + A_BYTES, ATOM, 1024);
#pragma unroll
        for (int ks = 0; ks < KT / 16; ++ks)   // 16 token rows = 2 KB per MMA
          ptx::umma_f16(tmem_base, da + (2048 >> 4) * ks, db + (2048 >> 4) * ks, idesc, (it | ks) != 0);
        ptx::umma_commit(&empty[s]);
      }
      ptx::umma_commit(done);
    }
  } else {
    const int q = warp & 3, r = q * 32 + lane;
    float* dst = p.part + ((long long)split * p.O + o0 + r) * p.I + i0;
    if (nk > 0) {
      ptx::mbar_wait(done, 0);
      ptx::tc_fence_after_sync();
#pragma unroll 1
      for (int c0 = 0; c0 < 256; c0 += 32) {
        uint32_t a[32];
        ptx::tmem_ld_32x32b_x32(tmem_base + (uint32_t(q * 32) << 16) + c0, a);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          *reinterpret_cast<float4*>(dst + c0 + j) = make_float4(__uint_as_float(a[j]), __uint_as_float(a[j + 1]),
                                                                 __uint_as_float(a[j + 2]), __uint_as_float(a[j + 3]));
      }
    } else {
      for (int c = 0; c < 256; c += 4) *reinterpret_cast<float4*>(dst + c) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after_sync();
    ptx::tmem_dealloc<256>(tmem_base);
  }
}

// dW[e] = sum over splits s = 0, 1, ... of part[s][e]
__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const float* __restrict__ part, long long n, int n_split,
                                                           float* __restrict__ dW) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  float s = 0.f;
  for (int k = 0; k < n_split; ++k) s += part[(long long)k * n + e];
  dW[e] = s;
}

}  // namespace clm
