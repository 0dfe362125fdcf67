// bf16 x bf16 -> fp32 GEMM on the 5th-gen tensor cores, with the predict path's epilogues.
//
//   D[M,N] = A[M,K] * W[N,K]^T      A = activations (tokens x features, K contiguous)
//                                   W = nn.Linear weight as stored (out x in, K contiguous)
//
// Reference ops this replaces (all `torch.nn.Linear` calls on the predict path):
//   in_proj / out_proj / fc1 / fc2 of the HF HyenaDNA block (SURVEY.md A.3, A.6) and the
//   attention-pool scorer `attention.0`/`attention.2` (chimeralm/models/components/hyena.py:50-53).
//
// Structure (one 128 x BN output tile per CTA, 2 CTAs co-resident per SM so one CTA's epilogue
// overlaps the other's loads/MMAs):
//   warp 0   : TMA producer  - cp.async.bulk.tensor tiles (128B swizzle) into a STAGES-deep ring
//   warp 1   : TMEM allocator + single-thread tcgen05.mma issuer, accumulator in TMEM
//   warps 2-5: epilogue      - tcgen05.ld (lane == output row), fused bias / GELU / residual /
//                              scorer reduction, vectorised global stores
#pragma once
#include <cuda_bf16.h>

#include "ptx.cuh"

namespace clm {

enum GemmEpilogue : int {
  EPI_BIAS_BF16 = 0,       // out_bf16 = acc + bias
  EPI_BIAS_GELU_TANH = 1,  // out_bf16 = gelu_tanh(acc + bias)          (HyenaMlp fc1, A.6)
  EPI_BIAS_RES_F32 = 2,    // out_f32  = acc + bias + res               (out_proj / fc2 + residual)
  EPI_SCORE = 3,           // score[m] = sum_n gelu_erf(acc + bias)[n] * w2[n] + b2   (needs BN == N)
  EPI_BIAS_GELU_TANH_KEEP = 4,   // EPI_BIAS_GELU_TANH, and out2_bf16 = acc + bias      (the tail's fc1 recompute)
  // dgrad GEMMs of the last block's tail (csrc/tail_train.cuh, gemm_tail_epilogue): bf16 out, per-warp column sums
  EPI_TAIL_DHID = 5,       // dz . W0 + w_t dp -> ln_f backward -> dr2                  (needs BN == N == 256)
  EPI_TAIL_DH = 6,         // dr2 . W2 -> * gelu_tanh'(h) -> dh
  EPI_TAIL_DR1 = 7,        // dh . W1 -> norm2 backward + dr2 -> dr1                    (needs BN == N == 256)
};

struct GemmParams {
  int M, N, K;
  const float* bias;   // [N]
  void* out;           // bf16 [M,ldo] or fp32 [M,ldo]
  const float* res;    // fp32 [M,ldo] (may alias out)
  const float* w2;     // EPI_SCORE: [N]
  float b2;            // EPI_SCORE
  float* score;        // EPI_SCORE: [M]
  long long ldo;
  int r32;             // EPI_BIAS_RES_F32: res/out use the R32 blocked layout (N must be 256)
  void* out2;          // EPI_BIAS_GELU_TANH_KEEP: bf16 [M,ldo] pre-activation
  // EPI_TAIL_*
  const __nv_bfloat16* nrm;   // DHID: n2, DR1: n1 (bf16 [M,256])
  const float* rho;           // DHID: rho2, DR1: rho1 ([M])
  const float* gam;           // DHID: ln_f.weight, DR1: norm2.weight
  const __nv_bfloat16* aux;   // DH: h (bf16 [M,ldo]), DR1: dr2 (bf16 [M,256])
  const float* score_in;      // DHID: the forward's scores [M]
  const float* rd;            // DHID: per read (softmax max, 1 / normaliser, -, -)
  const float* dp;            // DHID: dpooled [B,256]
  int T;                      // DHID: tokens per read (row = b * T + t)
  float* colsum;              // per-warp column partials [(M / 128) * 4][3 or 1][N]
};

template <int BN, int EPI>
__device__ void gemm_tail_epilogue(const GemmParams& p, uint32_t tmem_base, int m0, int n0, int q, int lane);   // tail_train.cuh

constexpr int GEMM_BM = 128;
constexpr int GEMM_BK = 64;   // 64 bf16 = 128 bytes = one swizzle row
constexpr int GEMM_THREADS = 192;

template <int BN, int STAGES>
struct GemmSmem {
  static constexpr int kABytes = GEMM_BM * GEMM_BK * 2;
  static constexpr int kBBytes = BN * GEMM_BK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kBarOffset = STAGES * kStageBytes;
  static constexpr int kTotal = kBarOffset + 256 + 1024;  // barriers + alignment slack
};

__device__ __forceinline__ float gelu_tanh_f(float x) {
  const float k0 = 0.7978845608028654f, k1 = 0.044715f;
  float u = k0 * (x + k1 * x * x * x);
  return 0.5f * x * (1.0f + tanhf(u));
}
__device__ __forceinline__ float gelu_erf_f(float x) { return 0.5f * x * (1.0f + erff(x * 0.7071067811865476f)); }

// two floats -> packed fp16 pair, `lo` in the low half
__device__ __forceinline__ uint32_t pack_f16(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

// packed fp32x2 arithmetic (FMUL2 / FFMA2 / FADD2 on sm_100): one instruction per two elements
typedef unsigned long long f2t;
__device__ __forceinline__ f2t f2_pack(float lo, float hi) { f2t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ f2t f2_packu(uint32_t lo, uint32_t hi) { f2t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi)); return r; }
__device__ __forceinline__ f2t f2_mul(f2t a, f2t b) { f2t d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ f2t f2_sub(f2t a, f2t b) { f2t d; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ f2t f2_fma(f2t a, f2t b, f2t c) { f2t d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ uint32_t f2_to_h2(f2t a) {   // two floats -> packed fp16 pair
  float lo, hi;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(a));
  return pack_f16(lo, hi);
}

__device__ __forceinline__ f2t f2_add(f2t a, f2t b) { f2t d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ void f2_unpack(f2t a, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(a)); }

template <int BN, int STAGES, int EPI>
__global__ void __launch_bounds__(GEMM_THREADS)
gemm_bf16_tn_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, GemmParams p) {
  using S = GemmSmem<BN, STAGES>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + S::kBarOffset);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full_bar = empty_bar + STAGES;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // 1-D grid, N-tile fastest: the CTAs that share an A tile are launched back to back, so the
  // tile is fetched from HBM once and served from L2 to the other N-tiles.
  const int n_tiles = p.N / BN;
  const int m0 = (blockIdx.x / n_tiles) * GEMM_BM;
  const int n0 = (blockIdx.x % n_tiles) * BN;
  const int num_k = p.K / GEMM_BK;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmA);
    ptx::prefetch_tmap(&tmB);
    for (int s = 0; s < STAGES; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], 1);
    }
    ptx::mbar_init(tmem_full_bar, 1);
    ptx::fence_mbar_init();
  } else if (warp == 1) {
    ptx::tmem_alloc<BN>(tmem_ptr);
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    if (lane == 0) {
      for (int kb = 0; kb < num_k; ++kb) {
        const int s = kb % STAGES;
        const uint32_t ph = (kb / STAGES) & 1;
        ptx::mbar_wait(&empty_bar[s], ph ^ 1);
        uint8_t* sa = smem + s * S::kStageBytes;
        uint8_t* sb = sa + S::kABytes;
        ptx::mbar_expect_tx(&full_bar[s], S::kStageBytes);
        ptx::tma_load_2d(sa, &tmA, &full_bar[s], kb * GEMM_BK, m0);
        ptx::tma_load_2d(sb, &tmB, &full_bar[s], kb * GEMM_BK, n0);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = ptx::idesc_bf16_f32(GEMM_BM, BN);
      for (int kb = 0; kb < num_k; ++kb) {
        const int s = kb % STAGES;
        const uint32_t ph = (kb / STAGES) & 1;
        ptx::mbar_wait(&full_bar[s], ph);
        ptx::tc_fence_after_sync();
        const uint32_t sa = ptx::smem_u32(smem + s * S::kStageBytes);
        const uint64_t da = ptx::smem_desc_k_sw128(sa);
        const uint64_t db = ptx::smem_desc_k_sw128(sa + S::kABytes);
#pragma unroll
        for (int k = 0; k < GEMM_BK / 16; ++k) {
          // advance 16 bf16 = 32 bytes along K inside the swizzled row: +2 in the (addr>>4) field
          ptx::umma_f16(tmem_base, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
        }
        ptx::umma_commit(&empty_bar[s]);
      }
      ptx::umma_commit(tmem_full_bar);
    }
  } else if constexpr (EPI >= EPI_TAIL_DHID) {
    ptx::mbar_wait(tmem_full_bar, 0);
    ptx::tc_fence_after_sync();
    gemm_tail_epilogue<BN, EPI>(p, tmem_base, m0, n0, warp & 3, lane);
    ptx::tc_fence_before_sync();
  } else {
    // ---------------- epilogue: warps 2..5, TMEM lane quarter = warp % 4
    const int q = warp & 3;
    const long long row = (long long)m0 + q * 32 + lane;
    const bool row_ok = row < p.M;
    ptx::mbar_wait(tmem_full_bar, 0);
    ptx::tc_fence_after_sync();
    float score_acc = 0.f;
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      uint32_t r[32];
      ptx::tmem_ld_32x32b_x32(tmem_base + (uint32_t(q * 32) << 16) + c0, r);
      ptx::tmem_ld_wait();
      const int n = n0 + c0;
      float v[32];
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + n + j));
        v[j + 0] = __uint_as_float(r[j + 0]) + b4.x;
        v[j + 1] = __uint_as_float(r[j + 1]) + b4.y;
        v[j + 2] = __uint_as_float(r[j + 2]) + b4.z;
        v[j + 3] = __uint_as_float(r[j + 3]) + b4.w;
      }
      if constexpr (EPI == EPI_BIAS_BF16 || EPI == EPI_BIAS_GELU_TANH || EPI == EPI_BIAS_GELU_TANH_KEEP) {
        if constexpr (EPI == EPI_BIAS_GELU_TANH_KEEP) {
          if (row_ok) {
            uint4* o2 = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.out2) + row * p.ldo + n);
#pragma unroll
            for (int j = 0; j < 32; j += 8)
              o2[j / 8] = make_uint4(pack_bf16(v[j], v[j + 1]), pack_bf16(v[j + 2], v[j + 3]), pack_bf16(v[j + 4], v[j + 5]),
                                     pack_bf16(v[j + 6], v[j + 7]));
          }
        }
        if constexpr (EPI == EPI_BIAS_GELU_TANH || EPI == EPI_BIAS_GELU_TANH_KEEP) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = gelu_tanh_f(v[j]);
        }
        if (row_ok) {
          __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(p.out) + row * p.ldo + n;
#pragma unroll
          for (int j = 0; j < 32; j += 8) {
            uint4 w;
            w.x = pack_bf16(v[j + 0], v[j + 1]);
            w.y = pack_bf16(v[j + 2], v[j + 3]);
            w.z = pack_bf16(v[j + 4], v[j + 5]);
            w.w = pack_bf16(v[j + 6], v[j + 7]);
            *reinterpret_cast<uint4*>(o + j) = w;
          }
        }
      } else if constexpr (EPI == EPI_BIAS_RES_F32) {
        if (row_ok) {
          // res/out: row-major when p.r32 == 0, the blocked residual layout (ptx::r32_off) otherwise
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const long long off = p.r32 ? ptx::r32_off(row, n + j) : row * p.ldo + n + j;
            float4 r4 = *reinterpret_cast<const float4*>(p.res + off);
            float4 w = make_float4(v[j] + r4.x, v[j + 1] + r4.y, v[j + 2] + r4.z, v[j + 3] + r4.w);
            *reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + off) = w;
          }
        }
      } else {  // EPI_SCORE
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          float4 w4 = __ldg(reinterpret_cast<const float4*>(p.w2 + n + j));
          score_acc += gelu_erf_f(v[j]) * w4.x + gelu_erf_f(v[j + 1]) * w4.y + gelu_erf_f(v[j + 2]) * w4.z +
                       gelu_erf_f(v[j + 3]) * w4.w;
        }
      }
    }
    if constexpr (EPI == EPI_SCORE) {
      if (row_ok) p.score[row] = score_acc + p.b2;
    }
    ptx::tc_fence_before_sync();
  }
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after_sync();
    ptx::tmem_dealloc<BN>(tmem_base);
  }
}

}  // namespace clm
