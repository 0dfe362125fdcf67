// C-ABI implementation: context, weights, workspaces and the launch sequence of the predict
// forward.  See include/chimeralm_b200.h for the contract of every export.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <map>
#include <set>
#include <string>
#include <vector>

#include "../../include/chimeralm_b200.h"
#include "block_in.cuh"
#include "embed_in.cuh"
#include "block_mlp.cuh"
#ifdef CLM_EXPERIMENTS   // recorded-slower variants of the block tail and the first long-convolution kernel: not in the product build
#include "block_in2.cuh"
#include "block_mlp2.cuh"
#include "block_mlp16.cuh"
#include "block_mlp_pp.cuh"
#endif
#include "gemm_tcgen05.cuh"
#include "kernels.cuh"
#include "longconv.cuh"
#include "longconv_fast.cuh"
#include "longconv_tc.cuh"
#include "longconv_tc2.cuh"
#include "score_pool.cuh"
#include "head_train.cuh"

using namespace clm;

namespace {

struct Tensor {
  float* d = nullptr;
  std::vector<int64_t> shape;
  int64_t numel = 0;
};

struct LayerW {
  const float *ln1_g, *ln1_b, *ln2_g, *ln2_b;
  const float *in_b, *out_b, *fc1_b, *fc2_b;
  const float *sc_w, *sc_b, *fbias;
  __nv_bfloat16 *in_w, *out_w, *fc1_w, *fc2_w;
  CUtensorMap tm_in, tm_out, tm_fc1, tm_fc2;
  // LayerNorm1 affine folded into in_proj (block_in kernel): W' = W diag(gamma), b' = b + W beta
  __nv_bfloat16* in_wf = nullptr;
  float* in_bf = nullptr;
  float* in_wf32 = nullptr;   // folded in_proj weights in fp32 (source of the bf16 tiles; layer 0's feed embed_in_table_kernel)
  CUtensorMap tm_inf;
  CUtensorMap tm_inf_h;   // same buffer, one k-block (128 rows) per box: the CTA-pair kernel's 16 KB slots
  // block_mlp operands, pre-tiled [N/rt][K/64][rt][64] so that every 32 KB ring slot is one TMA box
  __nv_bfloat16 *out_wt = nullptr, *fc1_wt = nullptr, *fc2_wt = nullptr;
  CUtensorMap tm_out_t, tm_fc1_t, tm_fc2_t;
  CUtensorMap tm_out_h, tm_fc1_h, tm_fc2_h;   // same buffers, half-tile boxes for the CTA-pair kernel
  __nv_bfloat16* fc1_w64 = nullptr;           // fc1 weights re-tiled with rt = 64: a 64-unit chunk is one 32 KB box
  CUtensorMap tm_fc1_64;                      // (block_mlp_pp.cuh)
  float* k = nullptr;                               // [D][Lk]
  float2* gspec[LONGCONV_MAX_LOGN + 1] = {nullptr};  // per LOGN: [n_seg][D][N]
  float2* gspecT[LONGCONV_MAX_LOGN + 1] = {nullptr}; // per LOGN: [D][16][N/16], bias folded (longconv_fast)
  __half2* gtc = nullptr;                            // [n_seg][D][16384] fp16 spectrum, lane-interleaved (longconv_tc)
  // longconv_tc dynamic-range factors (powers of two, see LongConvTcParams): table exponents, and two sets of
  // output/input factors - `cal` for the forward (input scale from the calibration draw), `unit` for a = 1 (raw fp16 entry)
  int* gexp = nullptr;                               // [n_seg][D]
  // four-reads-per-item form (reads of <= 4096 tokens): spectrum table of the filter truncated to 4096 taps, its exponents,
  // and 2^(gexp[0] - gexp4) per channel (applied on top of whichever output scale the launch uses)
  __half2* gtc4 = nullptr;
  int* gexp4 = nullptr;
  float* tc_adj4 = nullptr;
  // chunked two-in-flight form (reads longer than 8 200 tokens): V-form tables H_j = FFT([k_j | k_{j-1}]) (see
  // tc::spectrum_kernel), their exponents and 2^(e[0] - e[j]).  H_0 = G_0, so the output scale is the same as gtc's.
  __half2* gtcH = nullptr;
  int* gexpH = nullptr;
  float* tc_relH = nullptr;
  float *vx_scale = nullptr, *tc_osc = nullptr, *tc_inva = nullptr, *tc_rel = nullptr;
  float *unit_scale = nullptr, *unit_osc = nullptr, *unit_inva = nullptr;
  unsigned int* vx_amax = nullptr;                   // [D] float bits, calibration forward
};

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

constexpr int MIN_LOGN = 8;

}  // namespace

struct clm_ctx {
  clm_config cfg;
  int device = 0;
  int num_sms = 148;
  bool finalized = false;
  std::string err;
  std::map<std::string, Tensor> w;
  std::vector<LayerW> layers;
  long long Lk = 0;  // padded filter row length
  // head / final
  const float *lnf_g, *lnf_b, *emb;
  __nv_bfloat16* att0_w = nullptr;
  const float* att0_w32 = nullptr;   // attention.0.weight (fp32, as loaded; refreshed by clm_head_train_step)
  CUtensorMap tm_att0;
  // ln_f affine folded into the scorer (consumes the normalised xn emitted by the last block_mlp)
  __nv_bfloat16* att0_wf = nullptr;
  float* att0_bf = nullptr;
  float* att0_wf32 = nullptr;   // folded scorer weights in fp32 (source of att0_wf)
  CUtensorMap tm_att0f;
  __nv_bfloat16* emb_norm = nullptr;   // [vocab_rows,256] normalised embedding rows (layer-0 LayerNorm input)
  float *ones = nullptr, *zeros = nullptr;
  const float *att0_b, *att2_w;
  float att2_b = 0.f;
  HeadParams head{};
  // workspaces
  int max_B = 0, max_T = 0, Tp_max = 0;
  long long max_tokens = 0;      // token budget of the workspaces (<= max_B * max_T)
  size_t ct_elems = 0;           // elements of each channel-major buffer (VX, X0, Y)
  int last_B = 0, last_T = 0;   // shape of the last complete forward (clm_attention_weights)
  float* R = nullptr;
  __nv_bfloat16 *XN = nullptr, *U = nullptr, *VX = nullptr, *X0 = nullptr, *Y = nullptr, *YT = nullptr;
  float *score = nullptr, *part = nullptr, *pooled = nullptr;
  float* hbuf[4] = {nullptr, nullptr, nullptr, nullptr};   // head activations [max_B, 512]
  float2* scratch = nullptr;
  size_t scratch_bytes = 0;
  // Status word of the forward in flight: bit 0 = a token id outside [0, vocab_rows), bit 1 = the fp16 tensor-core
  // convolution produced a non-finite value.  The LAST kernel of every forward publishes (seq << 8 | bits) into the
  // mapped host ring h_status[seq & 7] and clears the word, so the host can read a finished forward's status without
  // another copy or synchronisation (clm_forward_status).
  int* d_err = nullptr;
  int* h_status = nullptr;       // pinned + mapped, 8 words
  int* d_status_map = nullptr;   // device alias of h_status
  long long fwd_seq = 0;
  long long tc_fallbacks = 0;    // batches clm_predict_host redid with the fp32 convolution
  bool calibrating = false;      // clm_finalize's calibration forward: record max |v*x1| per layer and channel
  int n_split = 1;
  // e2e staging
  cudaStream_t own_stream = nullptr;
  // copies of the host entry points run on their own streams, so that batch k + 1's H2D and batch k - 1's D2H overlap
  // batch k's kernels (one stream per direction: a D2H waits for its forward and must not hold the next H2D back)
  cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr;
  // Staging of the host entry points: HOST_SLOTS independent sets, so that clm_predict_host_submit can copy and enqueue
  // batch k + 1 (and k + 2) while batch k is still running; slot 0's buffers double as the calibration forward's.
  static constexpr int HOST_SLOTS = 3;
  struct HostSlot {
    uint8_t* bases = nullptr;
    int64_t* offsets = nullptr;
    uint8_t* ids = nullptr;
    float* logits = nullptr;
    uint8_t* labels = nullptr;
    cudaEvent_t done = nullptr, h2d_done = nullptr, fwd_done = nullptr;
    bool busy = false;
    long long seq = 0;
    int B = 0, T = 0;
    float* h_logits = nullptr;
    uint8_t* h_labels = nullptr;
  } slot[HOST_SLOTS];
  int next_slot = 0;
  size_t st_bases_cap = 0;
  uint8_t*& st_ids = slot[0].ids;
  float*& st_logits = slot[0].logits;
  uint8_t*& st_labels = slot[0].labels;
  // per-kernel-class device timing (CUDA events on the launching stream)
  bool prof_on = false;
  std::vector<cudaEvent_t> prof_pool;
  std::vector<int> prof_cat;      // category of event pair i (events 2i, 2i+1)
  size_t prof_used = 0;           // event pairs in flight
  double prof_ms[32] = {0};
  long long prof_n[32] = {0};
  bool fused_mlp = true;  // out_proj+res+LN2+fc1+gelu+fc2+res in one kernel
  bool fused_in = true;   // LN1+in_proj+short conv+gate in one kernel
  bool fast_conv = true;  // tuned single-chunk long convolution
  int mlp_stagger = 0;    // block_mlp: CTA phase stagger in cycles (0 = off)
  bool tc_conv = true;    // tensor-core FFT long convolution for reads of more than 2 056 tokens (needs fused_in)
  bool tc_pipe = true;    // single-transform reads (<= 8 200 tokens): two items in flight per SM (longconv_tc2_kernel)
  int tc_helpers_low = 0; // longconv_tc2: helper warps on the lowest warp ids (A/B switch)
  bool tc_pack4 = true;   // reads of 2 049 .. 4 096 tokens: four reads per transform (needs tc_pipe)
  bool tc_pipe_chunked = true;   // reads longer than 8 200 tokens on the two-in-flight kernel (V-form tables, no carry)
  __half* tc_S = nullptr; // shared-memory image of the DFT constant stack (longconv_tc)
  bool fused_head = true;         // pooling merge + classifier layers in one cooperative launch
  bool head_coop = true;          // 0: plain launch of the same kernel (A/B of the cooperative launch's own cost; <= 256 CTAs of 64 KB)
  unsigned int* head_counter = nullptr;
  unsigned int head_base = 0;
  bool fused_score_pool = true;   // scorer GEMM + pooling partials in one persistent kernel (needs the folded tail)
  bool tc_chunked = true; // tensor-core conv also for reads longer than 8200 tokens (overlap-add over 8192-token chunks)
  int tc_nseg = 0;        // filter segments of 8192 taps with a spectrum table
  float* tc_scratch = nullptr;
  size_t tc_scratch_floats = 0;
  bool mlp_2cta = false;  // CTA-pair (cta_group::2) version of the fused block tail
  bool mlp_epi16 = false; // fused block tail with 16 epilogue warps (block_mlp16.cuh)
  int mlp_helpers_high = 0;
  bool pdl = true;        // programmatic dependent launch of the step's kernels (launch_k)
  bool pdl_now = false;   // ... for the forward being issued: only when EVERY kernel between the embedding and the head takes part
                          // (the tensor-core conv; with the fp32 FFT conv in the chain the step measured 2.7 % slower, profiles/r2_ab_interleaved.txt)
  bool embed_in = true;   // block 0's first half by table lookup over the token ids (embed_in.cuh) instead of block_in_kernel
  float* u_tab0 = nullptr;   // [768][16] in_proj output of block 0 per vocabulary row
  float* emb_r32 = nullptr;  // embedding rows as a 32-row R32 table: block 0's residual input is looked up by token id
  bool embed_res = true;     // with embed_in: no embedding kernel at all (block_mlp of block 0 reads emb_r32)
  bool mlp_gather_tails = true;   // block_mlp: reads ending in a <= 64-token partial tile share gathered tiles (BlockMlpParams::gather_L)
  __nv_bfloat16* YG = nullptr;    // gathered tail columns of Y, channel-major [D][128 x gathered tiles]
  size_t yg_elems = 0;
  int mlp_store_a = 0;    // block_mlp: residual column groups stored in the statistics sweep of the output epilogue
  bool in_ext_tail = true;   // block_in: a read's tail of <= 16 tokens rides on its last full tile (BlockInParams::ext_L)
  int in_prefetch = 0;    // block_in: next token tile prefetched into L2 (measured: no effect, 0.667 vs 0.665 ms/step interleaved)
  int mlp_early_res = 33; // block_mlp: float4 of the next tile's residual half-row loaded before E3 (0, 16, 32; 33 = spread over E3)
  int mlp_fc2_lag = 1;    // block_mlp: fc2 of chunk j - lag is issued after fc1 of chunk j (2: recorded experiment, no faster)
  int mlp_grid = 0;       // block_mlp: cap on the number of CTAs (0 = one per SM); diagnostic
  bool mlp_pp = false;    // fused block tail with two interleaved fc1/GELU/fc2 chains of 64-unit chunks (block_mlp_pp.cuh)
  bool in_2cta = false;         // block_in on CTA pairs (block_in2.cuh)
  bool skip_dead_res = true;    // the last block does not store its fp32 residual (nothing reads it)
  bool y_channel_major = true;  // block_mlp reads the conv output channel-major (MN-major UMMA operand): no transpose
  // debug
  int dbg_layer = -1, dbg_stage = -1;
  long long launches = 0;
  EncodeTiledFn encode_tiled = nullptr;
  std::vector<void*> owned;  // device allocations freed at destroy
  std::vector<bm::LayerConsts> h_mlp;     // this model's block-tail constants (the __constant__ bank is per DEVICE, see bind_constants)
  std::set<const void*> smem_attr_done;   // kernels whose dynamic-smem limit was raised on THIS device (per context, not per process)
  // head fine-tuning (clm_head_train_*): everything is allocated by clm_head_train_begin, nothing per step
  struct HeadTrain {
    bool on = false;
    clm_head_train_cfg cfg{};
    int max_B = 0;
    uint32_t thr = 0;          // dropout: keep <=> (hash >> 8) >= thr
    float scale = 1.f;         // 1 / (1 - p)
    long long calls = 0;       // clm_head_train_step calls so far: the `step` of the dropout hash
    long long n = 0;           // elements of the flat head buffers
    float *param = nullptr, *grad = nullptr, *m = nullptr, *v = nullptr;   // fp32 master copy, gradient, AdamW state
    int* step = nullptr;       // AdamW steps applied (device)
    float *z0 = nullptr, *z1 = nullptr, *z2 = nullptr;                        // [B,512] pre-activations
    float *x1 = nullptr, *x2 = nullptr, *x3 = nullptr, *x4 = nullptr;        // [B,512] layer inputs (after dropout)
    float *logits = nullptr, *dlogits = nullptr, *fwd_logits = nullptr;      // [B,2]
    float *dA = nullptr, *dB = nullptr, *dC = nullptr, *dpooled = nullptr;  // [B,512] x3, [B,256]
    float *rd = nullptr, *gdp = nullptr;                                     // [B][4], [B][256]
    float *part_dw = nullptr, *part_vec = nullptr;                           // score_bwd_kernel partials
    int n_cta = 0;
  } ht;
};

namespace {

int fail(clm_ctx* c, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (c) c->err = buf;
  return code;
}

#define CLM_CUDA(ctx, expr)                                                                          \
  do {                                                                                               \
    cudaError_t e_ = (expr);                                                                         \
    if (e_ != cudaSuccess)                                                                           \
      return fail(ctx, CLM_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

// CLM_SYNC_CHECK=1 in the environment: synchronise after every launch so an execution fault names its kernel.
static const bool g_sync_check = [] { const char* e = getenv("CLM_SYNC_CHECK"); return e && e[0] == '1'; }();

#define CLM_LAUNCH_CHECK(ctx, what)                                                                  \
  do {                                                                                               \
    cudaError_t e_ = cudaGetLastError();                                                             \
    if (e_ != cudaSuccess) return fail(ctx, CLM_ERR_CUDA, "launch %s failed: %s", what, cudaGetErrorString(e_)); \
    if (g_sync_check) {                                                                              \
      e_ = cudaDeviceSynchronize();                                                                  \
      if (e_ != cudaSuccess) {                                                                       \
        fprintf(stderr, "[chimeralm_b200] kernel %s faulted: %s\n", what, cudaGetErrorString(e_));   \
        return fail(ctx, CLM_ERR_CUDA, "kernel %s faulted: %s", what, cudaGetErrorString(e_));       \
      }                                                                                              \
    }                                                                                                \
    (ctx)->launches++;                                                                               \
  } while (0)

// bm::c_mlp is ONE __constant__ bank per device, shared by every context (model) on it: before a block-tail launch make sure
// it holds THIS model's biases (a second model finalized on the same device would otherwise silently replace them).
const clm_ctx* g_const_owner[64] = {nullptr};
int bind_constants(clm_ctx* c, cudaStream_t st) {
  const int dev = c->device & 63;
  if (g_const_owner[dev] == c || c->h_mlp.empty()) return 0;
  CLM_CUDA(c, cudaMemcpyToSymbolAsync(bm::c_mlp, c->h_mlp.data(), c->h_mlp.size() * sizeof(bm::LayerConsts), 0, cudaMemcpyHostToDevice, st));
  g_const_owner[dev] = c;
  return 0;
}

// Launch with (c->pdl) or without programmatic stream serialization: every kernel launched through here calls
// ptx::griddep_wait() before it touches anything its predecessors wrote, so its prologue may overlap their tail.
template <typename... Params, typename... Args>
cudaError_t launch_k(clm_ctx* c, void (*kern)(Params...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at{};
  at.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at.val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = &at;
  cfg.numAttrs = (c->pdl_now && !c->prof_on) ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<Params>(args)...);
}

int ensure_smem_attr(clm_ctx* c, const void* func, int bytes) {
  if (c->smem_attr_done.count(func)) return 0;
  CLM_CUDA(c, cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  c->smem_attr_done.insert(func);
  return 0;
}

template <typename T>
int dev_alloc(clm_ctx* c, T** p, size_t count) {
  void* q = nullptr;
  cudaError_t e = cudaMalloc(&q, count * sizeof(T) + 256);
  if (e != cudaSuccess) {
    cudaGetLastError();   // clear the (non-sticky) error: the next launch check must not report this allocation failure
    return fail(c, CLM_ERR_NOMEM, "cudaMalloc(%zu bytes) failed: %s", count * sizeof(T), cudaGetErrorString(e));
  }
  c->owned.push_back(q);
  *p = reinterpret_cast<T*>(q);
  return 0;
}

void dev_free(clm_ctx* c, void* p) {
  if (!p) return;
  for (size_t i = 0; i < c->owned.size(); ++i)
    if (c->owned[i] == p) {
      cudaFree(p);
      c->owned[i] = c->owned.back();
      c->owned.pop_back();
      return;
    }
}

// frees *p and nulls it, so that a failed re-allocation can never leave a dangling workspace pointer behind
template <typename T>
void dev_release(clm_ctx* c, T** p) {
  dev_free(c, *p);
  *p = nullptr;
}

// dst[(((n/rt)*(K/64) + k/64)*rt + n%rt)*64 + k%64] = bf16(src[n][k])
__global__ void retile_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int N, int K, int rt) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)N * K) return;
  const int n = (int)(i / K), k = (int)(i % K);
  const long long o = ((((long long)(n / rt) * (K / 64) + k / 64) * rt + n % rt) << 6) + (k & 63);
  dst[o] = __float2bfloat16(src[i]);
}

__global__ void scale_f32_kernel(float* __restrict__ x, long long n, float f) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] *= f;
}

__global__ void f32_to_bf16_kernel(const float* __restrict__ s, __nv_bfloat16* __restrict__ d, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) d[i] = __float2bfloat16(s[i]);
}

int make_tmap_bf16_2d(clm_ctx* c, CUtensorMap* tm, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {cols * 2};
  cuuint32_t box[2] = {(cuuint32_t)GEMM_BK, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = c->encode_tiled(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box,
                               estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(c, CLM_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d (rows=%llu cols=%llu)", (int)r, (unsigned long long)rows, (unsigned long long)cols);
  return 0;
}

const Tensor* find(clm_ctx* c, const std::string& name) {
  auto it = c->w.find(name);
  return it == c->w.end() ? nullptr : &it->second;
}

int need(clm_ctx* c, const std::string& name, int64_t numel, const float** out) {
  const Tensor* t = find(c, name);
  if (!t) return fail(c, CLM_ERR_MISSING, "weight '%s' was not loaded", name.c_str());
  if (t->numel != numel) return fail(c, CLM_ERR_INVALID, "weight '%s' has %lld elements, expected %lld", name.c_str(), (long long)t->numel, (long long)numel);
  *out = t->d;
  return 0;
}

int retile(clm_ctx* c, const float* src, int N, int K, int rt, __nv_bfloat16** out, CUtensorMap* tm) {
  int rc = dev_alloc(c, out, (size_t)N * K);
  if (rc) return rc;
  retile_bf16_kernel<<<(unsigned)(((long long)N * K + 255) / 256), 256>>>(src, *out, N, K, rt);
  CLM_LAUNCH_CHECK(c, "retile_bf16");
  cuuint64_t dims[2] = {64, (cuuint64_t)((long long)N * K / 64)};
  cuuint64_t strides[1] = {128};
  cuuint32_t box[2] = {64, 256}, estr[2] = {1, 1};
  CUresult r = c->encode_tiled(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, *out, dims, strides, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(c, CLM_ERR_CUDA, "cuTensorMapEncodeTiled(retiled weight) failed with CUresult %d", (int)r);
  return 0;
}

// tensor map over an already re-tiled [rows x 64] bf16 weight buffer with a box of `box_rows` rows
int make_tmap_retiled(clm_ctx* c, CUtensorMap* tm, const void* buf, long long rows, int box_rows) {
  cuuint64_t dims[2] = {64, (cuuint64_t)rows};
  cuuint64_t strides[1] = {128};
  cuuint32_t box[2] = {64, (cuuint32_t)box_rows}, estr[2] = {1, 1};
  CUresult r = c->encode_tiled(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(buf), dims, strides, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(c, CLM_ERR_CUDA, "cuTensorMapEncodeTiled(retiled, box %d) failed with CUresult %d", box_rows, (int)r);
  return 0;
}

int to_bf16(clm_ctx* c, const float* src, int64_t n, __nv_bfloat16** out) {
  int rc = dev_alloc(c, out, (size_t)n);
  if (rc) return rc;
  f32_to_bf16_kernel<<<(unsigned)((n + 255) / 256), 256>>>(src, *out, n);
  CLM_LAUNCH_CHECK(c, "f32_to_bf16");
  return 0;
}

template <int BN, int STAGES, int EPI>
int launch_gemm_t(clm_ctx* c, const CUtensorMap& tmA, const CUtensorMap& tmB, const GemmParams& p, cudaStream_t st) {
  using S = GemmSmem<BN, STAGES>;
  auto kern = gemm_bf16_tn_kernel<BN, STAGES, EPI>;
  if (int rc_attr = ensure_smem_attr(c, (const void*)(kern), (int)(S::kTotal))) return rc_attr;
  dim3 grid((unsigned)(((p.M + GEMM_BM - 1) / GEMM_BM) * (p.N / BN)));
  kern<<<grid, GEMM_THREADS, S::kTotal, st>>>(tmA, tmB, p);
  CLM_LAUNCH_CHECK(c, "gemm_bf16_tn");
  return 0;
}

int launch_gemm(clm_ctx* c, const void* A, const CUtensorMap& tmB, const GemmParams& p, int epi, cudaStream_t st) {
  if (p.K % GEMM_BK != 0 || p.K <= 0) return fail(c, CLM_ERR_INVALID, "gemm: K=%d must be a positive multiple of %d", p.K, GEMM_BK);
  if (p.M <= 0) return fail(c, CLM_ERR_INVALID, "gemm: M=%d", p.M);
  CUtensorMap tmA;
  int rc = make_tmap_bf16_2d(c, &tmA, A, (uint64_t)p.M, (uint64_t)p.K, GEMM_BM);
  if (rc) return rc;
  if (epi == EPI_SCORE) {
    if (p.N != 256) return fail(c, CLM_ERR_INVALID, "gemm: scorer epilogue needs N == 256 (got %d)", p.N);
    return launch_gemm_t<256, 2, EPI_SCORE>(c, tmA, tmB, p, st);
  }
  if (p.N % 128 != 0) return fail(c, CLM_ERR_INVALID, "gemm: N=%d must be a multiple of 128", p.N);
  switch (epi) {
    case EPI_BIAS_BF16: return launch_gemm_t<128, 3, EPI_BIAS_BF16>(c, tmA, tmB, p, st);
    case EPI_BIAS_GELU_TANH: return launch_gemm_t<128, 3, EPI_BIAS_GELU_TANH>(c, tmA, tmB, p, st);
    case EPI_BIAS_RES_F32: return launch_gemm_t<128, 3, EPI_BIAS_RES_F32>(c, tmA, tmB, p, st);
    default: return fail(c, CLM_ERR_INVALID, "gemm: unknown epilogue %d", epi);
  }
}

int make_tmap_ct_bf16_3d(clm_ctx* c, CUtensorMap* tm, const void* base, int B, int D, int Tp) {
  cuuint64_t dims[3] = {(cuuint64_t)Tp, (cuuint64_t)D, (cuuint64_t)B};
  cuuint64_t strides[2] = {(cuuint64_t)Tp * 2, (cuuint64_t)Tp * D * 2};
  cuuint32_t box[3] = {64, 128, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = c->encode_tiled(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box,
                               estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(c, CLM_ERR_CUDA, "cuTensorMapEncodeTiled(3d) failed with CUresult %d", (int)r);
  return 0;
}

// xn as a 3-D tensor {col 256, t T, b B} over a token-major bf16 [B*T,256] buffer; box {64, box_rows, 1}
int make_tmap_xn(clm_ctx* c, CUtensorMap* tm, const void* base, int B, int T, int box_rows) {
  cuuint64_t dims[3] = {256, (cuuint64_t)T, (cuuint64_t)B};
  cuuint64_t strides[2] = {512, (cuuint64_t)T * 512};
  cuuint32_t box[3] = {64, (cuuint32_t)box_rows, 1}, estr[3] = {1, 1, 1};
  CUresult r = c->encode_tiled(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(c, CLM_ERR_CUDA, "cuTensorMapEncodeTiled(xn) failed with CUresult %d", (int)r);
  return 0;
}

int launch_block_in(clm_ctx* c, int layer, const __nv_bfloat16* xn, int B, int T, int Tp, __nv_bfloat16* vx,
                    __nv_bfloat16* x0, cudaStream_t st, long long* trace = nullptr, bool vx_f16 = false) {
  if (int rc_attr = ensure_smem_attr(c, (const void*)(block_in_kernel), (int)(bi::SMEM_TOTAL))) return rc_attr;
  LayerW& L = c->layers[layer];
  CUtensorMap tmVX, tmX0, tmXN;
  int rc;
  if ((rc = make_tmap_ct_bf16_3d(c, &tmVX, vx, B, c->cfg.d_model, Tp))) return rc;
  if ((rc = make_tmap_ct_bf16_3d(c, &tmX0, x0, B, c->cfg.d_model, Tp))) return rc;
#ifdef CLM_EXPERIMENTS
  const bool pair = c->in_2cta && c->num_sms >= 2;
  if ((rc = make_tmap_xn(c, &tmXN, xn, B, T, pair ? bi2::HALF : bi::NCOL))) return rc;
#else
  if ((rc = make_tmap_xn(c, &tmXN, xn, B, T, bi::NCOL))) return rc;
#endif
  BlockInParams p{};
  p.b_in = L.in_bf; p.cw = L.sc_w; p.cb = L.sc_b;
  p.B = B; p.T = T; p.trace = trace; p.vx_f16 = vx_f16 ? 1 : 0;
  p.vx_scale = vx_f16 ? L.vx_scale : nullptr;   // fp16 rows carry a[ch] * v*x1 (undone by the conv's output scale)
  p.prefetch_xn = c->in_prefetch;
  p.tiles_per_seq = (T + bi::BT - 1) / bi::BT;
  p.num_tiles = B * p.tiles_per_seq;
  CUtensorMap tmXNE = tmXN;
#ifdef CLM_EXPERIMENTS
  const bool ext_ok = !pair;
#else
  const bool ext_ok = true;
#endif
  if (ext_ok && c->in_ext_tail && T >= bi::BT && T % bi::BT >= 1 && T % bi::BT <= bi::EXT) {
    // tails of 1..16 tokens ride on the read's last full tile (BlockInParams::ext_L) instead of being a tile of their own
    if ((rc = make_tmap_xn(c, &tmXNE, xn, B, T, bi::NCOL_EXT))) return rc;
    p.ext_L = T % bi::BT;
    p.tiles_per_seq = T / bi::BT;
    p.num_tiles = B * p.tiles_per_seq;
  }
#ifdef CLM_EXPERIMENTS
  if (pair) {   // CTA pairs (cta_group::2): one tile per pair, each CTA half of the channels and half of the token rows
    if (int rc_attr = ensure_smem_attr(c, (const void*)(block_in2_kernel), (int)(bi2::SMEM_TOTAL2))) return rc_attr;
    const int grid2 = 2 * std::min(p.num_tiles, c->num_sms / 2);
    block_in2_kernel<<<grid2, bi::THREADS, bi2::SMEM_TOTAL2, st>>>(L.tm_inf_h, tmVX, tmX0, tmXN, p);
    CLM_LAUNCH_CHECK(c, "block_in2");
    return 0;
  }
#endif
  const int grid = std::min(p.num_tiles, c->num_sms);
  launch_k(c, block_in_kernel, dim3(grid), dim3(bi::THREADS), bi::SMEM_TOTAL, st, L.tm_inf, tmVX, tmX0, tmXN, tmXNE, p);
  CLM_LAUNCH_CHECK(c, "block_in");
  return 0;
}

// block 0's first half straight from the token ids (embed_in.cuh)
int launch_embed_in(clm_ctx* c, const void* d_ids, int ids_dtype, int B, int T, int Tp, void* vx, __nv_bfloat16* x0,
                    cudaStream_t st, bool vx_f16) {
  LayerW& L = c->layers[0];
  EmbedInParams p{};
  p.ids = d_ids; p.U = c->u_tab0; p.cw = L.sc_w; p.cb = L.sc_b;
  p.vx_scale = vx_f16 ? L.vx_scale : nullptr;
  p.x0 = x0; p.vx = vx; p.B = B; p.T = T; p.Tp = Tp; p.vx_f16 = vx_f16 ? 1 : 0; p.rows = c->cfg.vocab_rows;
  p.err = c->d_err;
  const dim3 grid((unsigned)((Tp + ei::BLOCK_TOK - 1) / ei::BLOCK_TOK), ei::D / ei::CG, (unsigned)B);
#define CLM_EI_LAUNCH(IdT)                                                          \
  if (vx_f16) launch_k(c, embed_in_kernel<IdT, true>, grid, dim3(ei::THREADS), 0, st, p);           \
  else launch_k(c, embed_in_kernel<IdT, false>, grid, dim3(ei::THREADS), 0, st, p)
  switch (ids_dtype) {
    case CLM_U8: CLM_EI_LAUNCH(uint8_t); break;
    case CLM_I32: CLM_EI_LAUNCH(int32_t); break;
    case CLM_I64: CLM_EI_LAUNCH(int64_t); break;
    default: return fail(c, CLM_ERR_INVALID, "embed_in: ids dtype %d not supported", ids_dtype);
  }
#undef CLM_EI_LAUNCH
  CLM_LAUNCH_CHECK(c, "embed_in");
  return 0;
}

// y token-major [M,256] when B == 0; channel-major [B][256][Tp] (M == B*T) otherwise
int launch_block_mlp(clm_ctx* c, int layer, const __nv_bfloat16* y, float* res, int M, cudaStream_t st,
                     long long* trace = nullptr, int B = 0, int T = 0, int Tp = 0, __nv_bfloat16* xn_out = nullptr,
                     bool skip_res_store = false, const void* ids = nullptr, int ids_dtype = 0) {
  if (int rc_c = bind_constants(c, st)) return rc_c;
  LayerW& L = c->layers[layer];
  CUtensorMap tmY;
  int rc;
  if (B > 0) {
    cuuint64_t dims[3] = {(cuuint64_t)Tp, (cuuint64_t)c->cfg.d_model, (cuuint64_t)B};
    cuuint64_t strides[2] = {(cuuint64_t)Tp * 2, (cuuint64_t)Tp * c->cfg.d_model * 2};
    cuuint32_t box[3] = {64, 64, 1}, estr[3] = {1, 1, 1};
    CUresult r = c->encode_tiled(&tmY, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<__nv_bfloat16*>(y), dims, strides, box,
                                 estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                 CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(c, CLM_ERR_CUDA, "cuTensorMapEncodeTiled(y channel-major) failed with CUresult %d", (int)r);
  } else if ((rc = make_tmap_bf16_2d(c, &tmY, y, (uint64_t)M, (uint64_t)c->cfg.d_model, 128))) {
    return rc;
  }
  BlockMlpParams p{};
  p.M = M; p.res = res; p.layer = layer;
  p.eps = c->cfg.layer_norm_eps;
  p.num_tiles = (M + bm::BM - 1) / bm::BM;
  p.trace = trace;
  p.stagger_cycles = c->mlp_stagger;
  p.helpers_high = c->mlp_helpers_high;
  p.store_a = c->mlp_store_a;
  p.skip_res_store = (skip_res_store && xn_out) ? 1 : 0;
  if (B > 0) {
    p.y_cm = 1; p.T = T; p.tiles_per_seq = (T + bm::BM - 1) / bm::BM; p.num_tiles = B * p.tiles_per_seq;
  }
  p.n_full_tiles = p.num_tiles; p.B = B; p.xn = xn_out;
  if (ids) { p.res_tab = c->emb_r32; p.ids = ids; p.ids_dtype = ids_dtype; p.vocab_rows = c->cfg.vocab_rows; }
  CUtensorMap tmYG = tmY;
#ifdef CLM_EXPERIMENTS
  const bool gather_ok = !(c->mlp_2cta && !trace) && !c->mlp_pp && !c->mlp_epi16;
#else
  const bool gather_ok = true;
#endif
  if (B > 1 && c->mlp_gather_tails && gather_ok && c->YG) {
    // tails of 1..64 tokens: 128 / L of them per gathered tile instead of one partial tile each (BlockMlpParams::gather_L)
    const int Lt = T % bm::BM;
    const int P = Lt > 0 ? bm::BM / Lt : 0;
    const int n_g = P >= 2 ? (B + P - 1) / P : 0;
    const int D = c->cfg.d_model;
    const size_t TG = (size_t)n_g * bm::BM;
    if (n_g > 0 && n_g < B && TG * D <= c->yg_elems) {
      launch_k(c, gather_tails_kernel, dim3((unsigned)((TG * D + 255) / 256)), dim3(256), 0, st, y, c->YG, B, D, Tp, (int)TG, T - Lt, Lt, P);
      CLM_LAUNCH_CHECK(c, "gather_tails");
      cuuint64_t dims[3] = {(cuuint64_t)TG, (cuuint64_t)D, 1};
      cuuint64_t strides[2] = {(cuuint64_t)TG * 2, (cuuint64_t)TG * D * 2};
      cuuint32_t box[3] = {64, 64, 1}, estr[3] = {1, 1, 1};
      CUresult r = c->encode_tiled(&tmYG, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, c->YG, dims, strides, box, estr,
                                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) return fail(c, CLM_ERR_CUDA, "cuTensorMapEncodeTiled(gathered tails) failed with CUresult %d", (int)r);
      p.gather_L = Lt; p.gather_P = P;
      p.tiles_per_seq = T / bm::BM;
      p.n_full_tiles = B * p.tiles_per_seq;
      p.num_tiles = p.n_full_tiles + n_g;
    }
  }
  CUtensorMap tmXN = tmY;
  if (xn_out) {
    p.write_xn = 1;
    if ((rc = make_tmap_xn(c, &tmXN, xn_out, B > 0 ? B : 1, B > 0 ? T : M, 128))) return rc;
  }
#ifdef CLM_EXPERIMENTS
  if (c->mlp_2cta && !trace) {
    if (int rc_attr = ensure_smem_attr(c, (const void*)(block_mlp2_kernel), (int)(bm2::SMEM_TOTAL2))) return rc_attr;
    const int n_pair_tiles = (p.num_tiles + 1) / 2;
    const int grid2 = 2 * std::min(n_pair_tiles, c->num_sms / 2);
    block_mlp2_kernel<<<grid2, bm::THREADS, bm2::SMEM_TOTAL2, st>>>(tmY, L.tm_out_h, L.tm_fc1_h, L.tm_fc2_h, tmXN, p);
    CLM_LAUNCH_CHECK(c, "block_mlp2");
    return 0;
  }
#endif
  const int grid = std::min(p.num_tiles, c->mlp_grid > 0 ? std::min(c->mlp_grid, c->num_sms) : c->num_sms);
#ifdef CLM_EXPERIMENTS
  if (c->mlp_pp) {
    if (int rc_attr = ensure_smem_attr(c, (const void*)(block_mlp_pp_kernel), (int)(bm::SMEM_TOTAL))) return rc_attr;
    block_mlp_pp_kernel<<<grid, bm::THREADS, bm::SMEM_TOTAL, st>>>(tmY, L.tm_out_t, L.tm_fc1_64, L.tm_fc2_t, tmXN, p);
    CLM_LAUNCH_CHECK(c, "block_mlp_pp");
    return 0;
  }
  if (c->mlp_epi16) {
    if (int rc_attr = ensure_smem_attr(c, (const void*)(block_mlp16_kernel), (int)(bm16::SMEM_TOTAL))) return rc_attr;
    block_mlp16_kernel<<<grid, bm16::THREADS, bm16::SMEM_TOTAL, st>>>(tmY, L.tm_out_t, L.tm_fc1_t, L.tm_fc2_t, tmXN, p);
    CLM_LAUNCH_CHECK(c, "block_mlp16");
    return 0;
  }
#endif
#define CLM_MLP_LAUNCH(E, LAG)                                                                                             \
  {                                                                                                                        \
    if (int rc_attr = ensure_smem_attr(c, (const void*)(block_mlp_kernel<E, LAG>), (int)(bm::SMEM_TOTAL))) return rc_attr;  \
    launch_k(c, block_mlp_kernel<E, LAG>, dim3(grid), dim3(bm::THREADS_WG), bm::SMEM_TOTAL, st, tmY, L.tm_out_t, L.tm_fc1_t, L.tm_fc2_t, tmXN, tmYG, p); \
  }
  if (c->mlp_fc2_lag >= 2) CLM_MLP_LAUNCH(33, 2)
  else if (c->mlp_early_res >= 33) CLM_MLP_LAUNCH(33, 1)
  else if (c->mlp_early_res >= 32) CLM_MLP_LAUNCH(32, 1)
  else if (c->mlp_early_res >= 16) CLM_MLP_LAUNCH(16, 1)
  else CLM_MLP_LAUNCH(0, 1)
#undef CLM_MLP_LAUNCH
  CLM_LAUNCH_CHECK(c, "block_mlp");
  return 0;
}

// ---- long convolution dispatch -------------------------------------------------------------
struct ConvPlan {
  int logn, n_chunks;
};

ConvPlan plan_conv(int T) {
  for (int logn = MIN_LOGN; logn <= LONGCONV_MAX_LOGN; ++logn) {
    const int C = 1 << (logn - 1);
    if (T <= C + LONGCONV_TAIL_MAX) return {logn, 1};
  }
  const int C = 1 << (LONGCONV_MAX_LOGN - 1);
  int n = T / C;
  if (T % C > LONGCONV_TAIL_MAX) n += 1;
  return {LONGCONV_MAX_LOGN, n};
}

int n_segments(const clm_ctx* c, int logn) {
  if (logn < LONGCONV_MAX_LOGN) return 1;
  const int C = 1 << (logn - 1);
  return (c->cfg.max_seq_len + C - 1) / C;
}

#ifdef CLM_EXPERIMENTS
template <int LOGN>
int spectrum_t(clm_ctx* c, LayerW& L) {
  using Cfg = ConvCfg<LOGN>;
  const int D = c->cfg.d_model, nseg = n_segments(c, LOGN);
  int rc = dev_alloc(c, &L.gspec[LOGN], (size_t)nseg * D * Cfg::N);
  if (rc) return rc;
  auto kern = filter_spectrum_kernel<LOGN>;
  CLM_CUDA(c, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM));
  kern<<<dim3(D, nseg), Cfg::THREADS, Cfg::SMEM>>>(L.k, c->Lk, c->cfg.max_seq_len, L.gspec[LOGN], D);
  CLM_LAUNCH_CHECK(c, "filter_spectrum");
  return 0;
}

#endif

template <int LOGN>
int spectrum_fast_t(clm_ctx* c, LayerW& L) {
  if constexpr (FastCfg<LOGN>::kSupported) {
    using Cfg = ConvCfg<LOGN>;
    const int D = c->cfg.d_model;
    const int nseg = n_segments(c, LOGN);
    int rc = dev_alloc(c, &L.gspecT[LOGN], (size_t)nseg * D * Cfg::N);
    if (rc) return rc;
    auto kern = filter_spectrum_fast_kernel<LOGN>;
    CLM_CUDA(c, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM));
    kern<<<dim3(D, nseg), Cfg::THREADS, Cfg::SMEM>>>(L.k, c->Lk, c->cfg.max_seq_len, L.fbias, L.gspecT[LOGN], D);
    CLM_LAUNCH_CHECK(c, "filter_spectrum_fast");
  }
  return 0;
}

template <int LOGN>
int conv_fast_t(clm_ctx* c, const LongConvFastParams& p, int grid, cudaStream_t st) {
  if constexpr (FastCfg<LOGN>::kSupported) {
    using F = FastCfg<LOGN>;
    auto kern = longconv_fast_kernel<LOGN>;
    if (int rc_attr = ensure_smem_attr(c, (const void*)(kern), (int)(F::SMEM))) return rc_attr;
    kern<<<grid, F::THREADS, F::SMEM, st>>>(p);
    CLM_LAUNCH_CHECK(c, "longconv_fast");
    return 0;
  } else {
    return fail(c, CLM_ERR_INVALID, "longconv_fast: unsupported size");
  }
}

#ifdef CLM_EXPERIMENTS
template <int LOGN>
int conv_t(clm_ctx* c, const LongConvParams& p, int grid, cudaStream_t st) {
  using Cfg = ConvCfg<LOGN>;
  auto kern = longconv_kernel<LOGN>;
  if (int rc_attr = ensure_smem_attr(c, (const void*)(kern), (int)(Cfg::SMEM))) return rc_attr;
  kern<<<grid, Cfg::THREADS, Cfg::SMEM, st>>>(p);
  CLM_LAUNCH_CHECK(c, "longconv");
  return 0;
}

#endif

size_t conv_scratch_bytes(const clm_ctx* c, int T) {
  ConvPlan pl = plan_conv(T);
  if (pl.n_chunks <= 1) return 0;
  return (size_t)c->num_sms * pl.n_chunks * ((size_t)1 << pl.logn) * sizeof(float2);
}

int launch_longconv(clm_ctx* c, int layer, const __nv_bfloat16* vx, const __nv_bfloat16* x0, __nv_bfloat16* out, int B,
                    int T, int Tp, float2* scratch, size_t scratch_bytes, cudaStream_t st) {
  if (T > c->cfg.max_seq_len) return fail(c, CLM_ERR_INVALID, "longconv: T=%d exceeds max_seq_len=%d", T, c->cfg.max_seq_len);
  const ConvPlan pl = plan_conv(T);
  LayerW& L = c->layers[layer];
#ifdef CLM_EXPERIMENTS
  const bool use_fast = c->fast_conv && L.gspecT[pl.logn] != nullptr;
#else
  const bool use_fast = true;
  if (L.gspecT[pl.logn] == nullptr) return fail(c, CLM_ERR_STATE, "longconv: no spectrum table for logN=%d", pl.logn);
#endif
  if (use_fast) {
    LongConvFastParams f{};
    f.vx = vx; f.x0 = x0; f.out = out; f.gT = L.gspecT[pl.logn]; f.k = L.k; f.dbias = L.fbias; f.Lk = c->Lk;
    f.B = B; f.D = c->cfg.d_model; f.T = T; f.Tp = Tp;
    f.n_chunks = pl.n_chunks; f.scratch = scratch;
    f.n_items = c->cfg.d_model * ((B + 1) / 2);
    int grid = f.n_items;
    if (pl.logn >= 13) grid = std::min(grid, c->num_sms);
    else grid = std::min(grid, c->num_sms * 4);
    if (pl.n_chunks > 1) {
      const size_t needb = (size_t)grid * pl.n_chunks * ((size_t)1 << pl.logn) * sizeof(float2);
      if (needb > scratch_bytes) return fail(c, CLM_ERR_STATE, "longconv: scratch too small (%zu < %zu); call clm_reserve with max_T >= %d", scratch_bytes, needb, T);
    }
    switch (pl.logn) {
      case 8: return conv_fast_t<8>(c, f, grid, st);
      case 12: return conv_fast_t<12>(c, f, grid, st);
      case 9: return conv_fast_t<9>(c, f, grid, st);
      case 10: return conv_fast_t<10>(c, f, grid, st);
      case 11: return conv_fast_t<11>(c, f, grid, st);
      case 13: return conv_fast_t<13>(c, f, grid, st);
      case 14: return conv_fast_t<14>(c, f, grid, st);
    }
  }
#ifdef CLM_EXPERIMENTS
  LongConvParams p{};
  p.vx = vx; p.x0 = x0; p.out = out;
  p.gspec = L.gspec[pl.logn];
  p.k = L.k; p.dbias = L.fbias; p.scratch = scratch; p.Lk = c->Lk;
  p.B = B; p.D = c->cfg.d_model; p.T = T; p.Tp = Tp;
  p.n_chunks = pl.n_chunks;
  p.n_items = c->cfg.d_model * ((B + 1) / 2);
  int grid = p.n_items;
  if (pl.logn == LONGCONV_MAX_LOGN) grid = std::min(grid, c->num_sms);  // 1 CTA/SM (139 KB smem), persistent
  else grid = std::min(grid, c->num_sms * 8);
  if (pl.n_chunks > 1) {
    const size_t needb = (size_t)grid * pl.n_chunks * ((size_t)1 << pl.logn) * sizeof(float2);
    if (needb > scratch_bytes) return fail(c, CLM_ERR_STATE, "longconv: scratch too small (%zu < %zu); call clm_reserve with max_T >= %d", scratch_bytes, needb, T);
  }
  switch (pl.logn) {
    case 8: return conv_t<8>(c, p, grid, st);
    case 9: return conv_t<9>(c, p, grid, st);
    case 10: return conv_t<10>(c, p, grid, st);
    case 11: return conv_t<11>(c, p, grid, st);
    case 12: return conv_t<12>(c, p, grid, st);
    case 13: return conv_t<13>(c, p, grid, st);
    case 14: return conv_t<14>(c, p, grid, st);
  }
#endif
  return fail(c, CLM_ERR_INVALID, "longconv: no plan for T=%d", T);
}

// Reads of 2057..8200 tokens (the N = 16384 transform class).  Below 8192 tokens the input rows past T are zero
// filled (TMA bounds + block_in writes zeros for t in [T, Tp)), so the same kernel serves them.
struct TcPlan { int nc, nt; };   // transforms (chunks of 8192 tokens) per read, tail tokens finished by direct products
TcPlan tc_plan(int T) {
  const int rem = T % tc::C;
  if (T > tc::C && rem > 0 && rem <= LONGCONV_TAIL_MAX) return {T / tc::C, rem};
  return {std::max(1, (T + tc::C - 1) / tc::C), 0};
}
size_t tc_scratch_per_cta(int nc) { return nc > 1 ? (size_t)(nc - 1) * tc::N + 2 * tc::C : 0; }   // floats (parked spectra are fp16 pairs)

// Four reads per item (longconv_tc2_kernel<., true>), reads of 2 049 .. 4 096 tokens: one item costs what a two-read item
// costs (~13.5 K cycles at the capped clock: the epilogue phases set the pace, the extra step-7 MMAs hide under them), so
// the conv time of these buckets halves (profiles/r2_v3_length_sweep.txt: 4 096 tokens 1.53 -> 0.92 ms per batch,
// 3 073 tokens 2.06 -> 1.19).  Up to 2 048 tokens the N = 4 096 fp32 transform is still cheaper per read (1 537 tokens:
// 1.92 ms against 2.18).
bool tc_pack4_applies(const clm_ctx* c, int T) {
  return c->tc_conv && c->tc_pipe && c->tc_pack4 && c->layers[0].gtc4 != nullptr && T > tc::C / 4 && T <= tc::C / 2;
}

bool tc_conv_applies(const clm_ctx* c, int T) {
  // Below 2 057 tokens the fp32 FFT kernels win (N = 4 096: ~8.3 K cycles per item); from there on one tensor-core item
  // (13.4-14.6 K cycles for two reads of up to 8 192 tokens, the rows past T are zeros) beats the N = 8 192 fp32 transform
  // (~16 K cycles per item; profiles/r2_length_sweep.txt)
  if (!c->tc_conv || c->layers[0].gtc == nullptr) return false;
  if (tc_pack4_applies(c, T)) return true;
  if (T <= tc::C / 4 + LONGCONV_TAIL_MAX) return false;
  const TcPlan pl = tc_plan(T);
  return pl.nc == 1 || (c->tc_chunked && pl.nc <= std::min(c->tc_nseg, 4));   // the kernel's segment loop is unrolled for <= 4 chunks
}

// vx is fp16 here (block_in writes it that way when the tensor-core conv follows)
// vx holds a[ch] * v*x1 with a = the layer's calibrated input scale, or plain values when unit_scale is set
int launch_longconv_tc(clm_ctx* c, int layer, const __half* vx, const __nv_bfloat16* x0, __nv_bfloat16* out, int B, int T,
                       int Tp, cudaStream_t st, long long* trace = nullptr, bool unit_scale = false,
                       const float* osc_override = nullptr, const float* inva_override = nullptr) {
  if (!tc_conv_applies(c, T)) return fail(c, CLM_ERR_INVALID, "longconv_tc: no tensor-core plan for T=%d", T);
  const TcPlan pl = tc_plan(T);
  const bool whole_rows = T >= tc::C && pl.nc == 1;   // every 128-token row the kernel touches lies inside [0, Tp)
  if (!whole_rows && Tp % 128 != 0) return fail(c, CLM_ERR_INVALID, "longconv_tc: Tp must be a multiple of 128 for T=%d", T);
  const cuuint64_t n_rows = (cuuint64_t)(whole_rows ? std::min(64, Tp / 128) : Tp / 128);   // 128-token rows per channel
  if (int rc_attr = ensure_smem_attr(c, (const void*)(longconv_tc_kernel<false>), (int)(tc::SMEM_TOTAL))) return rc_attr;
  if (int rc_attr = ensure_smem_attr(c, (const void*)(longconv_tc_kernel<true>), (int)(tc::SMEM_TOTAL))) return rc_attr;
  {
    const void* k2[] = {(const void*)(longconv_tc2_kernel<false, false, false>), (const void*)(longconv_tc2_kernel<true, false, false>),
                        (const void*)(longconv_tc2_kernel<false, true, false>),  (const void*)(longconv_tc2_kernel<true, true, false>),
                        (const void*)(longconv_tc2_kernel<false, false, true>),  (const void*)(longconv_tc2_kernel<true, false, true>)};
    for (const void* f : k2)
      if (int rc_attr = ensure_smem_attr(c, f, (int)(tc2::SMEM2_TOTAL))) return rc_attr;
  }
  const bool pack4 = tc_pack4_applies(c, T);   // four reads per item: 32-row boxes (one read's 4096 tokens) instead of 64
  const cuuint32_t box_rows = pack4 ? 32 : 64;
  if (tc_scratch_per_cta(pl.nc) * c->num_sms > c->tc_scratch_floats)
    return fail(c, CLM_ERR_STATE, "longconv_tc: scratch too small for T=%d; call clm_reserve with max_T >= %d", T, T);
  LayerW& L = c->layers[layer];
  const int D = c->cfg.d_model;
  CUtensorMap tm;
  {
    cuuint64_t dims[3] = {128, n_rows, (cuuint64_t)B * D};
    cuuint64_t strides[2] = {256, (cuuint64_t)Tp * 2};
    cuuint32_t box[3] = {64, box_rows, 1}, estr[3] = {1, 1, 1};
    CUresult r = c->encode_tiled(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<__half*>(vx), dims, strides, box, estr,
                                 CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                 CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(c, CLM_ERR_CUDA, "cuTensorMapEncodeTiled(vx fp16) failed with CUresult %d", (int)r);
  }
  CUtensorMap tmo;
  {
    cuuint64_t dims[3] = {128, n_rows, (cuuint64_t)B * D};
    cuuint64_t strides[2] = {256, (cuuint64_t)Tp * 2};
    cuuint32_t box[3] = {128, box_rows, 1}, estr[3] = {1, 1, 1};
    CUresult r = c->encode_tiled(&tmo, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, out, dims, strides, box, estr,
                                 CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                 CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(c, CLM_ERR_CUDA, "cuTensorMapEncodeTiled(conv out) failed with CUresult %d", (int)r);
  }
  CUtensorMap tmg;
  {
    cuuint64_t dims[3] = {128, n_rows, (cuuint64_t)B * D};
    cuuint64_t strides[2] = {256, (cuuint64_t)Tp * 2};
    cuuint32_t box[3] = {128, box_rows, 1}, estr[3] = {1, 1, 1};
    CUresult r = c->encode_tiled(&tmg, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<__nv_bfloat16*>(x0), dims, strides, box, estr,
                                 CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                 CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(c, CLM_ERR_CUDA, "cuTensorMapEncodeTiled(conv gate) failed with CUresult %d", (int)r);
  }
  LongConvTcParams p{};
  p.T = T; p.vx = vx; p.k = L.k; p.dbias = L.fbias; p.Lk = c->Lk;
  p.x0 = x0; p.out = out; p.S = reinterpret_cast<const uint4*>(c->tc_S); p.G = reinterpret_cast<const uint4*>(L.gtc);
  p.B = B; p.D = D; p.Tp = Tp; p.n_pairs = pack4 ? (B + 3) / 4 : (B + 1) / 2; p.n_items = D * p.n_pairs; p.trace = trace;
  if (pack4) { p.G = reinterpret_cast<const uint4*>(L.gtc4); p.osc_adj = L.tc_adj4; }
  p.helpers_low = c->tc_helpers_low;
  // chunked reads on the two-in-flight kernel: V-form tables (H_0 = G_0, so the output scale is unchanged)
  const bool pipe_ch = pl.nc > 1 && c->tc_pipe && c->tc_pipe_chunked && L.gtcH != nullptr;
  p.n_chunks = pl.nc; p.nt = pl.nt; p.scratch = c->tc_scratch; p.scratch_per_cta = (long long)tc_scratch_per_cta(pl.nc);
  p.g_seg_stride = (long long)D * (tc::N / 4);
  p.osc = osc_override ? osc_override : (unit_scale ? L.unit_osc : L.tc_osc);
  p.inva = inva_override ? inva_override : (unit_scale ? L.unit_inva : L.tc_inva);
  p.rel = L.tc_rel; p.err = (unit_scale || osc_override) ? c->d_err + 1 : c->d_err;
  const int grid = std::min(p.n_items, c->num_sms);
  if (pipe_ch) {
    p.G = reinterpret_cast<const uint4*>(L.gtcH);
    p.rel = L.tc_relH;
    if (trace) longconv_tc2_kernel<true, false, true><<<grid, tc2::THREADS2, tc2::SMEM2_TOTAL, st>>>(tm, tmo, tmg, p);
    else launch_k(c, longconv_tc2_kernel<false, false, true>, dim3(grid), dim3(tc2::THREADS2), tc2::SMEM2_TOTAL, st, tm, tmo, tmg, p);
  }
  else if (pl.nc > 1) longconv_tc_kernel<true><<<grid, tc::THREADS_CH, tc::SMEM_TOTAL, st>>>(tm, tmo, tmg, p);
  else if (pack4 && trace) longconv_tc2_kernel<true, true, false><<<grid, tc2::THREADS2, tc2::SMEM2_TOTAL, st>>>(tm, tmo, tmg, p);
  else if (pack4) launch_k(c, longconv_tc2_kernel<false, true, false>, dim3(grid), dim3(tc2::THREADS2), tc2::SMEM2_TOTAL, st, tm, tmo, tmg, p);
  else if (c->tc_pipe && trace) longconv_tc2_kernel<true, false, false><<<grid, tc2::THREADS2, tc2::SMEM2_TOTAL, st>>>(tm, tmo, tmg, p);
  else if (c->tc_pipe) launch_k(c, longconv_tc2_kernel<false, false, false>, dim3(grid), dim3(tc2::THREADS2), tc2::SMEM2_TOTAL, st, tm, tmo, tmg, p);
  else longconv_tc_kernel<false><<<grid, tc::THREADS, tc::SMEM_TOTAL, st>>>(tm, tmo, tmg, p);
  CLM_LAUNCH_CHECK(c, pl.nc > 1 ? "longconv_tc_chunked" : (c->tc_pipe ? "longconv_tc2" : "longconv_tc"));
  return 0;
}

int round_up(int x, int m) { return (x + m - 1) / m * m; }

enum ProfCat { PC_ENCODE = 0, PC_EMBED, PC_LN, PC_GEMM_IN, PC_SHORTCONV, PC_LONGCONV, PC_TRANSPOSE, PC_GEMM_OUT,
               PC_GEMM_FC1, PC_GEMM_FC2, PC_SCORE, PC_POOL, PC_HEAD, PC_BLOCK_MLP, PC_BLOCK_IN, PC_EMBED_IN, PC_HEAD_TRAIN, PC_COUNT };
const char* kProfNames[PC_COUNT] = {"encode", "embed", "layernorm", "gemm_in_proj", "shortconv_gate", "longconv",
                                    "transpose", "gemm_out_proj", "gemm_fc1", "gemm_fc2", "gemm_score", "pool",
                                    "head", "block_mlp", "block_in", "embed_in", "head_train"};

struct ProfScope {
  clm_ctx* c;
  cudaStream_t st;
  size_t idx = (size_t)-1;
  ProfScope(clm_ctx* c_, int cat, cudaStream_t st_) : c(c_), st(st_) {
    if (!c->prof_on) return;
    if (c->prof_used * 2 + 2 > c->prof_pool.size()) {
      cudaEvent_t a, b;
      if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) return;
      c->prof_pool.push_back(a);
      c->prof_pool.push_back(b);
      c->prof_cat.push_back(cat);
    }
    idx = c->prof_used++;
    c->prof_cat[idx] = cat;
    cudaEventRecord(c->prof_pool[2 * idx], st);
  }
  ~ProfScope() {
    if (idx != (size_t)-1) cudaEventRecord(c->prof_pool[2 * idx + 1], st);
  }
};

void prof_collect(clm_ctx* c) {
  for (size_t i = 0; i < c->prof_used; ++i) {
    float ms = 0.f;
    if (cudaEventSynchronize(c->prof_pool[2 * i + 1]) == cudaSuccess &&
        cudaEventElapsedTime(&ms, c->prof_pool[2 * i], c->prof_pool[2 * i + 1]) == cudaSuccess) {
      c->prof_ms[c->prof_cat[i]] += ms;
      c->prof_n[c->prof_cat[i]] += 1;
    }
  }
  c->prof_used = 0;
}

}  // namespace

// =============================================================================================
extern "C" {

void clm_default_config(clm_config* cfg) {
  cfg->d_model = 256; cfg->n_layer = 4; cfg->d_inner = 1024; cfg->vocab_rows = 16; cfg->max_seq_len = 32770;
  cfg->filter_order = 64; cfg->emb_dim = 5; cfg->short_filter_order = 3; cfg->num_inner_mlps = 2;
  cfg->head_hidden = 512; cfg->num_classes = 2;
  cfg->layer_norm_eps = 1e-5f; cfg->filter_shift = 0.05f;
  cfg->pooling = 0;
}

const char* clm_version(void) { return "chimeralm_b200 0.1 (sm_100a)"; }

const char* clm_last_error(const clm_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

long long clm_launch_count(const clm_ctx* ctx) { return ctx ? ctx->launches : 0; }

int clm_create(const clm_config* cfg, int device, clm_ctx** out) {
  if (!cfg || !out) return CLM_ERR_INVALID;
  *out = nullptr;
  // The kernels are specialised for the named architecture; refuse anything else loudly.
  if (cfg->d_model != 256 || cfg->d_inner != 1024 || cfg->head_hidden != 512 || cfg->num_classes != 2 ||
      cfg->short_filter_order != 3 || cfg->filter_order > 64 || cfg->num_inner_mlps != 2 || cfg->n_layer < 1 ||
      cfg->vocab_rows < 1 || cfg->vocab_rows > 16 || cfg->pooling < 0 || cfg->pooling > 3)
    return CLM_ERR_INVALID;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return CLM_ERR_CUDA;
  clm_ctx* c = new (std::nothrow) clm_ctx();
  if (!c) return CLM_ERR_NOMEM;
  c->cfg = *cfg;
  c->device = device;
  *out = c;
  CLM_CUDA(c, cudaSetDevice(device));
  cudaDeviceProp prop;
  CLM_CUDA(c, cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail(c, CLM_ERR_CUDA, "device %d is sm_%d%d; this library contains sm_100a code only", device, prop.major, prop.minor);
  c->num_sms = prop.multiProcessorCount;
  cudaDriverEntryPointQueryResult qres;
  void* fn = nullptr;
  CLM_CUDA(c, cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
  if (!fn || qres != cudaDriverEntryPointSuccess) return fail(c, CLM_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
  c->encode_tiled = reinterpret_cast<EncodeTiledFn>(fn);
  CLM_CUDA(c, cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
  CLM_CUDA(c, cudaStreamCreateWithFlags(&c->h2d_stream, cudaStreamNonBlocking));
  CLM_CUDA(c, cudaStreamCreateWithFlags(&c->d2h_stream, cudaStreamNonBlocking));
  uint8_t lut[256];
  memset(lut, 6, sizeof lut);  // [UNK]
  lut['A'] = 7; lut['C'] = 8; lut['G'] = 9; lut['T'] = 10; lut['N'] = 11;
  CLM_CUDA(c, cudaMemcpyToSymbol(c_base_lut, lut, sizeof lut));
  int rc = dev_alloc(c, &c->d_err, 2);   // [0] the forward's status word, [1] the unit-level entry points' own
  if (rc) return rc;
  CLM_CUDA(c, cudaMemset(c->d_err, 0, 2 * sizeof(int)));
  CLM_CUDA(c, cudaHostAlloc(reinterpret_cast<void**>(&c->h_status), 8 * sizeof(int), cudaHostAllocMapped | cudaHostAllocPortable));
  memset(c->h_status, 0xff, 8 * sizeof(int));
  CLM_CUDA(c, cudaHostGetDevicePointer(reinterpret_cast<void**>(&c->d_status_map), c->h_status, 0));
  c->layers.resize(cfg->n_layer);
  return 0;
}

void clm_destroy(clm_ctx* c) {
  if (!c) return;
  if (g_const_owner[c->device & 63] == c) g_const_owner[c->device & 63] = nullptr;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  for (void* p : c->owned)
    if (p) cudaFree(p);
  for (cudaEvent_t e : c->prof_pool) cudaEventDestroy(e);
  if (c->own_stream) cudaStreamDestroy(c->own_stream);
  if (c->h2d_stream) cudaStreamDestroy(c->h2d_stream);
  if (c->d2h_stream) cudaStreamDestroy(c->d2h_stream);
  if (c->h_status) cudaFreeHost(c->h_status);
  for (auto& sl : c->slot)
    for (cudaEvent_t e : {sl.done, sl.h2d_done, sl.fwd_done})
      if (e) cudaEventDestroy(e);
  delete c;
}

int clm_load_tensor(clm_ctx* c, const char* name, const void* data, int dtype, const int64_t* shape, int ndim) {
  if (!c || !name || !data || ndim < 0 || ndim > 8) return fail(c, CLM_ERR_INVALID, "clm_load_tensor: bad argument");
  if (dtype != CLM_F32) return fail(c, CLM_ERR_INVALID, "clm_load_tensor('%s'): only float32 host tensors are accepted", name);
  if (c->finalized) return fail(c, CLM_ERR_STATE, "clm_load_tensor after clm_finalize");
  const std::string n(name);
  if (n.rfind("net.", 0) != 0) return 1;  // not a model weight: ignored
  CLM_CUDA(c, cudaSetDevice(c->device));
  Tensor t;
  t.numel = 1;
  for (int i = 0; i < ndim; ++i) {
    t.shape.push_back(shape[i]);
    t.numel *= shape[i];
  }
  if (t.numel <= 0) return fail(c, CLM_ERR_INVALID, "clm_load_tensor('%s'): empty tensor", name);
  int rc = dev_alloc(c, &t.d, (size_t)t.numel);
  if (rc) return rc;
  CLM_CUDA(c, cudaMemcpy(t.d, data, (size_t)t.numel * sizeof(float), cudaMemcpyHostToDevice));
  c->w[n] = t;
  return 0;
}

// What the forward reads of the attention scorer, derived from attention.0.{weight,bias} and ln_f: the bf16 weights of the
// unfolded path and ln_f's affine folded into the scorer (W0' = W0 diag(g), b0' = b0 + W0 beta) for score_pool_kernel.
// clm_finalize builds them; clm_head_train_step rebuilds them in place after every optimizer step (same buffers, so the
// tensor maps stay valid).
static int refresh_scorer(clm_ctx* c, cudaStream_t st) {
  const int D = c->cfg.d_model;
  const long long n = (long long)D * D;
  f32_to_bf16_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(c->att0_w32, c->att0_w, n);
  CLM_LAUNCH_CHECK(c, "f32_to_bf16");
  fold_ln_kernel<<<D, 256, 0, st>>>(c->att0_w32, c->att0_b, c->lnf_g, c->lnf_b, c->att0_wf32, c->att0_bf, D);
  CLM_LAUNCH_CHECK(c, "fold_ln_f");
  f32_to_bf16_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(c->att0_wf32, c->att0_wf, n);
  CLM_LAUNCH_CHECK(c, "f32_to_bf16");
  return 0;
}

// Input scale of the tensor-core convolution, per layer and channel: one small forward (fp32 convolution) over a fixed
// synthetic draw - a read of random bases and a half-[PAD] read, the two regimes real batches consist of - records
// max |v * x1|, and tc::scales_kernel turns it into the power-of-two factors block_in / longconv_tc apply.  LayerNorm
// sits in front of in_proj, so these magnitudes are set by the weights, not by the read; what the draw cannot know is
// covered by the headroom (tc::scales_kernel) and, beyond that, by the non-finite check + fp32 rerun.
static int calibrate_tc_scales(clm_ctx* c) {
  const int B = 2, T = std::min(1024, c->cfg.max_seq_len), D = c->cfg.d_model;
  int rc = clm_reserve(c, B, T);
  if (rc) return rc;
  std::vector<uint8_t> ids((size_t)B * T);
  uint32_t x = 20251018u;
  for (int b = 0; b < B; ++b)
    for (int t = 0; t < T; ++t) {
      x = x * 1664525u + 1013904223u;
      uint8_t id = (uint8_t)(7 + ((x >> 24) & 3));
      if (b == 1 && t < T / 2) id = 4;   // [PAD] prefix of a left-padded batch
      if (t == T - 1) id = 1;            // [SEP]
      ids[(size_t)b * T + t] = id;
    }
  CLM_CUDA(c, cudaMemcpy(c->st_ids, ids.data(), ids.size(), cudaMemcpyHostToDevice));
  c->calibrating = true;
  rc = clm_forward(c, c->st_ids, CLM_U8, B, T, c->st_logits, c->st_labels, c->own_stream);
  c->calibrating = false;
  if (rc) return rc;
  for (auto& L : c->layers) {
    tc::scales_kernel<<<(D + 255) / 256, 256, 0, c->own_stream>>>(L.gexp, L.vx_amax, L.vx_scale, L.tc_osc, L.tc_inva, L.tc_rel, D, c->tc_nseg, 0);
    CLM_LAUNCH_CHECK(c, "tc_scales");
  }
  CLM_CUDA(c, cudaStreamSynchronize(c->own_stream));
  return 0;
}

int clm_finalize(clm_ctx* c) {
  if (!c) return CLM_ERR_INVALID;
  if (c->finalized) return 0;
  CLM_CUDA(c, cudaSetDevice(c->device));
  const clm_config& g = c->cfg;
  const int D = g.d_model, F = g.filter_order, E = g.emb_dim, Lmax = g.max_seq_len;
  const std::string BB = "net.backbone.backbone.", HD = "net.head.";
  int rc;
#define NEED(name, numel, dst)                         \
  if ((rc = need(c, name, numel, dst)) != 0) return rc
  NEED(BB + "embeddings.word_embeddings.weight", (int64_t)g.vocab_rows * D, &c->emb);
  NEED(BB + "ln_f.weight", D, &c->lnf_g);
  NEED(BB + "ln_f.bias", D, &c->lnf_b);
  c->Lk = round_up(Lmax, 64);
  for (int l = 0; l < g.n_layer; ++l) {
    LayerW& L = c->layers[l];
    const std::string P = BB + "layers." + std::to_string(l) + ".";
    const float *in_w, *out_w, *fc1_w, *fc2_w;
    NEED(P + "norm1.weight", D, &L.ln1_g);
    NEED(P + "norm1.bias", D, &L.ln1_b);
    NEED(P + "norm2.weight", D, &L.ln2_g);
    NEED(P + "norm2.bias", D, &L.ln2_b);
    NEED(P + "mixer.in_proj.weight", 3LL * D * D, &in_w);
    NEED(P + "mixer.in_proj.bias", 3LL * D, &L.in_b);
    NEED(P + "mixer.out_proj.weight", (int64_t)D * D, &out_w);
    NEED(P + "mixer.out_proj.bias", D, &L.out_b);
    NEED(P + "mixer.short_filter.weight", 3LL * D * 3, &L.sc_w);
    NEED(P + "mixer.short_filter.bias", 3LL * D, &L.sc_b);
    NEED(P + "mixer.filter_fn.bias", D, &L.fbias);
    NEED(P + "mlp.fc1.weight", (int64_t)g.d_inner * D, &fc1_w);
    NEED(P + "mlp.fc1.bias", g.d_inner, &L.fc1_b);
    NEED(P + "mlp.fc2.weight", (int64_t)g.d_inner * D, &fc2_w);
    NEED(P + "mlp.fc2.bias", D, &L.fc2_b);
    if ((rc = to_bf16(c, in_w, 3LL * D * D, &L.in_w))) return rc;
    if ((rc = to_bf16(c, out_w, (int64_t)D * D, &L.out_w))) return rc;
    if ((rc = to_bf16(c, fc1_w, (int64_t)g.d_inner * D, &L.fc1_w))) return rc;
    if ((rc = to_bf16(c, fc2_w, (int64_t)g.d_inner * D, &L.fc2_w))) return rc;
    if ((rc = make_tmap_bf16_2d(c, &L.tm_in, L.in_w, 3 * D, D, 128))) return rc;
    {
      float* wf = nullptr;
      if ((rc = dev_alloc(c, &wf, (size_t)3 * D * D))) return rc;
      if ((rc = dev_alloc(c, &L.in_bf, (size_t)3 * D))) return rc;
      fold_ln_kernel<<<3 * D, 256>>>(in_w, L.in_b, L.ln1_g, L.ln1_b, wf, L.in_bf, D);
      CLM_LAUNCH_CHECK(c, "fold_ln");
      if ((rc = retile(c, wf, 3 * D, D, 128, &L.in_wf, &L.tm_inf))) return rc;
      L.in_wf32 = wf;
#ifdef CLM_EXPERIMENTS
      if ((rc = make_tmap_retiled(c, &L.tm_inf_h, L.in_wf, (long long)3 * D * D / 64, 128))) return rc;
#endif
    }
    if ((rc = make_tmap_bf16_2d(c, &L.tm_out, L.out_w, D, D, 128))) return rc;
    if ((rc = make_tmap_bf16_2d(c, &L.tm_fc1, L.fc1_w, g.d_inner, D, 128))) return rc;
    if ((rc = make_tmap_bf16_2d(c, &L.tm_fc2, L.fc2_w, D, g.d_inner, 128))) return rc;
    {
      if (l >= bm::MAX_LAYERS) return fail(c, CLM_ERR_INVALID, "n_layer > %d not supported by the fused block kernel", bm::MAX_LAYERS);
      // LayerNorm2 affine folded into fc1: W1' = W1 diag(gamma2), b1' = b1 + W1 beta2
      float *w1f = nullptr, *b1f = nullptr;
      if ((rc = dev_alloc(c, &w1f, (size_t)g.d_inner * D))) return rc;
      if ((rc = dev_alloc(c, &b1f, (size_t)g.d_inner))) return rc;
      fold_ln_kernel<<<g.d_inner, 256>>>(fc1_w, L.fc1_b, L.ln2_g, L.ln2_b, w1f, b1f, D);
      CLM_LAUNCH_CHECK(c, "fold_ln2");
      // the fused block tail works on h = fc1(x) / 2 (bm::gelu_tanh_bf16x2): halve W1' and b1' (exact)
      scale_f32_kernel<<<(unsigned)(((size_t)g.d_inner * D + 255) / 256), 256>>>(w1f, (long long)g.d_inner * D, 0.5f);
      scale_f32_kernel<<<(unsigned)((g.d_inner + 255) / 256), 256>>>(b1f, g.d_inner, 0.5f);
      CLM_LAUNCH_CHECK(c, "scale_fc1");
      if ((rc = retile(c, out_w, D, D, 256, &L.out_wt, &L.tm_out_t))) return rc;
      if ((rc = retile(c, w1f, g.d_inner, D, 128, &L.fc1_wt, &L.tm_fc1_t))) return rc;
      if ((rc = retile(c, fc2_w, D, g.d_inner, 256, &L.fc2_wt, &L.tm_fc2_t))) return rc;
#ifdef CLM_EXPERIMENTS
      if ((rc = retile(c, w1f, g.d_inner, D, 64, &L.fc1_w64, &L.tm_fc1_64))) return rc;
      if ((rc = make_tmap_retiled(c, &L.tm_out_h, L.out_wt, (long long)D * D / 64, 128))) return rc;
      if ((rc = make_tmap_retiled(c, &L.tm_fc1_h, L.fc1_wt, (long long)g.d_inner * D / 64, 64))) return rc;
      if ((rc = make_tmap_retiled(c, &L.tm_fc2_h, L.fc2_wt, (long long)g.d_inner * D / 64, 128))) return rc;
#endif
      if ((int)c->h_mlp.size() <= l) c->h_mlp.resize(l + 1);
      bm::LayerConsts& hc = c->h_mlp[l];
      CLM_CUDA(c, cudaMemcpy(hc.b_out, L.out_b, sizeof hc.b_out, cudaMemcpyDeviceToHost));
      CLM_CUDA(c, cudaMemcpy(hc.b2, L.fc2_b, sizeof hc.b2, cudaMemcpyDeviceToHost));
      CLM_CUDA(c, cudaMemcpy(hc.b1, b1f, sizeof hc.b1, cudaMemcpyDeviceToHost));
    }
    // implicit filter k[l] = HyenaFilter.filter(Lmax)
    FilterGenParams fp{};
    const std::string Q = P + "mixer.filter_fn.";
    NEED(Q + "pos_emb.z", (int64_t)Lmax * E, &fp.z);
    NEED(Q + "pos_emb.t", Lmax, &fp.tpos);
    NEED(Q + "implicit_filter.0.weight", (int64_t)F * E, &fp.w[0]);
    NEED(Q + "implicit_filter.0.bias", F, &fp.b[0]);
    NEED(Q + "implicit_filter.1.freq", F, &fp.freq[0]);
    NEED(Q + "implicit_filter.2.weight", (int64_t)F * F, &fp.w[1]);
    NEED(Q + "implicit_filter.2.bias", F, &fp.b[1]);
    NEED(Q + "implicit_filter.3.freq", F, &fp.freq[1]);
    NEED(Q + "implicit_filter.4.weight", (int64_t)F * F, &fp.w[2]);
    NEED(Q + "implicit_filter.4.bias", F, &fp.b[2]);
    NEED(Q + "implicit_filter.5.freq", F, &fp.freq[2]);
    NEED(Q + "implicit_filter.6.weight", (int64_t)D * F, &fp.w[3]);
    NEED(Q + "modulation.deltas", D, &fp.deltas);
    fp.shift = g.filter_shift; fp.E = E; fp.F = F; fp.D = D; fp.L = Lmax; fp.Lk = c->Lk;
    if ((rc = dev_alloc(c, &L.k, (size_t)D * c->Lk))) return rc;
    CLM_CUDA(c, cudaMemset(L.k, 0, (size_t)D * c->Lk * sizeof(float)));
    fp.k_out = L.k;
    filter_gen_kernel<<<Lmax, 256>>>(fp);
    CLM_LAUNCH_CHECK(c, "filter_gen");
#ifdef CLM_EXPERIMENTS
    if ((rc = spectrum_t<8>(c, L))) return rc;
    if ((rc = spectrum_t<9>(c, L))) return rc;
    if ((rc = spectrum_t<10>(c, L))) return rc;
    if ((rc = spectrum_t<11>(c, L))) return rc;
    if ((rc = spectrum_t<12>(c, L))) return rc;
    if ((rc = spectrum_t<13>(c, L))) return rc;
    if ((rc = spectrum_t<14>(c, L))) return rc;
#endif
    if ((rc = spectrum_fast_t<8>(c, L))) return rc;
    if ((rc = spectrum_fast_t<12>(c, L))) return rc;
    if ((rc = spectrum_fast_t<9>(c, L))) return rc;
    if ((rc = spectrum_fast_t<10>(c, L))) return rc;
    if ((rc = spectrum_fast_t<11>(c, L))) return rc;
    if ((rc = spectrum_fast_t<13>(c, L))) return rc;
    if ((rc = spectrum_fast_t<14>(c, L))) return rc;
    if (c->cfg.max_seq_len >= tc::C) {
      c->tc_nseg = (c->cfg.max_seq_len + tc::C - 1) / tc::C;   // one spectrum table per 8192-tap filter segment
      if ((rc = dev_alloc(c, &L.gtc, (size_t)c->tc_nseg * D * tc::N))) return rc;
      if ((rc = dev_alloc(c, &L.gexp, (size_t)c->tc_nseg * D))) return rc;
      CLM_CUDA(c, cudaFuncSetAttribute(tc::spectrum_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::N * (int)sizeof(float2)));
      tc::spectrum_kernel<<<dim3(D, c->tc_nseg), 256, tc::N * sizeof(float2)>>>(L.k, c->Lk, c->cfg.max_seq_len, L.fbias, L.gtc, L.gexp);
      CLM_LAUNCH_CHECK(c, "tc_spectrum");
      float** arrs[] = {&L.vx_scale, &L.tc_osc, &L.tc_inva, &L.unit_scale, &L.unit_osc, &L.unit_inva};
      for (float** a : arrs)
        if ((rc = dev_alloc(c, a, (size_t)D))) return rc;
      if ((rc = dev_alloc(c, &L.tc_rel, (size_t)c->tc_nseg * D))) return rc;
      if ((rc = dev_alloc(c, &L.vx_amax, (size_t)D))) return rc;
      CLM_CUDA(c, cudaMemset(L.vx_amax, 0, D * sizeof(unsigned int)));
      // until the calibration forward at the end of clm_finalize has run, both sets are the unit-input-scale ones
      tc::scales_kernel<<<(D + 255) / 256, 256>>>(L.gexp, nullptr, L.unit_scale, L.unit_osc, L.unit_inva, L.tc_rel, D, c->tc_nseg, 0);
      tc::scales_kernel<<<(D + 255) / 256, 256>>>(L.gexp, nullptr, L.vx_scale, L.tc_osc, L.tc_inva, L.tc_rel, D, c->tc_nseg, 0);
      CLM_LAUNCH_CHECK(c, "tc_scales");
      // the same filter truncated to its first 4096 taps (all a read of <= 4096 tokens can see): four reads per transform
      if ((rc = dev_alloc(c, &L.gtc4, (size_t)D * tc::N))) return rc;
      if ((rc = dev_alloc(c, &L.gexp4, (size_t)D))) return rc;
      if ((rc = dev_alloc(c, &L.tc_adj4, (size_t)D))) return rc;
      tc::spectrum_kernel<<<dim3(D, 1), 256, tc::N * sizeof(float2)>>>(L.k, c->Lk, std::min(c->cfg.max_seq_len, tc::C / 2), L.fbias, L.gtc4, L.gexp4);
      tc::exp_adj_kernel<<<(D + 255) / 256, 256>>>(L.gexp, L.gexp4, L.tc_adj4, D);
      CLM_LAUNCH_CHECK(c, "tc_spectrum4");
      if (c->tc_nseg > 1) {
        if ((rc = dev_alloc(c, &L.gtcH, (size_t)c->tc_nseg * D * tc::N))) return rc;
        if ((rc = dev_alloc(c, &L.gexpH, (size_t)c->tc_nseg * D))) return rc;
        if ((rc = dev_alloc(c, &L.tc_relH, (size_t)c->tc_nseg * D))) return rc;
        tc::spectrum_kernel<<<dim3(D, c->tc_nseg), 256, tc::N * sizeof(float2)>>>(L.k, c->Lk, c->cfg.max_seq_len, L.fbias, L.gtcH, L.gexpH, 1);
        tc::rel_kernel<<<(D + 255) / 256, 256>>>(L.gexpH, L.tc_relH, D, c->tc_nseg);
        CLM_LAUNCH_CHECK(c, "tc_spectrumH");
      }
    }
  }
  if ((rc = dev_alloc(c, &c->tc_S, (size_t)tc::S_BYTES / 2))) return rc;
  tc::build_s_kernel<<<(tc::S_ROWS * 128 + 255) / 256, 256>>>(c->tc_S);
  CLM_LAUNCH_CHECK(c, "tc_build_s");
  if ((rc = dev_alloc(c, &c->head_counter, 1))) return rc;
  CLM_CUDA(c, cudaMemset(c->head_counter, 0, sizeof(unsigned int)));
  c->head_base = 0;
  // head
  const float *a0w, *a2b;
  if (g.pooling == 0) {
    NEED(HD + "attention.0.weight", (int64_t)D * D, &a0w);
    NEED(HD + "attention.0.bias", D, &c->att0_b);
    NEED(HD + "attention.2.weight", D, &c->att2_w);
    NEED(HD + "attention.2.bias", 1, &a2b);
    CLM_CUDA(c, cudaMemcpy(&c->att2_b, a2b, sizeof(float), cudaMemcpyDeviceToHost));
  } else {
    // mean / max / cls pooling: the module has no scorer (components/hyena.py:50-53); the kernels still run the scorer
    // GEMM on zero weights and ignore its scores, so the one fused tail serves every pooling type
    float* z = nullptr;
    if ((rc = dev_alloc(c, &z, (size_t)D * D + 2 * D))) return rc;
    CLM_CUDA(c, cudaMemset(z, 0, ((size_t)D * D + 2 * D) * sizeof(float)));
    a0w = z; c->att0_b = z + (size_t)D * D; c->att2_w = z + (size_t)D * D + D; c->att2_b = 0.f;
  }
  c->att0_w32 = a0w;
  if ((rc = dev_alloc(c, &c->att0_w, (size_t)D * D))) return rc;
  if ((rc = dev_alloc(c, &c->att0_wf32, (size_t)D * D))) return rc;
  if ((rc = dev_alloc(c, &c->att0_bf, (size_t)D))) return rc;
  if ((rc = dev_alloc(c, &c->att0_wf, (size_t)D * D))) return rc;
  if ((rc = refresh_scorer(c, 0))) return rc;
  if ((rc = make_tmap_bf16_2d(c, &c->tm_att0, c->att0_w, D, D, 256))) return rc;
  {
    if ((rc = make_tmap_bf16_2d(c, &c->tm_att0f, c->att0_wf, D, D, 256))) return rc;
    if ((rc = dev_alloc(c, &c->emb_norm, (size_t)g.vocab_rows * D))) return rc;
    embed_norm_table_kernel<<<g.vocab_rows, 32>>>(c->emb, c->emb_norm, g.vocab_rows, g.layer_norm_eps);
    CLM_LAUNCH_CHECK(c, "embed_norm_table");
    if (g.n_layer > 0 && g.vocab_rows <= ei::NV && D == ei::D && c->layers[0].in_wf32) {
      if ((rc = dev_alloc(c, &c->u_tab0, (size_t)3 * D * ei::NV))) return rc;
      embed_in_table_kernel<<<3 * D, 32>>>(c->layers[0].in_wf32, c->layers[0].in_bf, c->emb_norm, c->u_tab0, g.vocab_rows);
      CLM_LAUNCH_CHECK(c, "embed_in_table");
      if ((rc = dev_alloc(c, &c->emb_r32, (size_t)32 * D))) return rc;
      embed_r32_table_kernel<<<32, 256>>>(c->emb, c->emb_r32, g.vocab_rows);
      CLM_LAUNCH_CHECK(c, "embed_r32_table");
    }
    std::vector<float> h1(D, 1.0f);
    if ((rc = dev_alloc(c, &c->ones, (size_t)D))) return rc;
    if ((rc = dev_alloc(c, &c->zeros, (size_t)D))) return rc;
    CLM_CUDA(c, cudaMemcpy(c->ones, h1.data(), D * sizeof(float), cudaMemcpyHostToDevice));
    CLM_CUDA(c, cudaMemset(c->zeros, 0, D * sizeof(float)));
  }
  const int H = g.head_hidden;
  NEED(HD + "classifier.0.weight", (int64_t)H * D, &c->head.w0);
  NEED(HD + "classifier.0.bias", H, &c->head.b0);
  NEED(HD + "classifier.3.weight", (int64_t)H * H, &c->head.w1);
  NEED(HD + "classifier.3.bias", H, &c->head.b1);
  NEED(HD + "classifier.6.layers.0.weight", (int64_t)H * H, &c->head.wr0);
  NEED(HD + "classifier.6.layers.0.bias", H, &c->head.br0);
  NEED(HD + "classifier.6.layers.3.weight", (int64_t)H * H, &c->head.wr1);
  NEED(HD + "classifier.6.layers.3.bias", H, &c->head.br1);
  NEED(HD + "output_layer.weight", 2LL * H, &c->head.wo);
  NEED(HD + "output_layer.bias", 2, &c->head.bo);
#undef NEED
  CLM_CUDA(c, cudaDeviceSynchronize());
  c->finalized = true;
  if (c->tc_nseg > 0 && (rc = calibrate_tc_scales(c)) != 0) {
    c->finalized = false;
    return rc;
  }
  return 0;
}

int clm_reserve(clm_ctx* c, int max_B, int max_T) {
  return clm_reserve_tokens(c, max_B, max_T, (long long)max_B * (long long)max_T);
}

int clm_reserve_tokens(clm_ctx* c, int max_B, int max_T, long long max_tokens) {
  if (!c || max_B <= 0 || max_T <= 0 || max_tokens < max_T || max_tokens > (long long)max_B * max_T || max_tokens > 0x7fffffffLL)
    return fail(c, CLM_ERR_INVALID, "clm_reserve: bad sizes");
  if (max_T > c->cfg.max_seq_len) return fail(c, CLM_ERR_INVALID, "clm_reserve: max_T=%d exceeds max_seq_len=%d", max_T, c->cfg.max_seq_len);
  CLM_CUDA(c, cudaSetDevice(c->device));
  CLM_CUDA(c, cudaDeviceSynchronize());
  // Release everything and forget the old limits FIRST: if an allocation below fails (a B x 32 769 batch that does not
  // fit), the context is left with no workspaces and max_B = max_T = 0, so every later forward is refused until a
  // smaller clm_reserve succeeds - never a launch on freed memory.
  c->max_B = c->max_T = c->Tp_max = 0;
  c->max_tokens = 0; c->ct_elems = 0; c->yg_elems = 0;
  c->scratch_bytes = 0; c->tc_scratch_floats = 0; c->st_bases_cap = 0;
  dev_release(c, &c->R); dev_release(c, &c->XN); dev_release(c, &c->U); dev_release(c, &c->VX); dev_release(c, &c->X0);
  dev_release(c, &c->Y); dev_release(c, &c->YG); dev_release(c, &c->YT); dev_release(c, &c->score); dev_release(c, &c->part);
  dev_release(c, &c->pooled); dev_release(c, &c->scratch); dev_release(c, &c->tc_scratch);
  for (auto& sl : c->slot) {
    dev_release(c, &sl.bases); dev_release(c, &sl.offsets); dev_release(c, &sl.ids); dev_release(c, &sl.logits);
    dev_release(c, &sl.labels);
    sl.busy = false;
  }
  for (int i = 0; i < 4; ++i) dev_release(c, &c->hbuf[i]);
  const int D = c->cfg.d_model;
  // token-proportional buffers are sized by the token budget, per-read ones by max_B: a context that serves length
  // buckets (256 reads of 1 kb ... 8 reads of 32 kb, <= 262 k tokens each) does not pay for 256 x 32 769 tokens
  const size_t M = (size_t)max_tokens;
  const int Tp = round_up(max_T, 128);
  const size_t CT = (size_t)D * std::min((size_t)max_B * Tp, M + (size_t)127 * max_B);   // sum over reads of round_up(T, 128)
  int rc;
  if ((rc = dev_alloc(c, &c->R, (M + 160) * D))) return rc;  // R32 layout: whole 32-row groups + tile overhang
  if ((rc = dev_alloc(c, &c->XN, M * D))) return rc;
  if ((rc = dev_alloc(c, &c->U, M * (size_t)c->cfg.d_inner))) return rc;  // in_proj out (3D) and fc1 out (d_inner)
  if ((rc = dev_alloc(c, &c->VX, CT))) return rc;
  if ((rc = dev_alloc(c, &c->X0, CT))) return rc;
  if ((rc = dev_alloc(c, &c->Y, CT))) return rc;
  {   // at most ceil(max_B / 2) gathered tiles of 128 columns
    const size_t yg = (size_t)D * bm::BM * ((size_t)(max_B + 1) / 2);
    if ((rc = dev_alloc(c, &c->YG, yg))) return rc;
    c->yg_elems = yg;
  }
  if ((rc = dev_alloc(c, &c->YT, M * D))) return rc;
  if ((rc = dev_alloc(c, &c->score, M))) return rc;
  c->n_split = std::max(1, std::min(64, (2 * c->num_sms + max_B - 1) / max_B));
  {   // pooling partials: per read max(n_split, ceil(T / 128)) slices of (2 + D) floats
    const size_t slices = std::max((size_t)max_B * c->n_split, std::min((size_t)max_B * ((max_T + 127) / 128), M / 128 + max_B));
    if ((rc = dev_alloc(c, &c->part, slices * (2 + D)))) return rc;
  }
  if ((rc = dev_alloc(c, &c->pooled, (size_t)max_B * D))) return rc;
  for (int i = 0; i < 4; ++i)
    if ((rc = dev_alloc(c, &c->hbuf[i], (size_t)max_B * c->cfg.head_hidden))) return rc;
  size_t scratch_bytes = conv_scratch_bytes(c, max_T);
  if (scratch_bytes) {
    // any T <= max_T that takes the chunked path needs at most this much
    const int C = 1 << (LONGCONV_MAX_LOGN - 1);
    const size_t worst = (size_t)c->num_sms * ((max_T + C - 1) / C) * ((size_t)1 << LONGCONV_MAX_LOGN) * sizeof(float2);
    scratch_bytes = std::max(scratch_bytes, worst);
    if ((rc = dev_alloc(c, reinterpret_cast<uint8_t**>(&c->scratch), scratch_bytes))) return rc;
    c->scratch_bytes = scratch_bytes;
  }
  {
    const size_t need = tc_scratch_per_cta(tc_plan(max_T).nc) * c->num_sms;
    if (need) {
      if ((rc = dev_alloc(c, &c->tc_scratch, need))) return rc;
      c->tc_scratch_floats = need;
    }
  }
  // staging of clm_predict_host (sized here: nothing is allocated on the forward path)
  for (auto& sl : c->slot) {
    if ((rc = dev_alloc(c, &sl.offsets, (size_t)max_B + 1))) return rc;
    if ((rc = dev_alloc(c, &sl.ids, M))) return rc;
    if ((rc = dev_alloc(c, &sl.logits, (size_t)max_B * 2))) return rc;
    if ((rc = dev_alloc(c, &sl.labels, (size_t)max_B))) return rc;
    if ((rc = dev_alloc(c, &sl.bases, M))) return rc;   // a read contributes at most one base per token
    for (cudaEvent_t* e : {&sl.done, &sl.h2d_done, &sl.fwd_done})
      if (!*e) CLM_CUDA(c, cudaEventCreateWithFlags(e, cudaEventDisableTiming));
  }
  c->st_bases_cap = M;
  c->max_B = max_B; c->max_T = max_T; c->Tp_max = Tp;   // only now: every workspace exists
  c->max_tokens = max_tokens; c->ct_elems = CT;
  return 0;
}

int clm_encode_batch(clm_ctx* c, const uint8_t* d_bases, const int64_t* d_offsets, int B, int T_pad, int add_cls,
                     int add_sep, int pad_left, int max_bases, uint8_t* d_ids_out, int32_t* d_lens_out,
                     void* stream) {
  if (!c || !d_bases || !d_offsets || !d_ids_out || B <= 0 || T_pad <= 0 || max_bases < 0)
    return fail(c, CLM_ERR_INVALID, "clm_encode_batch: bad argument");
  EncodeParams p{d_bases, d_offsets, d_ids_out, d_lens_out, B, T_pad, add_cls ? 1 : 0, add_sep ? 1 : 0, pad_left ? 1 : 0, max_bases};
  ProfScope ps_(c, PC_ENCODE, (cudaStream_t)stream);
  dim3 grid(std::min(64, (T_pad + 255) / 256), B);
  encode_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(p);
  CLM_LAUNCH_CHECK(c, "encode");
  return 0;
}

int clm_set_debug_stop(clm_ctx* c, int layer, int stage) {
  if (!c) return CLM_ERR_INVALID;
  c->dbg_layer = layer;
  c->dbg_stage = stage;
  return 0;
}

int clm_forward(clm_ctx* c, const void* d_ids, int ids_dtype, int B, int T, float* d_logits, uint8_t* d_labels,
                void* stream) {
  if (!c) return CLM_ERR_INVALID;
  if (!c->finalized) return fail(c, CLM_ERR_STATE, "clm_forward before clm_finalize");
  if (!d_ids || !d_logits || B <= 0 || T <= 0) return fail(c, CLM_ERR_INVALID, "clm_forward: bad argument");
  if (B > c->max_B || T > c->max_T || (long long)B * T > c->max_tokens)
    return fail(c, CLM_ERR_STATE, "clm_forward: batch %dx%d exceeds reserved %dx%d (%lld tokens); call clm_reserve", B, T, c->max_B, c->max_T, c->max_tokens);
  cudaStream_t st = (cudaStream_t)stream;
  const clm_config& g = c->cfg;
  const int D = g.d_model;
  const long long M = (long long)B * T;
  if (M > 0x7fffffffLL) return fail(c, CLM_ERR_INVALID, "clm_forward: B*T too large");
  const int Tp = round_up(T, 128);   // whole 128-token rows per channel: the tensor-core conv views a channel as [n1][128]
  const unsigned rows32e = (unsigned)((M + 31) / 32);   // embed_kernel: one CTA per 32-row block of the R32 layout
  const unsigned rows32 = (unsigned)((M + 31) / 32);
  int rc;
  const long long seq = ++c->fwd_seq;
  int* status_slot = c->d_status_map + (seq & 7);
  const int status_tag = (int)((seq & 0x7fffff) << 8);
#define STOP_AFTER(layer, stage) \
  if (c->dbg_layer == (layer) && c->dbg_stage == (stage)) return 0

  c->pdl_now = c->pdl && c->fused_in && c->fused_mlp && c->tc_pipe && c->dbg_layer < 0 && tc_conv_applies(c, T) &&
               (tc_plan(T).nc == 1 || c->tc_pipe_chunked);
  struct PdlReset { clm_ctx* c; ~PdlReset() { c->pdl_now = false; } } pdl_reset_{c};
  // block 0's first half reads the ids directly (table lookup), so nobody consumes the embedding's xn rows
  const bool ei0 = c->embed_in && c->u_tab0 && c->fused_in && c->dbg_layer != 0 && g.n_layer > 0 && B <= 65535;
  __nv_bfloat16* const emb_xn = ei0 ? nullptr : c->XN;
#ifdef CLM_EXPERIMENTS
  const bool mlp_product = !c->mlp_2cta && !c->mlp_pp && !c->mlp_epi16;
#else
  const bool mlp_product = true;
#endif
  // ... and block 0's second half looks its residual input up by token id: no embedding kernel at all
  const bool ei_res = ei0 && c->embed_res && c->emb_r32 && c->fused_mlp && mlp_product;
  if (!ei_res) { ProfScope ps_(c, PC_EMBED, st);
  switch (ids_dtype) {
    case CLM_U8: embed_kernel<uint8_t><<<rows32e, 256, 0, st>>>((const uint8_t*)d_ids, c->emb, c->emb_norm, c->R, emb_xn, M, D, g.vocab_rows, c->d_err); break;
    case CLM_I32: embed_kernel<int32_t><<<rows32e, 256, 0, st>>>((const int32_t*)d_ids, c->emb, c->emb_norm, c->R, emb_xn, M, D, g.vocab_rows, c->d_err); break;
    case CLM_I64: embed_kernel<int64_t><<<rows32e, 256, 0, st>>>((const int64_t*)d_ids, c->emb, c->emb_norm, c->R, emb_xn, M, D, g.vocab_rows, c->d_err); break;
    default: return fail(c, CLM_ERR_INVALID, "clm_forward: ids dtype %d not supported", ids_dtype);
  }
  CLM_LAUNCH_CHECK(c, "embed"); }
  STOP_AFTER(0, 0);
  bool xn_valid = true;   // XN holds the normalised (no affine) residual for the next LayerNorm consumer

  for (int l = 0; l < g.n_layer; ++l) {
    LayerW& L = c->layers[l];
    bool use_tc = false;   // this layer's VX is fp16 and feeds the tensor-core long convolution
    if (c->fused_in && c->dbg_layer != l) {
      if (!xn_valid) {
        ProfScope ps_(c, PC_LN, st);
        layernorm_bf16_kernel<<<rows32, 256, 0, st>>>(c->R, c->ones, c->zeros, c->XN, M, g.layer_norm_eps);
        CLM_LAUNCH_CHECK(c, "normalize");
      }
      ProfScope ps_(c, (l == 0 && ei0) ? PC_EMBED_IN : PC_BLOCK_IN, st);
      use_tc = tc_conv_applies(c, T);
      if (l == 0 && ei0) rc = launch_embed_in(c, d_ids, ids_dtype, B, T, Tp, c->VX, c->X0, st, use_tc);
      else rc = launch_block_in(c, l, c->XN, B, T, Tp, c->VX, c->X0, st, nullptr, use_tc);
      if (rc) return rc;
      if (c->calibrating && !use_tc && L.vx_amax) {
        tc::amax_cm_kernel<<<dim3(D, B), 256, 0, st>>>(c->VX, D, Tp, T, L.vx_amax);
        CLM_LAUNCH_CHECK(c, "vx_amax");
      }
    } else {
    { ProfScope ps_(c, PC_LN, st);
      layernorm_bf16_kernel<<<rows32, 256, 0, st>>>(c->R, L.ln1_g, L.ln1_b, c->XN, M, g.layer_norm_eps);
      CLM_LAUNCH_CHECK(c, "ln1"); }
      STOP_AFTER(l, 1);
      GemmParams p{};
      p.M = (int)M; p.N = 3 * D; p.K = D; p.bias = L.in_b; p.out = c->U; p.ldo = 3 * D;
      { ProfScope ps_(c, PC_GEMM_IN, st);
      if ((rc = launch_gemm(c, c->XN, L.tm_in, p, EPI_BIAS_BF16, st))) return rc; }
      STOP_AFTER(l, 2);
      { ProfScope ps_(c, PC_SHORTCONV, st);
      shortconv_gate_kernel<<<dim3((Tp + 63) / 64, D / 32, B), 256, 0, st>>>(c->U, L.sc_w, L.sc_b, c->VX, c->X0, T, Tp, D);
      CLM_LAUNCH_CHECK(c, "shortconv_gate"); }
    }
    STOP_AFTER(l, 3);
    { ProfScope ps_(c, PC_LONGCONV, st);
    if (use_tc) rc = launch_longconv_tc(c, l, reinterpret_cast<const __half*>(c->VX), c->X0, c->Y, B, T, Tp, st);
    else rc = launch_longconv(c, l, c->VX, c->X0, c->Y, B, T, Tp, c->scratch, c->scratch_bytes, st);
    if (rc) return rc; }
    STOP_AFTER(l, 4);
    const bool mlp_fused = c->fused_mlp && c->dbg_layer != l;
    if (!(mlp_fused && c->y_channel_major)) {
      ProfScope ps_(c, PC_TRANSPOSE, st);
      transpose_ct_kernel<<<dim3((T + 63) / 64, D / 64, B), 256, 0, st>>>(c->Y, c->YT, T, Tp, D);
      CLM_LAUNCH_CHECK(c, "transpose_ct");
    }
    STOP_AFTER(l, 5);
    if (mlp_fused) {
      ProfScope ps_(c, PC_BLOCK_MLP, st);
      // the last block's residual has no reader on the folded tail (scorer + pooling read xn); any debug stop keeps it
      const bool dead_res = l == g.n_layer - 1 && c->dbg_layer < 0 && c->skip_dead_res;
      const void* tab_ids = (l == 0 && ei_res) ? d_ids : nullptr;
      if (c->y_channel_major) rc = launch_block_mlp(c, l, c->Y, c->R, (int)M, st, nullptr, B, T, Tp, c->XN, dead_res, tab_ids, ids_dtype);
      else rc = launch_block_mlp(c, l, c->YT, c->R, (int)M, st, nullptr, 0, 0, 0, c->XN, dead_res, tab_ids, ids_dtype);
      if (rc) return rc;
      xn_valid = true;
    } else {
      GemmParams p{};
      p.M = (int)M; p.N = D; p.K = D; p.bias = L.out_b; p.out = c->R; p.res = c->R; p.ldo = D; p.r32 = 1;
      { ProfScope ps_(c, PC_GEMM_OUT, st);
      if ((rc = launch_gemm(c, c->YT, L.tm_out, p, EPI_BIAS_RES_F32, st))) return rc; }
      STOP_AFTER(l, 6);
      { ProfScope ps_(c, PC_LN, st);
      layernorm_bf16_kernel<<<rows32, 256, 0, st>>>(c->R, L.ln2_g, L.ln2_b, c->XN, M, g.layer_norm_eps);
      CLM_LAUNCH_CHECK(c, "ln2"); }
      STOP_AFTER(l, 7);
      p = GemmParams{};
      p.M = (int)M; p.N = g.d_inner; p.K = D; p.bias = L.fc1_b; p.out = c->U; p.ldo = g.d_inner;
      { ProfScope ps_(c, PC_GEMM_FC1, st);
      if ((rc = launch_gemm(c, c->XN, L.tm_fc1, p, EPI_BIAS_GELU_TANH, st))) return rc; }
      STOP_AFTER(l, 8);
      p = GemmParams{};
      p.M = (int)M; p.N = D; p.K = g.d_inner; p.bias = L.fc2_b; p.out = c->R; p.res = c->R; p.ldo = D; p.r32 = 1;
      { ProfScope ps_(c, PC_GEMM_FC2, st);
      if ((rc = launch_gemm(c, c->U, L.tm_fc2, p, EPI_BIAS_RES_F32, st))) return rc; }
    }
    if (!mlp_fused) xn_valid = false;
    STOP_AFTER(l, 9);
  }
  const int NL = g.n_layer;
  const bool tail_folded = xn_valid && c->dbg_layer != NL;
  if (!tail_folded) {
    ProfScope ps_(c, PC_LN, st);
    layernorm_bf16_kernel<<<rows32, 256, 0, st>>>(c->R, c->lnf_g, c->lnf_b, c->XN, M, g.layer_norm_eps);
    CLM_LAUNCH_CHECK(c, "ln_f");
  }
  STOP_AFTER(NL, 10);
  // dbg stages 11 (scores) and 12 (pooling) are separate kernels only on the unfused path
  const bool sp_fused = tail_folded && c->fused_score_pool && c->dbg_layer != NL;
  int n_split = c->n_split;
  if (sp_fused) {
    if (int rc_attr = ensure_smem_attr(c, (const void*)(score_pool_kernel), (int)(sp::SMEM_TOTAL))) return rc_attr;
    ProfScope ps_(c, PC_SCORE, st);
    CUtensorMap tmA;
    if ((rc = make_tmap_xn(c, &tmA, c->XN, B, T, sp::BM))) return rc;
    ScorePoolParams sp_{};
    sp_.b0 = c->att0_bf; sp_.w2 = c->att2_w; sp_.b2 = c->att2_b; sp_.g = c->lnf_g; sp_.beta = c->lnf_b;
    sp_.score = c->score; sp_.part = c->part; sp_.B = B; sp_.T = T;
    sp_.tiles_per_seq = (T + sp::BM - 1) / sp::BM; sp_.num_tiles = B * sp_.tiles_per_seq;
    sp_.pool_mode = g.pooling;
    n_split = sp_.tiles_per_seq;
    launch_k(c, score_pool_kernel, dim3(std::min(sp_.num_tiles, c->num_sms)), dim3(sp::THREADS), sp::SMEM_TOTAL, st, tmA, c->tm_att0f, sp_);
    CLM_LAUNCH_CHECK(c, "score_pool");
  } else {
  {
    GemmParams p{};
    p.M = (int)M; p.N = D; p.K = D; p.w2 = c->att2_w; p.b2 = c->att2_b; p.score = c->score; p.ldo = D;
    ProfScope ps_(c, PC_SCORE, st);
    if (tail_folded) {   // XN = normalised residual from the last block: ln_f's affine lives in the folded scorer weights
      p.bias = c->att0_bf;
      if ((rc = launch_gemm(c, c->XN, c->tm_att0f, p, EPI_SCORE, st))) return rc;
    } else {
      p.bias = c->att0_b;
      if ((rc = launch_gemm(c, c->XN, c->tm_att0, p, EPI_SCORE, st))) return rc;
    }
  }
  STOP_AFTER(NL, 11);
  { ProfScope ps_(c, PC_POOL, st);
  if (!tail_folded) {   // XN currently holds ln_f WITH affine (scorer input): re-emit the plain normalised rows for pooling
    ProfScope ps2_(c, PC_LN, st);
    layernorm_bf16_kernel<<<rows32, 256, 0, st>>>(c->R, c->ones, c->zeros, c->XN, M, g.layer_norm_eps);
    CLM_LAUNCH_CHECK(c, "normalize_for_pool");
  }
  pool_partial_kernel<<<dim3(c->n_split, B), 256, 0, st>>>(c->XN, c->score, c->lnf_g, c->lnf_b, c->part, T, c->n_split, g.pooling);
  CLM_LAUNCH_CHECK(c, "pool_partial"); }
  STOP_AFTER(NL, 12);
  }
  {
    ProfScope ps_(c, PC_HEAD, st);
    const HeadParams& hp = c->head;
    const int H = g.head_hidden;
    if (c->fused_head && c->head_counter && H == 512 && D == 256) {
      HeadFusedParams hf{};
      hf.part = c->part; hf.n_split = n_split;
      hf.w0 = hp.w0; hf.b0 = hp.b0; hf.w1 = hp.w1; hf.b1 = hp.b1; hf.wr0 = hp.wr0; hf.br0 = hp.br0; hf.wr1 = hp.wr1; hf.br1 = hp.br1;
      hf.wo = hp.wo; hf.bo = hp.bo;
      hf.pooled = c->pooled; hf.h0 = c->hbuf[0]; hf.h1 = c->hbuf[1]; hf.h2 = c->hbuf[2]; hf.h3 = c->hbuf[3];
      hf.logits = d_logits; hf.labels = d_labels; hf.counter = c->head_counter; hf.base = c->head_base; hf.B = B;
      hf.err = c->d_err; hf.status_out = status_slot; hf.status_tag = status_tag; hf.pool_mode = g.pooling;
      // (H / 8) neuron groups x up to 4 read slices of whole 32-read tiles; 256 CTAs of 64 KB are co-resident on 148 SMs
      const int slices = std::max(1, std::min(4, (B + HEAD_BT - 1) / HEAD_BT));
      const dim3 grid(H / 8, slices);
      void* args[] = {&hf};
      constexpr size_t head_smem = (size_t)HEAD_BT * 512 * sizeof(float);
      if (int rc_attr = ensure_smem_attr(c, (const void*)(head_fused_kernel), (int)((int)head_smem))) return rc_attr;
      if (c->head_coop) CLM_CUDA(c, cudaLaunchCooperativeKernel((const void*)head_fused_kernel, grid, dim3(256), args, head_smem, st));
      else head_fused_kernel<<<grid, 256, head_smem, st>>>(hf);
      CLM_LAUNCH_CHECK(c, "head_fused");
      // five grid barriers + one final arrival per CTA and launch; the device counter is never reset.  Advanced only once
      // the launch was accepted: a rejected launch must not move the host's idea of the counter ahead of the device's.
      c->head_base += 6u * (unsigned)(grid.x * grid.y);
    } else {
    pool_merge_kernel<<<B, 256, 0, st>>>(c->part, n_split, c->pooled, g.pooling);
    CLM_LAUNCH_CHECK(c, "pool_merge");
    head_layer_kernel<256, true, false, false><<<dim3(H / 8, (B + 31) / 32), 256, 0, st>>>(hp.w0, hp.b0, c->pooled, nullptr, c->hbuf[0], nullptr, B, H);
    CLM_LAUNCH_CHECK(c, "head_l0");
    head_layer_kernel<512, true, false, false><<<dim3(H / 8, (B + 31) / 32), 256, 0, st>>>(hp.w1, hp.b1, c->hbuf[0], nullptr, c->hbuf[1], nullptr, B, H);
    CLM_LAUNCH_CHECK(c, "head_l1");
    head_layer_kernel<512, true, false, false><<<dim3(H / 8, (B + 31) / 32), 256, 0, st>>>(hp.wr0, hp.br0, c->hbuf[1], nullptr, c->hbuf[2], nullptr, B, H);
    CLM_LAUNCH_CHECK(c, "head_r0");
    head_layer_kernel<512, false, true, false><<<dim3(H / 8, (B + 31) / 32), 256, 0, st>>>(hp.wr1, hp.br1, c->hbuf[2], c->hbuf[1], c->hbuf[3], nullptr, B, H);
    CLM_LAUNCH_CHECK(c, "head_r1");
    head_layer_kernel<512, false, false, true><<<dim3(1, (B + 31) / 32), 256, 0, st>>>(hp.wo, hp.bo, c->hbuf[3], nullptr, d_logits, d_labels, B, 2);
    CLM_LAUNCH_CHECK(c, "head_out");
    publish_status_kernel<<<1, 1, 0, st>>>(c->d_err, status_slot, status_tag);
    CLM_LAUNCH_CHECK(c, "publish_status");
    }
  }
#undef STOP_AFTER
  c->last_B = B; c->last_T = T;
  return 0;
}

long long clm_forward_seq(const clm_ctx* c) { return c ? c->fwd_seq : 0; }

int clm_forward_status(clm_ctx* c, long long seq) {
  if (!c) return CLM_ERR_INVALID;
  if (seq <= 0 || seq > c->fwd_seq || seq + 8 <= c->fwd_seq)
    return fail(c, CLM_ERR_INVALID, "clm_forward_status: forward %lld is not one of the last 8 (latest is %lld)", seq, c->fwd_seq);
  const int v = *reinterpret_cast<volatile int*>(c->h_status + (seq & 7));
  if ((v >> 8) != (int)(seq & 0x7fffff))
    return fail(c, CLM_ERR_STATE, "clm_forward_status: forward %lld has not completed; synchronise its stream first", seq);
  if (v & 1) return fail(c, CLM_ERR_TOKEN_RANGE, "forward %lld: a token id lies outside [0, %d) (the reference's nn.Embedding raises IndexError)", seq, c->cfg.vocab_rows);
  if (v & 2) return fail(c, CLM_ERR_FP16_RANGE, "forward %lld: the fp16 tensor-core long convolution produced a non-finite value; "
                         "rerun the batch with clm_set_option(\"tc_conv\", 0) (clm_predict_host does so by itself)", seq);
  return 0;
}

int clm_predict_host_submit(clm_ctx* c, const uint8_t* h_bases, const int64_t* h_offsets, int B, int T_pad, int add_cls,
                            int add_sep, int pad_left, int max_bases, float* h_logits, uint8_t* h_labels, int* ticket) {
  if (!c || !h_bases || !h_offsets || !h_logits || !ticket || B <= 0) return fail(c, CLM_ERR_INVALID, "clm_predict_host: bad argument");
  if (B > c->max_B || T_pad > c->max_T || (long long)B * T_pad > c->max_tokens)
    return fail(c, CLM_ERR_STATE, "clm_predict_host: batch %dx%d exceeds reserved %dx%d (%lld tokens)", B, T_pad, c->max_B, c->max_T, c->max_tokens);
  CLM_CUDA(c, cudaSetDevice(c->device));
  const size_t nbytes = (size_t)h_offsets[B];
  // the staging buffers were sized by clm_reserve (one base per token of the budget); nothing is allocated here.  Bases
  // beyond max_bases per read are never looked at by the encoder, but they still have to fit the copy.
  if (nbytes > c->st_bases_cap)
    return fail(c, CLM_ERR_STATE, "clm_predict_host: %zu bases exceed the staging buffer of %zu reserved by clm_reserve(%d, %d); "
                "truncate the reads to max_bases on the host or reserve more", nbytes, c->st_bases_cap, c->max_B, c->max_T);
  clm_ctx::HostSlot& sl = c->slot[c->next_slot];
  if (sl.busy) return fail(c, CLM_ERR_STATE, "clm_predict_host_submit: %d batches are already in flight; call clm_predict_host_wait", clm_ctx::HOST_SLOTS);
  cudaStream_t st = c->own_stream;
  CLM_CUDA(c, cudaMemcpyAsync(sl.bases, h_bases, nbytes, cudaMemcpyHostToDevice, c->h2d_stream));
  CLM_CUDA(c, cudaMemcpyAsync(sl.offsets, h_offsets, (size_t)(B + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, c->h2d_stream));
  CLM_CUDA(c, cudaEventRecord(sl.h2d_done, c->h2d_stream));
  CLM_CUDA(c, cudaStreamWaitEvent(st, sl.h2d_done, 0));
  int rc = clm_encode_batch(c, sl.bases, sl.offsets, B, T_pad, add_cls, add_sep, pad_left, max_bases, sl.ids, nullptr, st);
  if (rc) return rc;
  rc = clm_forward(c, sl.ids, CLM_U8, B, T_pad, sl.logits, sl.labels, st);
  if (rc) return rc;
  CLM_CUDA(c, cudaEventRecord(sl.fwd_done, st));
  CLM_CUDA(c, cudaStreamWaitEvent(c->d2h_stream, sl.fwd_done, 0));
  CLM_CUDA(c, cudaMemcpyAsync(h_logits, sl.logits, (size_t)B * 2 * sizeof(float), cudaMemcpyDeviceToHost, c->d2h_stream));
  if (h_labels) CLM_CUDA(c, cudaMemcpyAsync(h_labels, sl.labels, (size_t)B, cudaMemcpyDeviceToHost, c->d2h_stream));
  CLM_CUDA(c, cudaEventRecord(sl.done, c->d2h_stream));
  sl.busy = true; sl.seq = c->fwd_seq; sl.B = B; sl.T = T_pad; sl.h_logits = h_logits; sl.h_labels = h_labels;
  *ticket = c->next_slot;
  c->next_slot = (c->next_slot + 1) % clm_ctx::HOST_SLOTS;
  return 0;
}

int clm_predict_host_wait(clm_ctx* c, int ticket) {
  if (!c || ticket < 0 || ticket >= clm_ctx::HOST_SLOTS) return fail(c, CLM_ERR_INVALID, "clm_predict_host_wait: bad ticket");
  clm_ctx::HostSlot& sl = c->slot[ticket];
  if (!sl.busy) return fail(c, CLM_ERR_STATE, "clm_predict_host_wait: ticket %d is not in flight", ticket);
  sl.busy = false;
  CLM_CUDA(c, cudaSetDevice(c->device));
  CLM_CUDA(c, cudaEventSynchronize(sl.done));
  if (c->dbg_layer >= 0) return 0;   // stopped early: no status was published
  int rc = clm_forward_status(c, sl.seq);
  if (rc != CLM_ERR_FP16_RANGE || !c->tc_conv) return rc;
  // automatic switch: this batch left the fp16 range of the tensor-core convolution - redo it with the fp32 FFT kernel
  // (its token ids are still in the slot; later batches already queued on the stream are not disturbed)
  struct Restore {
    clm_ctx* c; bool tc;
    ~Restore() { c->tc_conv = tc; }
  } restore{c, c->tc_conv};
  c->tc_conv = false;
  c->tc_fallbacks++;
  cudaStream_t st = c->own_stream;
  rc = clm_forward(c, sl.ids, CLM_U8, sl.B, sl.T, sl.logits, sl.labels, st);
  if (rc) return rc;
  CLM_CUDA(c, cudaMemcpyAsync(sl.h_logits, sl.logits, (size_t)sl.B * 2 * sizeof(float), cudaMemcpyDeviceToHost, st));
  if (sl.h_labels) CLM_CUDA(c, cudaMemcpyAsync(sl.h_labels, sl.labels, (size_t)sl.B, cudaMemcpyDeviceToHost, st));
  CLM_CUDA(c, cudaStreamSynchronize(st));
  return clm_forward_status(c, c->fwd_seq);
}

int clm_predict_host(clm_ctx* c, const uint8_t* h_bases, const int64_t* h_offsets, int B, int T_pad, int add_cls,
                     int add_sep, int pad_left, int max_bases, float* h_logits, uint8_t* h_labels) {
  int ticket = -1;
  int rc = clm_predict_host_submit(c, h_bases, h_offsets, B, T_pad, add_cls, add_sep, pad_left, max_bases, h_logits, h_labels, &ticket);
  if (rc) return rc;
  return clm_predict_host_wait(c, ticket);
}

int clm_gemm(clm_ctx* c, const void* d_A, const void* d_W, const float* d_bias, int M, int N, int K, int epi,
             void* d_out, const float* d_res, const float* d_w2, float b2, float* d_score, void* stream) {
  if (!c || !d_A || !d_W || !d_bias) return fail(c, CLM_ERR_INVALID, "clm_gemm: bad argument");
  CUtensorMap tmB;
  int rc = make_tmap_bf16_2d(c, &tmB, d_W, (uint64_t)N, (uint64_t)K, epi == EPI_SCORE ? 256 : 128);
  if (rc) return rc;
  GemmParams p{};
  p.M = M; p.N = N; p.K = K; p.bias = d_bias; p.out = d_out; p.res = d_res; p.w2 = d_w2; p.b2 = b2; p.score = d_score; p.ldo = N;
  return launch_gemm(c, d_A, tmB, p, epi, (cudaStream_t)stream);
}

int clm_set_option(clm_ctx* c, const char* name, int value) {
  if (!c || !name) return CLM_ERR_INVALID;
  const std::string n(name);
  if (n == "fused_mlp") c->fused_mlp = value != 0;
  else if (n == "fused_in") c->fused_in = value != 0;
#ifdef CLM_EXPERIMENTS
  else if (n == "fast_conv") c->fast_conv = value != 0;
  else if (n == "in_2cta") c->in_2cta = value != 0;
  else if (n == "mlp_2cta") c->mlp_2cta = value != 0;
  else if (n == "mlp_epi16") c->mlp_epi16 = value != 0;
  else if (n == "mlp_pp") c->mlp_pp = value != 0;
#else
  else if (n == "fast_conv" || n == "in_2cta" || n == "mlp_2cta" || n == "mlp_epi16" || n == "mlp_pp")
    return fail(c, CLM_ERR_INVALID, "clm_set_option: '%s' selects an experiment kernel that is not compiled in (build with -DCLM_EXPERIMENTS)", name);
#endif
  else if (n == "tc_conv") c->tc_conv = value != 0;
  else if (n == "tc_chunked") c->tc_chunked = value != 0;
  else if (n == "tc_pipe") c->tc_pipe = value != 0;
  else if (n == "tc_pack4") c->tc_pack4 = value != 0;
  else if (n == "tc_helpers_low") c->tc_helpers_low = value;
  else if (n == "tc_pipe_chunked") c->tc_pipe_chunked = value != 0;
  else if (n == "fused_score_pool") c->fused_score_pool = value != 0;
  else if (n == "fused_head") c->fused_head = value != 0;
  else if (n == "head_coop") c->head_coop = value != 0;
  else if (n == "mlp_stagger") c->mlp_stagger = value;
  else if (n == "y_channel_major") c->y_channel_major = value != 0;
  else if (n == "mlp_grid") c->mlp_grid = value;
  else if (n == "skip_dead_res") c->skip_dead_res = value != 0;

  else if (n == "tc_scale_shift") {   // test hook: move the calibrated input scale of the tensor-core conv by 2^value
    if (!c->finalized) return fail(c, CLM_ERR_STATE, "clm_set_option(tc_scale_shift) before clm_finalize");
    CLM_CUDA(c, cudaDeviceSynchronize());
    for (auto& L : c->layers)
      if (L.gexp)
        tc::scales_kernel<<<(c->cfg.d_model + 255) / 256, 256>>>(L.gexp, L.vx_amax, L.vx_scale, L.tc_osc, L.tc_inva, L.tc_rel,
                                                                 c->cfg.d_model, c->tc_nseg, value);
    CLM_CUDA(c, cudaDeviceSynchronize());
  }
  else if (n == "mlp_fc2_lag") c->mlp_fc2_lag = value;
  else if (n == "mlp_early_res") c->mlp_early_res = value;
  else if (n == "mlp_helpers_high") c->mlp_helpers_high = value;
  else if (n == "mlp_store_a") c->mlp_store_a = value;
  else if (n == "embed_in") c->embed_in = value != 0;
  else if (n == "pdl") c->pdl = value != 0;
  else if (n == "embed_res") c->embed_res = value != 0;
  else if (n == "mlp_gather_tails") c->mlp_gather_tails = value != 0;
  else if (n == "in_prefetch") c->in_prefetch = value;
  else if (n == "in_ext_tail") c->in_ext_tail = value != 0;
  else return fail(c, CLM_ERR_INVALID, "clm_set_option: unknown option '%s'", name);
  return 0;
}

// d_res (R32) is first normalised into the context's XN workspace (needs clm_reserve >= B x T)
int normalize_for_block_in(clm_ctx* c, const float* d_res, int B, int T, cudaStream_t st) {
  if ((long long)B * T > c->max_tokens) return fail(c, CLM_ERR_STATE, "clm_block_in: call clm_reserve(B, T) first");
  const long long M = (long long)B * T;
  layernorm_bf16_kernel<<<(unsigned)((M + 31) / 32), 256, 0, st>>>(d_res, c->ones, c->zeros, c->XN, M, c->cfg.layer_norm_eps);
  CLM_LAUNCH_CHECK(c, "normalize");
  return 0;
}

int clm_block_in(clm_ctx* c, int layer, const float* d_res, int B, int T, int Tp, void* d_vx, void* d_x0, void* stream) {
  if (!c || !c->finalized) return fail(c, CLM_ERR_STATE, "clm_block_in before clm_finalize");
  if (layer < 0 || layer >= c->cfg.n_layer || !d_res || !d_vx || !d_x0 || B <= 0 || T <= 0 || Tp < T || Tp % 64 != 0)
    return fail(c, CLM_ERR_INVALID, "clm_block_in: bad argument");
  int rc = normalize_for_block_in(c, d_res, B, T, (cudaStream_t)stream);
  if (rc) return rc;
  return launch_block_in(c, layer, c->XN, B, T, Tp, (__nv_bfloat16*)d_vx, (__nv_bfloat16*)d_x0, (cudaStream_t)stream);
}

int clm_block_in_trace(clm_ctx* c, int layer, const float* d_res, int B, int T, int Tp, void* d_vx, void* d_x0,
                       long long* d_trace, void* stream) {
  if (!c || !c->finalized) return fail(c, CLM_ERR_STATE, "clm_block_in_trace before clm_finalize");
  if (layer < 0 || layer >= c->cfg.n_layer || !d_res || !d_vx || !d_x0 || !d_trace || B <= 0 || T <= 0 || Tp < T || Tp % 64 != 0)
    return fail(c, CLM_ERR_INVALID, "clm_block_in_trace: bad argument");
  int rc = normalize_for_block_in(c, d_res, B, T, (cudaStream_t)stream);
  if (rc) return rc;
  return launch_block_in(c, layer, c->XN, B, T, Tp, (__nv_bfloat16*)d_vx, (__nv_bfloat16*)d_x0, (cudaStream_t)stream, d_trace);
}

int clm_block_mlp(clm_ctx* c, int layer, const void* d_y, float* d_res, int M, void* stream) {
  if (!c || !c->finalized) return fail(c, CLM_ERR_STATE, "clm_block_mlp before clm_finalize");
  if (layer < 0 || layer >= c->cfg.n_layer || !d_y || !d_res || M <= 0) return fail(c, CLM_ERR_INVALID, "clm_block_mlp: bad argument");
  return launch_block_mlp(c, layer, (const __nv_bfloat16*)d_y, d_res, M, (cudaStream_t)stream);
}

int clm_block_mlp_cm(clm_ctx* c, int layer, const void* d_y_cm, float* d_res, int B, int T, int Tp, void* stream) {
  if (!c || !c->finalized) return fail(c, CLM_ERR_STATE, "clm_block_mlp_cm before clm_finalize");
  if (layer < 0 || layer >= c->cfg.n_layer || !d_y_cm || !d_res || B <= 0 || T <= 0 || Tp < T || Tp % 64 != 0)
    return fail(c, CLM_ERR_INVALID, "clm_block_mlp_cm: bad argument");
  return launch_block_mlp(c, layer, (const __nv_bfloat16*)d_y_cm, d_res, B * T, (cudaStream_t)stream, nullptr, B, T, Tp);
}

int clm_block_mlp_cm_trace(clm_ctx* c, int layer, const void* d_y_cm, float* d_res, int B, int T, int Tp, int write_xn,
                           long long* d_trace, void* stream) {
  if (!c || !c->finalized) return fail(c, CLM_ERR_STATE, "clm_block_mlp_cm_trace before clm_finalize");
  if (layer < 0 || layer >= c->cfg.n_layer || !d_y_cm || !d_res || B <= 0 || T <= 0 || Tp < T || Tp % 64 != 0)
    return fail(c, CLM_ERR_INVALID, "clm_block_mlp_cm_trace: bad argument");
  if (write_xn && (long long)B * T > c->max_tokens) return fail(c, CLM_ERR_STATE, "clm_block_mlp_cm_trace: call clm_reserve(B, T) first");
  return launch_block_mlp(c, layer, (const __nv_bfloat16*)d_y_cm, d_res, B * T, (cudaStream_t)stream, d_trace, B, T, Tp,
                          write_xn ? c->XN : nullptr);
}

int clm_block_mlp_trace(clm_ctx* c, int layer, const void* d_y, float* d_res, int M, long long* d_trace, void* stream) {
  if (!c || !c->finalized) return fail(c, CLM_ERR_STATE, "clm_block_mlp_trace before clm_finalize");
  if (layer < 0 || layer >= c->cfg.n_layer || !d_y || !d_res || M <= 0 || !d_trace) return fail(c, CLM_ERR_INVALID, "clm_block_mlp_trace: bad argument");
  return launch_block_mlp(c, layer, (const __nv_bfloat16*)d_y, d_res, M, (cudaStream_t)stream, d_trace);
}

int clm_longconv(clm_ctx* c, int layer, const void* d_vx, const void* d_x0, void* d_out, int B, int T, int Tp,
                 void* stream) {
  if (!c || !c->finalized) return fail(c, CLM_ERR_STATE, "clm_longconv before clm_finalize");
  if (layer < 0 || layer >= c->cfg.n_layer || B <= 0 || T <= 0 || Tp < T || Tp % 64 != 0) return fail(c, CLM_ERR_INVALID, "clm_longconv: bad argument (Tp must be a multiple of 64 and >= T)");
  const size_t needb = conv_scratch_bytes(c, T);
  if (needb > c->scratch_bytes) {
    CLM_CUDA(c, cudaDeviceSynchronize());
    dev_release(c, &c->scratch);
    c->scratch_bytes = 0;
    int rc = dev_alloc(c, reinterpret_cast<uint8_t**>(&c->scratch), needb);
    if (rc) return rc;
    c->scratch_bytes = needb;
  }
  return launch_longconv(c, layer, (const __nv_bfloat16*)d_vx, (const __nv_bfloat16*)d_x0, (__nv_bfloat16*)d_out, B, T, Tp,
                         c->scratch, c->scratch_bytes, (cudaStream_t)stream);
}

int ensure_tc_scratch(clm_ctx* c, int T) {
  const size_t need = tc_scratch_per_cta(tc_plan(T).nc) * c->num_sms;
  if (need <= c->tc_scratch_floats) return 0;
  CLM_CUDA(c, cudaDeviceSynchronize());
  dev_release(c, &c->tc_scratch);
  c->tc_scratch_floats = 0;
  int rc = dev_alloc(c, &c->tc_scratch, need);
  if (rc) return rc;
  c->tc_scratch_floats = need;
  return 0;
}

int clm_longconv_tc_trace(clm_ctx* c, int layer, const void* d_vx_f16, const void* d_x0, void* d_out, int B, int T, int Tp,
                          long long* d_trace, void* stream) {
  if (!c || !c->finalized) return fail(c, CLM_ERR_STATE, "clm_longconv_tc_trace before clm_finalize");
  if (layer < 0 || layer >= c->cfg.n_layer || !d_vx_f16 || !d_x0 || !d_out || !d_trace || B <= 0 || Tp < T || Tp % 64 != 0)
    return fail(c, CLM_ERR_INVALID, "clm_longconv_tc_trace: bad argument");
  if (int rc = ensure_tc_scratch(c, T)) return rc;
  return launch_longconv_tc(c, layer, (const __half*)d_vx_f16, (const __nv_bfloat16*)d_x0, (__nv_bfloat16*)d_out, B, T, Tp,
                            (cudaStream_t)stream, d_trace, /*unit_scale=*/true);
}

int clm_longconv_tc(clm_ctx* c, int layer, const void* d_vx_f16, const void* d_x0, void* d_out, int B, int T, int Tp,
                    void* stream) {
  if (!c || !c->finalized) return fail(c, CLM_ERR_STATE, "clm_longconv_tc before clm_finalize");
  if (layer < 0 || layer >= c->cfg.n_layer || !d_vx_f16 || !d_x0 || !d_out || B <= 0 || Tp < T || Tp % 64 != 0)
    return fail(c, CLM_ERR_INVALID, "clm_longconv_tc: bad argument");
  if (int rc = ensure_tc_scratch(c, T)) return rc;
  return launch_longconv_tc(c, layer, (const __half*)d_vx_f16, (const __nv_bfloat16*)d_x0, (__nv_bfloat16*)d_out, B, T, Tp,
                            (cudaStream_t)stream, nullptr, /*unit_scale=*/true);
}

int clm_longconv_tc_auto(clm_ctx* c, int layer, const void* d_vx_bf16, const void* d_x0, void* d_out, int B, int T, int Tp,
                         void* stream) {
  if (!c || !c->finalized) return fail(c, CLM_ERR_STATE, "clm_longconv_tc_auto before clm_finalize");
  if (layer < 0 || layer >= c->cfg.n_layer || !d_vx_bf16 || !d_x0 || !d_out || B <= 0 || Tp < T || Tp % 64 != 0)
    return fail(c, CLM_ERR_INVALID, "clm_longconv_tc_auto: bad argument");
  if (int rc = ensure_tc_scratch(c, T)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  LayerW& L = c->layers[layer];
  const int D = c->cfg.d_model;
  __half* vxh = nullptr;
  unsigned int* amax = nullptr;
  float* f = nullptr;   // scale | osc | inva | rel
  int rc = dev_alloc(c, &vxh, (size_t)B * D * Tp);
  if (!rc) rc = dev_alloc(c, &amax, (size_t)D);
  if (!rc) rc = dev_alloc(c, &f, (size_t)D * (3 + c->tc_nseg));
  if (!rc) {
    cudaMemsetAsync(amax, 0, D * sizeof(unsigned int), st);
    cudaMemsetAsync(c->d_err + 1, 0, sizeof(int), st);
    tc::amax_cm_kernel<<<dim3(D, B), 256, 0, st>>>((const __nv_bfloat16*)d_vx_bf16, D, Tp, T, amax);
    tc::scales_kernel<<<(D + 255) / 256, 256, 0, st>>>(L.gexp, amax, f, f + D, f + 2 * D, f + 3 * D, D, c->tc_nseg, 0);
    tc::scale_to_f16_kernel<<<dim3(D, B), 256, 0, st>>>((const __nv_bfloat16*)d_vx_bf16, vxh, f, D, Tp, T);
    rc = launch_longconv_tc(c, layer, vxh, (const __nv_bfloat16*)d_x0, (__nv_bfloat16*)d_out, B, T, Tp, st, nullptr, false, f + D, f + 2 * D);
  }
  int flags = 0;
  if (!rc) {
    cudaError_t e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaMemcpy(&flags, c->d_err + 1, sizeof(int), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) rc = fail(c, CLM_ERR_CUDA, "clm_longconv_tc_auto: %s", cudaGetErrorString(e));
  }
  dev_free(c, vxh); dev_free(c, amax); dev_free(c, f);
  if (!rc && (flags & 2)) return fail(c, CLM_ERR_FP16_RANGE, "clm_longconv_tc_auto: non-finite output (fp16 range exceeded)");
  return rc;
}

long long clm_tc_fallback_count(const clm_ctx* c) { return c ? c->tc_fallbacks : 0; }

int clm_longconv_variant(const clm_ctx* c, int T) {
  if (!c || !c->finalized || T <= 0) return -1;
  if (c->fused_in && tc_conv_applies(c, T)) return 2;
  const ConvPlan pl = plan_conv(T);
  return (c->fast_conv && c->layers[0].gspecT[pl.logn] != nullptr) ? 1 : 0;
}

int clm_attention_weights(clm_ctx* c, float* d_out, int B, int T, void* stream) {
  if (!c || !c->finalized) return fail(c, CLM_ERR_STATE, "clm_attention_weights before clm_finalize");
  if (!d_out || B <= 0 || T <= 0) return fail(c, CLM_ERR_INVALID, "clm_attention_weights: bad argument");
  if (B != c->last_B || T != c->last_T) return fail(c, CLM_ERR_STATE, "clm_attention_weights: the last forward was %d x %d, not %d x %d", c->last_B, c->last_T, B, T);
  attention_softmax_kernel<<<B, 256, 0, (cudaStream_t)stream>>>(c->score, d_out, T);
  CLM_LAUNCH_CHECK(c, "attention_softmax");
  return 0;
}

int clm_get_filter(clm_ctx* c, int layer, float* d_out, int L, void* stream) {
  if (!c || !c->finalized) return fail(c, CLM_ERR_STATE, "clm_get_filter before clm_finalize");
  if (layer < 0 || layer >= c->cfg.n_layer || L <= 0 || L > c->cfg.max_seq_len) return fail(c, CLM_ERR_INVALID, "clm_get_filter: bad argument");
  CLM_CUDA(c, cudaMemcpy2DAsync(d_out, (size_t)L * sizeof(float), c->layers[layer].k, (size_t)c->Lk * sizeof(float),
                                (size_t)L * sizeof(float), c->cfg.d_model, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}

int clm_profile_enable(clm_ctx* c, int on) {
  if (!c) return CLM_ERR_INVALID;
  if (!on && c->prof_on) prof_collect(c);
  c->prof_on = on != 0;
  return 0;
}

int clm_profile_reset(clm_ctx* c) {
  if (!c) return CLM_ERR_INVALID;
  prof_collect(c);
  for (int i = 0; i < 32; ++i) { c->prof_ms[i] = 0; c->prof_n[i] = 0; }
  return 0;
}

int clm_profile_num(void) { return PC_COUNT; }

const char* clm_profile_name(int cat) { return (cat >= 0 && cat < PC_COUNT) ? kProfNames[cat] : ""; }

int clm_profile_get(clm_ctx* c, int cat, double* total_ms, long long* launches) {
  if (!c || cat < 0 || cat >= PC_COUNT || !total_ms || !launches) return fail(c, CLM_ERR_INVALID, "clm_profile_get: bad argument");
  prof_collect(c);
  *total_ms = c->prof_ms[cat];
  *launches = c->prof_n[cat];
  return 0;
}

int clm_debug_copy(clm_ctx* c, const char* what, void* d_dst, size_t max_bytes, void* stream) {
  if (!c || !what || !d_dst) return fail(c, CLM_ERR_INVALID, "clm_debug_copy: bad argument");
  const size_t M = (size_t)c->max_tokens, D = c->cfg.d_model;
  const size_t CT = c->ct_elems;
  const void* src = nullptr;
  size_t bytes = 0;
  const std::string w(what);
  if (w == "resid") { src = c->R; bytes = (M + 128) * D * 4; }  // R32 blocked layout
  else if (w == "xn") { src = c->XN; bytes = M * D * 2; }
  else if (w == "u") { src = c->U; bytes = M * c->cfg.d_inner * 2; }
  else if (w == "vx") { src = c->VX; bytes = CT * 2; }
  else if (w == "x0") { src = c->X0; bytes = CT * 2; }
  else if (w == "y") { src = c->Y; bytes = CT * 2; }
  else if (w == "yt") { src = c->YT; bytes = M * D * 2; }
  else if (w == "score") { src = c->score; bytes = M * 4; }
  else if (w == "pooled") { src = c->pooled; bytes = (size_t)c->max_B * D * 4; }
  else return fail(c, CLM_ERR_INVALID, "clm_debug_copy: unknown buffer '%s'", what);
  if (!src) return fail(c, CLM_ERR_STATE, "clm_debug_copy: workspaces not reserved");
  CLM_CUDA(c, cudaMemcpyAsync(d_dst, src, std::min(bytes, max_bytes), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}

}  // extern "C"

// =============================================================================================
// Head fine-tuning (include/chimeralm_b200.h, "Fine-tuning of the head"; csrc/head_train.cuh for the kernels)
namespace {

// The head tensors in the order of the flat master / gradient / AdamW buffers (offsets rounded up to 64 floats).
struct HeadTensorInfo { const char* name; long long numel; };
constexpr HeadTensorInfo kHeadTensors[] = {
    {"attention.0.weight", 256 * 256}, {"attention.0.bias", 256}, {"attention.2.weight", 256}, {"attention.2.bias", 1},
    {"classifier.0.weight", 512 * 256}, {"classifier.0.bias", 512}, {"classifier.3.weight", 512 * 512},
    {"classifier.3.bias", 512}, {"classifier.6.layers.0.weight", 512 * 512}, {"classifier.6.layers.0.bias", 512},
    {"classifier.6.layers.3.weight", 512 * 512}, {"classifier.6.layers.3.bias", 512}, {"output_layer.weight", 2 * 512},
    {"output_layer.bias", 2}};
constexpr int kNumHeadTensors = (int)(sizeof(kHeadTensors) / sizeof(kHeadTensors[0]));
enum { HT_A0W, HT_A0B, HT_A2W, HT_A2B, HT_C0W, HT_C0B, HT_C3W, HT_C3B, HT_R0W, HT_R0B, HT_R3W, HT_R3B, HT_OW, HT_OB };

long long head_offset(int i) {
  long long off = 0;
  for (int k = 0; k < i; ++k) off += (kHeadTensors[k].numel + 63) / 64 * 64;
  return off;
}

int head_index(const char* name) {
  std::string n(name ? name : "");
  if (n.rfind("net.", 0) != 0) n = "net." + n;
  for (int i = 0; i < kNumHeadTensors; ++i)
    if (n == std::string("net.head.") + kHeadTensors[i].name) return i;
  return -1;
}

// the tensor the forward reads (as loaded by clm_load_tensor)
float* head_live(clm_ctx* c, int i) {
  auto it = c->w.find(std::string("net.head.") + kHeadTensors[i].name);
  return it == c->w.end() ? nullptr : it->second.d;
}

}  // namespace

int clm_head_train_begin(clm_ctx* c, const clm_head_train_cfg* cfg) {
  if (!c || !cfg) return fail(c, CLM_ERR_INVALID, "clm_head_train_begin: bad argument");
  if (c->cfg.pooling != 0)
    return fail(c, CLM_ERR_INVALID, "clm_head_train_begin: only attention pooling can be trained (pooling = %d); ChimeraLM's head "
                "uses attention pooling (chimeralm/models/lm.py:46-55)", c->cfg.pooling);
  if (!c->finalized) return fail(c, CLM_ERR_STATE, "clm_head_train_begin before clm_finalize");
  if (c->max_B <= 0) return fail(c, CLM_ERR_STATE, "clm_head_train_begin before clm_reserve");
  if (c->ht.on) return fail(c, CLM_ERR_STATE, "clm_head_train_begin: training state already exists on this context");
  if (!(cfg->dropout >= 0.0 && cfg->dropout < 1.0) || !(cfg->lr >= 0.f) || !(cfg->eps > 0.f) || !(cfg->beta1 >= 0.f && cfg->beta1 < 1.f) ||
      !(cfg->beta2 >= 0.f && cfg->beta2 < 1.f) || !(cfg->weight_decay >= 0.f))
    return fail(c, CLM_ERR_INVALID, "clm_head_train_begin: lr >= 0, 0 <= betas < 1, eps > 0, weight_decay >= 0, 0 <= dropout < 1");
  for (int i = 0; i < kNumHeadTensors; ++i)
    if (!head_live(c, i)) return fail(c, CLM_ERR_MISSING, "clm_head_train_begin: weight 'net.head.%s' was not loaded", kHeadTensors[i].name);
  CLM_CUDA(c, cudaSetDevice(c->device));
  clm_ctx::HeadTrain& h = c->ht;
  const int B = c->max_B, H = c->cfg.head_hidden, D = c->cfg.d_model;
  h.n = head_offset(kNumHeadTensors);
  int rc;
  for (float** p : {&h.param, &h.grad, &h.m, &h.v})
    if ((rc = dev_alloc(c, p, (size_t)h.n))) return rc;
  if ((rc = dev_alloc(c, &h.step, 1))) return rc;
  for (float** p : {&h.z0, &h.z1, &h.z2, &h.x1, &h.x2, &h.x3, &h.x4, &h.dA, &h.dB, &h.dC})
    if ((rc = dev_alloc(c, p, (size_t)B * H))) return rc;
  for (float** p : {&h.logits, &h.dlogits, &h.fwd_logits})
    if ((rc = dev_alloc(c, p, (size_t)B * 2))) return rc;
  if ((rc = dev_alloc(c, &h.dpooled, (size_t)B * D))) return rc;
  if ((rc = dev_alloc(c, &h.rd, (size_t)B * 4))) return rc;
  if ((rc = dev_alloc(c, &h.gdp, (size_t)B * D))) return rc;
  h.n_cta = std::max(2, c->num_sms / 2 * 2);
  if ((rc = dev_alloc(c, &h.part_dw, (size_t)h.n_cta * 128 * 256))) return rc;
  if ((rc = dev_alloc(c, &h.part_vec, (size_t)h.n_cta * 3 * 128))) return rc;
  CLM_CUDA(c, cudaMemset(h.param, 0, (size_t)h.n * sizeof(float)));
  CLM_CUDA(c, cudaMemset(h.grad, 0, (size_t)h.n * sizeof(float)));
  CLM_CUDA(c, cudaMemset(h.m, 0, (size_t)h.n * sizeof(float)));
  CLM_CUDA(c, cudaMemset(h.v, 0, (size_t)h.n * sizeof(float)));
  CLM_CUDA(c, cudaMemset(h.step, 0, sizeof(int)));
  for (int i = 0; i < kNumHeadTensors; ++i)
    CLM_CUDA(c, cudaMemcpy(h.param + head_offset(i), head_live(c, i), (size_t)kHeadTensors[i].numel * sizeof(float), cudaMemcpyDeviceToDevice));
  CLM_CUDA(c, cudaDeviceSynchronize());
  h.cfg = *cfg;
  h.max_B = B;
  h.thr = (uint32_t)std::floor(cfg->dropout * 16777216.0 + 0.5);
  h.scale = (float)(1.0 / (1.0 - cfg->dropout));
  h.calls = 0;
  h.on = true;
  return 0;
}

int clm_head_train_step(clm_ctx* c, const void* d_ids, int ids_dtype, int B, int T, const int64_t* d_targets,
                        float* d_loss_out, void* stream) {
  if (!c) return CLM_ERR_INVALID;
  clm_ctx::HeadTrain& h = c->ht;
  if (!h.on) return fail(c, CLM_ERR_STATE, "clm_head_train_step before clm_head_train_begin");
  if (!d_ids || !d_targets || B <= 0 || T <= 0) return fail(c, CLM_ERR_INVALID, "clm_head_train_step: bad argument");
  if (B > h.max_B) return fail(c, CLM_ERR_STATE, "clm_head_train_step: batch of %d reads exceeds the %d sized by clm_head_train_begin", B, h.max_B);
  // the backward reads what the folded tail leaves behind: XN from the last block, the per-tile softmax partials of
  // score_pool_kernel and pooled from head_fused_kernel
  if (!c->fused_mlp || !c->fused_score_pool || !c->fused_head || c->dbg_layer >= 0)
    return fail(c, CLM_ERR_STATE, "clm_head_train_step needs the fused forward (options fused_mlp, fused_score_pool, fused_head on, no debug stop)");
  cudaStream_t st = (cudaStream_t)stream;
  int rc = clm_forward(c, d_ids, ids_dtype, B, T, h.fwd_logits, nullptr, st);
  if (rc) return rc;
  const int* status = c->d_status_map + (c->fwd_seq & 7);
  ProfScope ps_(c, PC_HEAD_TRAIN, st);   // everything after the forward: classifier again, backward, AdamW, refresh
  const int H = c->cfg.head_hidden, D = c->cfg.d_model;
  const HeadParams& hp = c->head;
  const DropoutCfg dc{h.cfg.seed, (uint32_t)h.calls, h.thr, h.scale};
  const unsigned bt = (unsigned)((B + 31) / 32), bx = (unsigned)((B + HT_RB - 1) / HT_RB);
  float* G[kNumHeadTensors];
  for (int i = 0; i < kNumHeadTensors; ++i) G[i] = h.grad + head_offset(i);
  // ---- classifier forward with dropout (classifier.2, classifier.5, classifier.6.layers.2)
  ht_fwd_kernel<256, 0><<<dim3(H / 8, bt), 256, 0, st>>>(hp.w0, hp.b0, c->pooled, nullptr, h.z0, h.x1, B, H, dc, 0);
  CLM_LAUNCH_CHECK(c, "ht_fwd");
  ht_fwd_kernel<512, 0><<<dim3(H / 8, bt), 256, 0, st>>>(hp.w1, hp.b1, h.x1, nullptr, h.z1, h.x2, B, H, dc, 1);
  CLM_LAUNCH_CHECK(c, "ht_fwd");
  ht_fwd_kernel<512, 0><<<dim3(H / 8, bt), 256, 0, st>>>(hp.wr0, hp.br0, h.x2, nullptr, h.z2, h.x3, B, H, dc, 2);
  CLM_LAUNCH_CHECK(c, "ht_fwd");
  ht_fwd_kernel<512, 1><<<dim3(H / 8, bt), 256, 0, st>>>(hp.wr1, hp.br1, h.x3, h.x2, nullptr, h.x4, B, H, dc, 0);
  CLM_LAUNCH_CHECK(c, "ht_fwd");
  ht_fwd_kernel<512, 2><<<dim3(1, bt), 256, 0, st>>>(hp.wo, hp.bo, h.x4, nullptr, nullptr, h.logits, B, 2, dc, 0);
  CLM_LAUNCH_CHECK(c, "ht_fwd");
  ht_loss_kernel<<<1, 256, 0, st>>>(h.logits, d_targets, h.dlogits, d_loss_out, B);
  CLM_LAUNCH_CHECK(c, "ht_loss");
  // ---- classifier backward: output_layer, ResidualBlock, classifier.3, classifier.0 -> dpooled
  ht_bwd_w_kernel<<<dim3(2, 2), 256, 0, st>>>(h.dlogits, h.x4, G[HT_OW], G[HT_OB], B, 2, H);
  CLM_LAUNCH_CHECK(c, "ht_bwd_w");
  ht_bwd_x_kernel<<<dim3(H / 256, bx), 256, 0, st>>>(hp.wo, h.dlogits, nullptr, nullptr, h.dA, B, 2, H, dc, 0);          // dx4
  CLM_LAUNCH_CHECK(c, "ht_bwd_x");
  ht_bwd_w_kernel<<<dim3(H / 256, H), 256, 0, st>>>(h.dA, h.x3, G[HT_R3W], G[HT_R3B], B, H, H);
  CLM_LAUNCH_CHECK(c, "ht_bwd_w");
  ht_bwd_x_kernel<<<dim3(H / 256, bx), 256, 0, st>>>(hp.wr1, h.dA, nullptr, h.z2, h.dB, B, H, H, dc, 2);                // dz2
  CLM_LAUNCH_CHECK(c, "ht_bwd_x");
  ht_bwd_w_kernel<<<dim3(H / 256, H), 256, 0, st>>>(h.dB, h.x2, G[HT_R0W], G[HT_R0B], B, H, H);
  CLM_LAUNCH_CHECK(c, "ht_bwd_w");
  ht_bwd_x_kernel<<<dim3(H / 256, bx), 256, 0, st>>>(hp.wr0, h.dB, h.dA, h.z1, h.dC, B, H, H, dc, 1);                   // dz1 (+ skip)
  CLM_LAUNCH_CHECK(c, "ht_bwd_x");
  ht_bwd_w_kernel<<<dim3(H / 256, H), 256, 0, st>>>(h.dC, h.x1, G[HT_C3W], G[HT_C3B], B, H, H);
  CLM_LAUNCH_CHECK(c, "ht_bwd_w");
  ht_bwd_x_kernel<<<dim3(H / 256, bx), 256, 0, st>>>(hp.w1, h.dC, nullptr, h.z0, h.dA, B, H, H, dc, 0);                 // dz0
  CLM_LAUNCH_CHECK(c, "ht_bwd_x");
  ht_bwd_w_kernel<<<dim3(D / 256, H), 256, 0, st>>>(h.dA, c->pooled, G[HT_C0W], G[HT_C0B], B, H, D);
  CLM_LAUNCH_CHECK(c, "ht_bwd_w");
  ht_bwd_x_kernel<<<dim3(D / 256, bx), 256, 0, st>>>(hp.w0, h.dA, nullptr, nullptr, h.dpooled, B, H, D, dc, 0);         // dpooled
  CLM_LAUNCH_CHECK(c, "ht_bwd_x");
  // ---- pooling + scorer backward
  const int tiles_per_seq = (T + sb::BM - 1) / sb::BM;
  ht_pool_prep_kernel<<<B, 256, 0, st>>>(c->part, tiles_per_seq, c->pooled, h.dpooled, c->lnf_g, c->lnf_b, h.rd, h.gdp);
  CLM_LAUNCH_CHECK(c, "ht_pool_prep");
  {
    if (int rc_attr = ensure_smem_attr(c, (const void*)(score_bwd_kernel), (int)(sb::SMEM_TOTAL))) return rc_attr;
    CUtensorMap tmX, tmW;
    if ((rc = make_tmap_xn(c, &tmX, c->XN, B, T, sb::BM))) return rc;
    if ((rc = make_tmap_bf16_2d(c, &tmW, c->att0_wf, D, D, sb::HALF))) return rc;   // the forward's folded weights, half a box
    ScoreBwdParams sp{};
    sp.b0f = c->att0_bf; sp.w2 = c->att2_w; sp.score = c->score; sp.rd = h.rd; sp.gdp = h.gdp;
    sp.part_dw = h.part_dw; sp.part_vec = h.part_vec;
    sp.B = B; sp.T = T; sp.tiles_per_seq = tiles_per_seq; sp.num_tiles = B * tiles_per_seq;
    const int grid = 2 * std::min(sp.num_tiles, h.n_cta / 2);
    score_bwd_kernel<<<grid, sb::THREADS, sb::SMEM_TOTAL, st>>>(tmX, tmW, sp);
    CLM_LAUNCH_CHECK(c, "score_bwd");
    score_bwd_reduce_kernel<<<D, 256, 0, st>>>(h.part_dw, h.part_vec, grid, c->lnf_g, c->lnf_b, G[HT_A0W], G[HT_A0B], G[HT_A2W], G[HT_A2B]);
    CLM_LAUNCH_CHECK(c, "score_bwd_reduce");
  }
  // ---- AdamW on the master copies, then refresh what the forward reads
  AdamWParams ap{};
  ap.p = h.param; ap.m = h.m; ap.v = h.v; ap.g = h.grad; ap.n = h.n;
  ap.lr = h.cfg.lr; ap.beta1 = h.cfg.beta1; ap.beta2 = h.cfg.beta2; ap.eps = h.cfg.eps; ap.wd = h.cfg.weight_decay;
  ap.step = h.step; ap.status = status;
  adamw_kernel<<<(unsigned)std::min<long long>((h.n + 255) / 256, 4LL * c->num_sms), 256, 0, st>>>(ap);
  CLM_LAUNCH_CHECK(c, "adamw");
  adamw_step_kernel<<<1, 1, 0, st>>>(h.step, status);
  CLM_LAUNCH_CHECK(c, "adamw_step");
  for (int i = 0; i < kNumHeadTensors; ++i)
    CLM_CUDA(c, cudaMemcpyAsync(head_live(c, i), h.param + head_offset(i), (size_t)kHeadTensors[i].numel * sizeof(float),
                                cudaMemcpyDeviceToDevice, st));
  if ((rc = refresh_scorer(c, st))) return rc;
  ++h.calls;
  return 0;
}

int clm_head_grad_copy(clm_ctx* c, const char* name, float* d_dst, void* stream) {
  if (!c || !name || !d_dst) return fail(c, CLM_ERR_INVALID, "clm_head_grad_copy: bad argument");
  if (!c->ht.on) return fail(c, CLM_ERR_STATE, "clm_head_grad_copy before clm_head_train_begin");
  const int i = head_index(name);
  if (i < 0) return fail(c, CLM_ERR_INVALID, "clm_head_grad_copy: '%s' is not a trainable head tensor", name);
  CLM_CUDA(c, cudaMemcpyAsync(d_dst, c->ht.grad + head_offset(i), (size_t)kHeadTensors[i].numel * sizeof(float),
                              cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}

int clm_head_export(clm_ctx* c, const char* name, float* h_dst) {
  if (!c || !name || !h_dst) return fail(c, CLM_ERR_INVALID, "clm_head_export: bad argument");
  if (!c->finalized) return fail(c, CLM_ERR_STATE, "clm_head_export before clm_finalize");
  const int i = head_index(name);
  if (i < 0) return fail(c, CLM_ERR_INVALID, "clm_head_export: '%s' is not a head tensor", name);
  CLM_CUDA(c, cudaSetDevice(c->device));
  CLM_CUDA(c, cudaDeviceSynchronize());
  const float* src = c->ht.on ? c->ht.param + head_offset(i) : head_live(c, i);
  if (!src) return fail(c, CLM_ERR_MISSING, "clm_head_export: weight '%s' was not loaded", name);
  CLM_CUDA(c, cudaMemcpy(h_dst, src, (size_t)kHeadTensors[i].numel * sizeof(float), cudaMemcpyDeviceToHost));
  if (c->ht.on)
    CLM_CUDA(c, cudaMemcpy(&c->att2_b, c->ht.param + head_offset(HT_A2B), sizeof(float), cudaMemcpyDeviceToHost));
  return 0;
}
