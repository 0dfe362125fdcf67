/* chimeralm_b200 — C ABI of the B200-native `chimeralm predict` hot path.
 *
 * Plain C, no torch types: pointers, sizes and an opaque context.  One context per device;
 * calls on a context are serialised by the caller and are asynchronous on the given CUDA
 * stream unless stated otherwise.  Every function returns 0 on success or a negative
 * clm_status; clm_last_error() gives the message.  No C++ exception crosses this boundary and
 * the library never calls exit().
 *
 * Each entry point names the reference interface it replaces (paths relative to the
 * ylab-hi/ChimeraLM tree).  INTEGRATION.md shows the ctypes binding a maintainer would add.
 */
#ifndef CHIMERALM_B200_H_
#define CHIMERALM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct clm_ctx clm_ctx;

typedef enum {
  CLM_OK = 0,
  CLM_ERR_INVALID = -1,   /* bad argument / shape */
  CLM_ERR_CUDA = -2,      /* CUDA runtime or driver error (message has the detail) */
  CLM_ERR_STATE = -3,     /* call order violated (e.g. forward before finalize) */
  CLM_ERR_MISSING = -4,   /* a required weight tensor was never loaded */
  CLM_ERR_NOMEM = -5,
  CLM_ERR_TOKEN_RANGE = -6, /* a token id outside [0, vocab_rows): the reference's nn.Embedding raises IndexError */
  CLM_ERR_FP16_RANGE = -7   /* the fp16 tensor-core convolution left its range for this batch (see clm_forward_status) */
} clm_status;

typedef enum { CLM_F32 = 0, CLM_BF16 = 1, CLM_U8 = 2, CLM_I32 = 3, CLM_I64 = 4 } clm_dtype;

/* Architecture constants; defaults = LongSafari/hyenadna-small-32k-seqlen-hf config.json +
 * chimeralm/models/lm.py:46-55 (head).  clm_default_config() fills them in. */
typedef struct {
  int d_model, n_layer, d_inner, vocab_rows, max_seq_len;
  int filter_order, emb_dim, short_filter_order, num_inner_mlps;
  int head_hidden, num_classes;
  float layer_norm_eps, filter_shift;
  /* pooling of the head (BinarySequenceClassifier.pooling_type, chimeralm/models/components/hyena.py:22,97-136; no mask on
   * the predict path): 0 attention (what ChimeraLM uses, chimeralm/models/lm.py:46-55), 1 mean, 2 max, 3 cls.  With a
   * pooling other than attention the `net.head.attention.*` tensors are not required. */
  int pooling;
} clm_config;

void clm_default_config(clm_config* cfg);
const char* clm_version(void);

/* Lifetime.  Replaces model construction: ChimeraLM.new()/from_pretrained()
 * (chimeralm/models/lm.py:12-61) + Lightning's module-to-device move. */
int clm_create(const clm_config* cfg, int device, clm_ctx** out);
void clm_destroy(clm_ctx* ctx);
const char* clm_last_error(const clm_ctx* ctx);

/* Weights.  `name` is the reference state-dict key (e.g.
 * "net.backbone.backbone.layers.0.mixer.in_proj.weight", "net.head.output_layer.bias";
 * layout probed from ClassificationLit(net=HyenaDna(...)), chimeralm/models/basic_module.py:39).
 * `data` is a HOST pointer, copied; the caller keeps ownership.  Unknown names are ignored
 * (returns 1) so a whole checkpoint can be streamed in.  Replaces load_state_dict /
 * trainer.predict(ckpt_path=...) (chimeralm/__main__.py:317). */
int clm_load_tensor(clm_ctx* ctx, const char* name, const void* data, int dtype, const int64_t* shape, int ndim);
/* Converts GEMM weights to bf16, generates the implicit long filters for all layers
 * (HyenaFilter.filter, recomputed on every forward in the reference) and their spectra. */
int clm_finalize(clm_ctx* ctx);
/* Sizes the activation workspaces (and clm_predict_host's staging) for batches up to max_B reads of max_T tokens.
 * No allocation happens inside clm_forward or clm_predict_host.  If it fails (CLM_ERR_NOMEM) the context holds NO
 * workspaces and refuses forwards until a smaller clm_reserve succeeds. */
int clm_reserve(clm_ctx* ctx, int max_B, int max_T);
/* Same with an explicit token budget: batches of up to max_B reads and up to max_T tokens per read whose padded size
 * B * T stays <= max_tokens (clm_reserve uses max_B * max_T).  This is what length-bucketed prediction wants - 256 reads
 * of 1 kb or 8 reads of 32 kb per batch - and what the reference's fixed `--batch-size` cannot express
 * (chimeralm/__main__.py:253; chimeralm/data/bam.py:287-299). */
int clm_reserve_tokens(clm_ctx* ctx, int max_B, int max_T, long long max_tokens);

/* Tokenisation + collation on the device.  Replaces tokenizer(seq, truncation=True,
 * max_length=...) (chimeralm/data/tokenizer.py:97, CharacterTokenizer :264-306) and
 * DataCollator.torch_call's padding (:152-159).
 *   d_bases   : device, concatenated ASCII bases of B reads
 *   d_offsets : device, int64[B+1] start offsets into d_bases
 *   max_bases : truncation (first max_bases bases are kept)
 *   d_ids_out : device, uint8[B, T_pad]; T_pad >= min(len,max_bases)+add_cls+add_sep for all reads
 *   d_lens_out: device, int32[B] token counts incl. specials (may be NULL) */
int clm_encode_batch(clm_ctx* ctx, const uint8_t* d_bases, const int64_t* d_offsets, int B, int T_pad, int add_cls,
                     int add_sep, int pad_left, int max_bases, uint8_t* d_ids_out, int32_t* d_lens_out,
                     void* stream);

/* The model forward.  Replaces ClassificationLit.forward / predict_step
 * (chimeralm/models/basic_module.py:67-77,177-187) = HyenaDna.forward
 * (chimeralm/models/components/hyena.py:244-256) and PredictionWriter's argmax
 * (chimeralm/models/callbacks.py:107).
 *   d_ids    : device, [B, T] token ids of dtype ids_dtype (CLM_U8, CLM_I32 or CLM_I64)
 *   d_logits : device, float32[B, 2]
 *   d_labels : device, uint8[B] = argmax(logits) with ties -> 0 (may be NULL) */
int clm_forward(clm_ctx* ctx, const void* d_ids, int ids_dtype, int B, int T, float* d_logits, uint8_t* d_labels,
                void* stream);

/* Status of an asynchronous clm_forward.  clm_forward_seq() is the sequence number of the forward issued last on this
 * context; once that forward's stream work is complete (the caller synchronises), clm_forward_status(ctx, seq)
 * returns 0, CLM_ERR_TOKEN_RANGE, or CLM_ERR_FP16_RANGE - the last kernel of every forward publishes the status word
 * into mapped host memory, so this costs no copy and no synchronisation.  The last 8 forwards can be queried;
 * CLM_ERR_STATE means the forward has not finished.  On CLM_ERR_FP16_RANGE the logits of that batch are invalid:
 * rerun it after clm_set_option(ctx, "tc_conv", 0), which selects the fp32 FFT convolution (the reference computes
 * fftconv in fp32: HF modeling_hyena.fftconv via chimeralm/models/components/hyena.py:249).  clm_predict_host does
 * this by itself; clm_tc_fallback_count() says how often. */
long long clm_forward_seq(const clm_ctx* ctx);
int clm_forward_status(clm_ctx* ctx, long long seq);
long long clm_tc_fallback_count(const clm_ctx* ctx);

/* End-to-end convenience with HOST buffers (pinned recommended): H2D copy of bases/offsets,
 * encode, forward, D2H copy of logits/labels, stream synchronise.  This is what bench.py's
 * `e2e` figure and the Python predict loop time. */
int clm_predict_host(clm_ctx* ctx, const uint8_t* h_bases, const int64_t* h_offsets, int B, int T_pad, int add_cls,
                     int add_sep, int pad_left, int max_bases, float* h_logits, uint8_t* h_labels);
/* The same in two halves, so that the host can prepare and enqueue batch k + 1 while batch k runs (the reference's
 * DataLoader workers + Lightning loop overlap the same way, chimeralm/__main__.py:308-317): submit copies and enqueues
 * one batch on the context's own stream and returns a ticket at once; wait blocks until THAT batch's h_logits /
 * h_labels are valid and returns its status (a batch that left the fp16 range of the tensor-core convolution is redone
 * with the fp32 kernel before wait returns).  Up to 3 batches may be in flight; the host buffers of a batch must stay
 * valid until its wait returns.  clm_predict_host == submit + wait. */
int clm_predict_host_submit(clm_ctx* ctx, const uint8_t* h_bases, const int64_t* h_offsets, int B, int T_pad, int add_cls,
                            int add_sep, int pad_left, int max_bases, float* h_logits, uint8_t* h_labels, int* ticket);
int clm_predict_host_wait(clm_ctx* ctx, int ticket);

/* Number of kernel launches issued by this context since creation (bench.py's gpu_launches). */
long long clm_launch_count(const clm_ctx* ctx);

/* Per-kernel-class device timing: while enabled, every launch is bracketed by CUDA events on
 * its own stream; clm_profile_get synchronises on them and returns the accumulated time and
 * launch count of one class (names from clm_profile_name, 0 <= cat < clm_profile_num()). */
int clm_profile_enable(clm_ctx* ctx, int on);
int clm_profile_reset(clm_ctx* ctx);
int clm_profile_num(void);
const char* clm_profile_name(int cat);
int clm_profile_get(clm_ctx* ctx, int cat, double* total_ms, long long* launches);

/* ---- unit-level entry points (parity tests call the kernels one by one through these) ---- */
/* out = epilogue(A[M,K] (bf16) * W[N,K]^T (bf16)); epi: 0 bias->bf16, 1 bias+gelu_tanh->bf16,
 * 2 bias+res->f32, 3 scorer (score[m] = sum_n gelu_erf(.)*w2[n] + b2, needs N == 256). */
int clm_gemm(clm_ctx* ctx, const void* d_A, const void* d_W, const float* d_bias, int M, int N, int K, int epi,
             void* d_out, const float* d_res, const float* d_w2, float b2, float* d_score, void* stream);
/* Fused first half of block `layer` (LayerNorm1 + in_proj + causal short conv + first gate; HF
 * HyenaBlock/HyenaOperator.forward, SURVEY.md A.3/A.6): d_res fp32 residual stream of B*T tokens in
 * the blocked R32 layout (with >= 160 rows of slack after the last token); outputs vx = v*x1 and
 * x0 as channel-major bf16 [B][256][Tp], Tp % 64 == 0. */
int clm_block_in(clm_ctx* ctx, int layer, const float* d_res, int B, int T, int Tp, void* d_vx, void* d_x0, void* stream);
/* Same, and CTA 0 records clock64() stamps (int64 [2][64], zero-filled by the caller): tuning aid. */
int clm_block_in_trace(clm_ctx* ctx, int layer, const float* d_res, int B, int T, int Tp, void* d_vx, void* d_x0,
                       long long* d_trace, void* stream);
/* Fused second half of block `layer` (out_proj + residual + LayerNorm2 + fc1 + GELU + fc2 +
 * residual; HF HyenaBlock.forward, SURVEY.md A.6): d_y bf16 [M,256] token-major, d_res fp32
 * [M,256] read and overwritten with the block output. */
int clm_block_mlp(clm_ctx* ctx, int layer, const void* d_y, float* d_res, int M, void* stream);
/* Same block tail, but y is the long convolution's channel-major output bf16 [B][256][Tp] (consumed as
 * an MN-major tensor-core operand, no transpose); d_res holds B*T rows in the R32 layout. */
int clm_block_mlp_cm(clm_ctx* ctx, int layer, const void* d_y_cm, float* d_res, int B, int T, int Tp, void* stream);
/* Same, and CTA 0 records clock64() stamps of its producer / MMA / epilogue roles into
 * d_trace (int64 [3][64], zero-filled by the caller) - a timeline for tuning, not a product path. */
int clm_block_mlp_trace(clm_ctx* ctx, int layer, const void* d_y, float* d_res, int M, long long* d_trace, void* stream);
/* Production form of the fused block tail (channel-major y, optional normalised-xn output into the context's
 * workspace) with the optional clock trace (d_trace may be NULL). */
int clm_block_mlp_cm_trace(clm_ctx* ctx, int layer, const void* d_y_cm, float* d_res, int B, int T, int Tp, int write_xn,
                           long long* d_trace, void* stream);
/* Runtime switches: "fused_mlp" / "fused_in" (default 1) select the fused block kernels in clm_forward.  Others select a
 * different kernel for the same math (A/B partners and test hooks; every one of them is held to the logit tolerance by
 * tests/test_gpu_forward.py::test_kernel_variants_agree): "tc_conv", "tc_pipe", "tc_pack4", "tc_chunked",
 * "tc_pipe_chunked" (forms of the long convolution), "fused_score_pool", "fused_head", "head_coop", "skip_dead_res",
 * "embed_in" / "embed_res" (block 0's first half and residual input by table lookup over the token ids, default 1),
 * "mlp_gather_tails" / "in_ext_tail" (tail tokens share tiles, default 1), "y_channel_major".  Unknown names are an error. */
int clm_set_option(clm_ctx* ctx, const char* name, int value);
/* out = (causal_long_conv(vx, k_layer) + bias_layer * vx) * x0 on channel-major bf16 [B][D][Tp]. */
int clm_longconv(clm_ctx* ctx, int layer, const void* d_vx, const void* d_x0, void* d_out, int B, int T, int Tp,
                 void* stream);
/* Copies the generated time-domain filter k[layer][:, :L] (float32 [D, L]) to a device buffer. */
/* Attention-pooling weights of the LAST clm_forward (same B, T): d_out[b*T + t] = softmax_t(score[b, :]).  Replaces
 * `save_attention=True` / `BinarySequenceClassifier.attention_weights` (chimeralm/models/components/hyena.py:129-130,
 * chimeralm/models/lm.py:14,30). */
int clm_attention_weights(clm_ctx* ctx, float* d_out, int B, int T, void* stream);
/* Tensor-core FFT long convolution (reads of 2 057 .. 32 769 tokens; rows past T must be zero below 8 192 tokens, Tp a multiple of 128): same contract as clm_longconv except
 * that d_vx holds fp16 values (what the fused in_proj kernel emits when this kernel follows). */
int clm_longconv_tc(clm_ctx* ctx, int layer, const void* d_vx_f16, const void* d_x0, void* d_out, int B, int T, int Tp,
                    void* stream);
/* Unit-test form of what the forward does around that kernel: d_vx holds bf16 values of ANY magnitude; the per-channel
 * power-of-two input scale is taken from the data itself (in the forward it comes from clm_finalize's calibration
 * draw and is applied by the fused in_proj kernel), the rows are converted to fp16, the kernel runs and the output is
 * scaled back.  Synchronous; returns CLM_ERR_FP16_RANGE when an intermediate overflowed. */
int clm_longconv_tc_auto(clm_ctx* ctx, int layer, const void* d_vx_bf16, const void* d_x0, void* d_out, int B, int T, int Tp,
                         void* stream);
/* Which long-convolution kernel clm_forward uses for reads of T tokens: 0 = first fp32 FFT kernel, 1 = tuned fp32
 * FFT kernel, 2 = tensor-core FFT kernel; -1 before clm_finalize. */
int clm_longconv_variant(const clm_ctx* ctx, int T);
/* Same, and CTA 0 writes clock64() stamps into d_trace (int64, zero-filled by the caller): the two-items-in-flight kernel
 * (default) fills [9][64] - row 0 the MMA issuer (start / barrier passed / end per slot), rows 1..8 the epilogue warps; the
 * one-item kernels (options tc_pipe=0, tc_pipe_chunked=0) fill [2][64]. */
int clm_longconv_tc_trace(clm_ctx* ctx, int layer, const void* d_vx_f16, const void* d_x0, void* d_out, int B, int T,
                          int Tp, long long* d_trace, void* stream);
int clm_get_filter(clm_ctx* ctx, int layer, float* d_out, int L, void* stream);
/* Forward stops after (layer, stage); layer == n_layer addresses the final stages; -1 disables.
 * Stages: 0 embed | per layer 1 ln1 2 in_proj 3 shortconv+gate 4 longconv 5 transpose 6 out_proj
 * 7 ln2 8 fc1 9 fc2 | final 10 ln_f 11 scores 12 pooling 13 head. */
int clm_set_debug_stop(clm_ctx* ctx, int layer, int stage);
/* Copies a named workspace ("resid","xn","u","vx","x0","y","yt","score","pooled") to d_dst. */
int clm_debug_copy(clm_ctx* ctx, const char* what, void* d_dst, size_t max_bytes, void* stream);

/* ---- Fine-tuning of the head with the backbone frozen ---------------------------------------
 * Replaces ClassificationLit.training_step / model_step (cross-entropy on net(input_ids),
 * chimeralm/models/basic_module.py:87-104,106-...) and configure_optimizers (AdamW, :200-223) for the
 * head's 986 627 parameters (net.head.attention.* and net.head.classifier.* / output_layer.*); the
 * backbone's weights, filters and spectrum tables are never written.  Attention pooling only (the
 * named architecture, chimeralm/models/lm.py:46-55): other poolings return CLM_ERR_INVALID.
 * Without a clm_head_train_begin call the library behaves exactly as without these entry points. */
typedef struct {
  float lr, beta1, beta2, eps, weight_decay;   /* torch.optim.AdamW semantics, bias correction included */
  double dropout;                              /* p of the head's three nn.Dropout layers (0.1 in the reference) */
  unsigned int seed;                           /* dropout masks: see the hash in csrc/head_train.cuh */
} clm_head_train_cfg;

/* Allocates the fp32 master copies of the head tensors (initialised from the loaded weights), the AdamW state and every
 * buffer a step needs, for batches of up to the max_B of the last clm_reserve.  The only allocation: a step allocates
 * nothing.  Needs clm_finalize and clm_reserve first; a second call returns CLM_ERR_STATE. */
int clm_head_train_begin(clm_ctx* ctx, const clm_head_train_cfg* cfg);
/* One optimizer step on a batch: clm_forward with the loaded backbone, the classifier again with dropout, mean cross-
 * entropy against d_targets (device, int64[B], values 0 / 1), the head's backward and AdamW; afterwards the forward reads
 * the updated head.  Asynchronous on `stream`; d_loss_out (device float, may be NULL) receives the batch's loss.  The
 * step's status is that of its forward: clm_forward_status(ctx, clm_forward_seq(ctx)) - and when that is not 0 the step
 * changed no weight (a batch that left the fp16 range of the tensor-core convolution can be redone with
 * clm_set_option(ctx, "tc_conv", 0)).  The dropout masks of the k-th call (k = 0, 1, ...) use step = k. */
int clm_head_train_step(clm_ctx* ctx, const void* d_ids, int ids_dtype, int B, int T, const int64_t* d_targets,
                        float* d_loss_out, void* stream);
/* Copies the gradient of head tensor `name` (state-dict key, e.g. "net.head.attention.0.weight") of the last step to the
 * device buffer d_dst (float32, the tensor's element count).  For parity tests. */
int clm_head_grad_copy(clm_ctx* ctx, const char* name, float* d_dst, void* stream);
/* Copies the current value of head tensor `name` to the HOST buffer h_dst (float32).  Synchronises the device.  It also
 * refreshes the forward's host-side copy of net.head.attention.2.bias, which enters every score of a read equally and so
 * changes no logit, attention weight or label. */
int clm_head_export(clm_ctx* ctx, const char* name, float* h_dst);

/* ---- Native BAM ingest (host only, no GPU needed) ----------------------------------------
 * Replaces, for `chimeralm predict`, pysam.AlignmentFile iteration + is_chimeric +
 * parse_bam_file (chimeralm/data/bam.py:21-38) and the per-read Python objects the HF dataset
 * generator builds from them (chimeralm/data/bam.py:129-174).  BGZF blocks are inflated by
 * n_threads workers (<= 0: all host cores) one chunk ahead of the parser; CRCs are checked. */
typedef struct clm_bam clm_bam;
int clm_bam_open(const char* path, int n_threads, clm_bam** out);
void clm_bam_close(clm_bam* r);
/* Message of the last failure on `r`; with r == NULL, of the last failed clm_bam_open on the
 * calling thread. */
const char* clm_bam_error(const clm_bam* r);
/* Records consumed so far (kept or not). */
long long clm_bam_records_seen(const clm_bam* r);
/* Compressed bytes read from the file per background load (default 16 MiB); mainly for tests of the block / record carry
 * across loads. */
int clm_bam_set_chunk_bytes(clm_bam* r, long long bytes);
/* Data-parallel sharding (Lightning's predict sampler: rank r takes kept reads r, r+W, ...,
 * chimeralm/data/bam.py:287-299 under DDP): after this call clm_bam_next only returns the
 * kept reads whose running index i satisfies i % world == rank; the others are skipped
 * without being decoded. */
int clm_bam_set_shard(clm_bam* r, int rank, int world);
/* Decodes the next reads, in file order, into caller-owned (ideally pinned) host buffers:
 *   bases   : ASCII bases of the kept reads back to back, each cut to its first max_bases
 *   offsets : int64[max_reads + 1] start offsets into bases (offsets[0] = 0)
 *   names   : max_reads rows of name_stride bytes, NUL-terminated query names (may be NULL)
 * chimeric_only != 0 keeps only records passing the reference's is_chimeric (mapped, SA tag,
 * not secondary, not supplementary).  Stops at max_reads, when the next read would overflow
 * bases_cap (it is kept for the next call), or at end of file.  Returns the number of reads
 * written (0 = end of file) or a negative clm_status. */
long long clm_bam_next(clm_bam* r, long long max_reads, long long max_bases, int chimeric_only, uint8_t* bases,
                       long long bases_cap, int64_t* offsets, char* names, int name_stride);

#ifdef __cplusplus
}
#endif
#endif /* CHIMERALM_B200_H_ */
