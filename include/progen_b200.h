/* libprogen_b200.so — C ABI of the B200-native ProGen hot path.
 *
 * Drop-in boundary (SURVEY.md §8(b)): the reference exposes `ProGen(**kwargs) -> .init / .apply`
 * (lucidrains/progen progen_transformer/progen.py:235-243) and everything below that call is executed by XLA.
 * This library replaces that device path.  Each entry point names the reference lines whose arithmetic it owns.
 *
 * Conventions
 *  - every function returns 0 on success or a negative PROGEN_ERR_* code; `progen_last_error()` (thread-local) has
 *    the text.  Nothing allocates: the caller owns every buffer and workspace.  All work is asynchronous on `stream`
 *    (a cudaStream_t passed as void*), no internal synchronisation, no global mutable state except a cache of TMA
 *    descriptors keyed by (pointer, shape).
 *  - tokens are rows: activations are row-major [T = B * seq_len, features]; `ld*` are element strides.
 *  - dtype codes: PROGEN_F32 = 0, PROGEN_BF16 = 1.  The residual stream and all parameter gradients are fp32.
 *  - sm_100a only (`progen_device_check`); there is no CPU or other-architecture fallback.
 */
#ifndef PROGEN_B200_H
#define PROGEN_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PROGEN_F32 0
#define PROGEN_BF16 1

#define PROGEN_BACKEND_SIMT 0     /* fp32-exact CUDA-core GEMM (mixed_precision=False path, progen.py:235) */
#define PROGEN_BACKEND_TCGEN05 1  /* TMA + tcgen05.mma + TMEM GEMM, bf16 operands / fp32 accumulate */

/* GEMM epilogues (fused with the matmul the reference line performs) */
#define PROGEN_EPI_STORE 0     /* out = acc (+bias)                      progen.py:219-222 (logits), 185 (SGU proj)   */
#define PROGEN_EPI_ROTARY 1    /* out = rotary(acc)                      progen.py:83-87 (to_qkv, rotary on q,k,v)    */
#define PROGEN_EPI_RESIDUAL 2  /* out(f32) = (aux|out)(f32) + acc + bias   progen.py:103+230, 148+231                    */
#define PROGEN_EPI_GLU 3       /* out2 = pre-act, out = val*gelu(gate)   progen.py:137-141                             */
#define PROGEN_EPI_GELU 4      /* out2 = pre-act, out = gelu(pre)        progen.py:137,143                             */
#define PROGEN_EPI_GLU_BWD 5   /* out = d(pre-act) from acc = d(GLU out) (backward of 3)                               */
#define PROGEN_EPI_GELU_BWD 6  /* out = acc * gelu'(pre-act)             (backward of 4)                               */
#define PROGEN_EPI_ACCUM 7     /* out(f32) += acc  (weight gradients; optional tril mask for SGU spatial_weights)     */

const char* progen_version(void);
const char* progen_last_error(void);
int progen_device_check(void);
/* number of kernels this library has launched in this process (bench.py reports the per-run delta) */
long long progen_launch_count(void);

/* D[M,N] (+)= A[M,K] * B[N,K]^T.  Operand X(m,k): K-major -> X[m*ld + k]; MN-major -> X[k*ld + m].
 * Replaces every jnp matmul/einsum of the path: hk.Linear (progen.py:70-71,125-126,164,221), the SGU spatial
 * einsum 'n d, m n -> m d' (progen.py:181; causal=1 skips the masked upper-triangular K tiles), and their
 * transposes in the backward pass (jax.value_and_grad, utils.py:72). */
typedef struct progen_gemm_t {
  int32_t M, N, K;
  int32_t a_mn_major, b_mn_major;
  int32_t batch;         /* independent problems (grid z), >= 1 */
  int32_t batch_reduce;  /* 1: all batches accumulate into the same output (needs EPI_ACCUM + atomic) */
  int32_t causal;        /* 0 none, 1 lower (k < m0+128 only), 2 upper (k >= m0 only) */
  int32_t split_k;       /* >= 1; > 1 needs EPI_ACCUM + atomic */
  int32_t in_dtype, out_dtype, epi_kind, backend;
  int32_t seq_len, dim_head;          /* EPI_ROTARY */
  int32_t atomic, tril, tril_rows;    /* EPI_ACCUM */
  int64_t lda, ldb;
  int64_t a_batch_rows, b_batch_rows, d_batch_rows;   /* stored rows to skip per batch (0 = operand shared) */
  int64_t ldo, ldo2, ldaux;
  const void* A;
  const void* B;
  void* out;
  void* out2;
  const float* bias;
  const void* aux;
  const float* rot_sin;   /* [seq_len, dim_head/2], fixed_pos_embedding progen.py:24-28 */
  const float* rot_cos;
} progen_gemm_t;

int progen_gemm(const progen_gemm_t* desc, void* stream);

/* hk.Embed row gather — progen.py:207,226.  x is the fp32 residual stream [T, d]. */
int progen_embed_fwd(const int* tokens, const float* table, float* x, long long T, int d, int V, void* stream);
/* gradient of the gather: dtable[v,:] += sum_{t: tokens[t]==v} dx[t,:] */
int progen_embed_bwd(const int* tokens, const float* dx, float* dtable, long long T, int d, int V, void* stream);

/* y = shift_tokens(LayerNorm(x) * scale) — progen.py:22,43-46,74-77,132-135 (shift=1) and 170, 220 (shift=0).
 * Saves mean / rstd per row for the backward pass. */
int progen_ln_shift_fwd(const void* x, long long ldx, int x_dtype, const float* scale, void* y, long long ldy, int y_dtype,
                        float* mean, float* rstd, long long T, int d, int seq_len, int shift, void* stream);
/* backward of the above; residual=1 accumulates into the fp32 residual gradient `dres` [T,d] and mirrors it to `dout`;
 * `dres_colsum` (nullable, residual only) += column sums of the updated dres = the bias gradient of the Linear that
 * produced this residual branch's input (saves a separate pass over dres). */
int progen_ln_shift_bwd(const void* dy, long long lddy, int act_dtype, const void* x, long long ldx, int x_dtype,
                        const float* scale, const float* mean, const float* rstd, float* dres, void* dout, long long ldo,
                        float* dscale, float* dres_colsum, long long T, int d, int seq_len, int shift, int residual,
                        void* stream);

/* out[c] += sum_t in[t,c] — bias gradients of every hk.Linear */
int progen_colsum(const void* in, long long ld, int dtype, float* out, long long T, int N, void* stream);

/* cross_entropy + masked_mean + batch mean — utils.py:42-59,76 (pad-as-EOS mask, Q8); fused forward + d(logits).
 * *loss must be zeroed by the caller; inv_batch = 1/global_batch (DDP: a sum over ranks yields the global mean). */
int progen_ce_fwd_bwd(const void* logits, int dtype, const int* labels, float* weights, float* loss, void* dlogits,
                      int dlogits_dtype, int B, int n, int V, float inv_batch, void* stream);

/* backward of apply_rotary_pos_emb (progen.py:36-41) on the [T, ncols] q|k|v gradient, in place */
int progen_rotary_bwd(void* dqkv, long long ld, int dtype, const float* sin_t, const float* cos_t, long long T, int ncols,
                      int seq_len, int dim_head, void* stream);

/* sliding-window attention with one look-back window — progen.py:88-102 (q,k,v already rotated, [T, 3*heads*dim_head]).
 * `_simt`: fp32-exact CUDA-core kernels.  lse / delta: [T, heads] fp32. */
int progen_local_attn_fwd_simt(const void* qkv, void* out, float* lse, int dtype, int B, int seq_len, int window, int heads,
                               int dim_head, void* stream);
int progen_local_attn_bwd_simt(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv,
                               float* delta, int dtype, int B, int seq_len, int window, int heads, int dim_head,
                               void* stream);

/* tensor-core version (bf16, dim_head 64, window % 64 == 0): flash-style, scores stay on chip; same buffers as above */
int progen_local_attn_fwd(const void* qkv, void* out, float* lse, int B, int seq_len, int window, int heads, int dim_head,
                          void* stream);
int progen_local_attn_bwd(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv, float* delta,
                          const float* rot_sin, const float* rot_cos, int B, int seq_len, int window, int heads, int dim_head,
                          void* stream);

/* tcgen05 forward (TMA-staged K/V, QK^T and PV as tcgen05.mma with S/O in TMEM, softmax by row-owning threads);
 * window % 128 == 0.  Same buffers as progen_local_attn_fwd. */
int progen_local_attn_fwd_tc(const void* qkv, void* out, float* lse, int B, int seq_len, int window, int heads, int dim_head,
                             void* stream);

/* tcgen05 backward (dQ kernel + dK/dV kernel, no atomics; delta produced by the dQ kernel); window % 128 == 0 */
int progen_local_attn_bwd_tc(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv, float* delta,
                             const float* rot_sin, const float* rot_cos, int B, int seq_len, int window, int heads, int dim_head,
                             void* stream);
/* Same, with the rotary tables also given transposed (rot_sin_t / rot_cos_t: [dim_head/2, seq_len], or both null; the
 * [seq_len, dim_head/2] tables are then required too) and the kernel variant chosen per call: mode 0 round-1 kernels,
 * 1 / 2 / 3 round-2 kernels (3: gradient tiles stored through TMA, reading the transposed tables), -1 the
 * PROGEN_ATTN_BWD_TS environment variable (default 3).  All modes compute the same gradients. */
int progen_local_attn_bwd_tc_ex(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv, float* delta,
                                const float* rot_sin, const float* rot_cos, const float* rot_sin_t, const float* rot_cos_t, int B,
                                int seq_len, int window, int heads, int dim_head, int mode, void* stream);

/* SGU gating — progen.py:182-184: out = xs * (Gp + spatial_biases[m]) and its backward (dxs, dGp, dbias) */
int progen_sgu_gate_fwd(const void* xs, long long ldx, const void* gp, long long ldg, const float* bias, void* out,
                        long long ldo, int dtype, long long T, int C, int seq_len, void* stream);
int progen_sgu_gate_bwd(const void* ds, long long ldds, const void* xs, long long ldx, const void* gp, long long ldg,
                        const float* bias, void* dxs, long long lddx, void* dgp, long long lddg, float* dbias, int dtype,
                        long long T, int C, int seq_len, void* stream);
/* da *= gelu'(u) (tanh-approximate GELU, jax.nn.gelu default — progen.py:143) */
int progen_gelu_bwd(void* da, const void* u, int dtype, long long numel, void* stream);
int progen_cast_f32(const float* in, void* out, int out_dtype, long long numel, void* stream);
/* out = tril(spatial_weights) in the act dtype — the mask of progen.py:178-179 applied once per parameter update */
int progen_tril_cast(const float* w, void* out, int out_dtype, int n, void* stream);

/* optimizer: optax.chain(clip_by_global_norm, adamw(mask = ndim > 1), apply_every(k)) — train.py:115-121,189-190 */
int progen_optim_workspace_floats(void);
int progen_grad_sqnorm(const float* g, long long n, float* workspace, float* out_sqnorm, void* stream);
int progen_adamw_step(float* p, void* p_lp, const float* g, float* m, float* v, float* acc, long long n, long long n_decay,
                      const float* gnorm_sq, float lr, float b1, float b2, float eps, float wd, float max_norm,
                      long long step, int emit, void* stream);
/* same call with the step-dependent scalars (Adam count, bias corrections, emit = count % apply_every == 0) kept in a
 * 32-byte device `state` ({int64 count; float bc1, bc2; int32 emit; pad}) that a 1-thread kernel advances: every launch
 * argument is step-invariant, so a captured CUDA graph of the whole training step (train.py:186-190) can be replayed */
int progen_adamw_step_dev(float* p, void* p_lp, const float* g, float* m, float* v, float* acc, long long n, long long n_decay,
                          const float* gnorm_sq, float lr, float b1, float b2, float eps, float wd, float max_norm,
                          int apply_every, void* state, void* stream);

/* ---- KV-cached decode (BASELINE config 5; replaces the full re-forward per token of utils.py:115-117) ----
 * Weights are TRANSPOSED copies ([out, in], fp32 or bf16 per `wdtype`); caches and scratch are fp32 device buffers owned
 * by the caller.  `layers` is a HOST array of `depth` entries. */
typedef struct progen_decode_layer_t {
  int32_t kind;                /* 0 GLU, 1 GELU, 2 gMLP/SGU  (progen.py:210-212) */
  int32_t _pad;
  const float* ln1_scale;      /* [d] */
  const void* wqkv_t;          /* [3*inner, d] */
  const void* wo_t;            /* [d, inner] */
  const float* bo;             /* [d] */
  const float* ln2_scale;      /* [d] */
  const void* win_t;           /* [2*hid | hid, d]; GLU: rows [0,hid) value, [hid,2hid) gate */
  const float* bin;
  const void* wout_t;          /* [d, hid | hid/2] */
  const float* bout;           /* [d] */
  const float* sgu_ln_scale;   /* [hid/2] */
  const float* sgu_w;          /* [n, n] fp32 spatial_weights (row p is read up to column p) */
  const float* sgu_b;          /* [n] */
  const void* sgu_proj_t;      /* [hid/2, hid/2] */
  const float* sgu_proj_b;
  float* kcache;               /* [n, inner] rotated keys */
  float* vcache;               /* [n, inner] rotated values */
  float* shift1;               /* [2][d/2] previous position's LN half (attention block), indexed by position parity */
  float* shift2;               /* [2][d/2] previous position's LN half (feed-forward block) */
  float* gn_hist;              /* [n, hid/2] normalised gate history (gMLP layers) */
} progen_decode_layer_t;

typedef struct progen_decode_t {
  int32_t n, d, heads, dim_head, inner, window, hid, V, depth, wdtype, shift_tokens, top_k;
  const float* embed;          /* [V, d] */
  const float* lnf_scale;      /* [d] */
  const void* whead_t;         /* [V, d] */
  const float* bhead;          /* [V] */
  const float* rot_sin;        /* [n, dim_head/2] */
  const float* rot_cos;
  const progen_decode_layer_t* layers;
  int32_t* seq;                /* [n] device: token ids; sampled ids are ADDED in place (utils.py:129) */
  int32_t* pos;                /* device scalar: position consumed by the next step */
  const float* noise;          /* [n, V] gumbel noise, or NULL for the greedy limit */
  float* logits_all;           /* [n, V] every step's logits (may be NULL) */
  float *x, *y, *q, *att, *u, *gn, *sg, *pj, *logits;   /* scratch: d, d, inner, inner, 2*hid, hid/2, hid/2, hid/2, V */
} progen_decode_t;

int progen_decode_step(const progen_decode_t* model, int do_sample, void* stream);

/* Whole-generation decode in ONE persistent cooperative kernel (csrc/decode_persist.cu): consumes positions
 * pos0 .. pos0 + nsteps - 1 of B sequences in lock step (reference utils.py:106-135 per sequence; sample.py:66-71).
 * `layers` is a DEVICE array of `depth` progen_decode_layer_t whose cache / state pointers are batch-major:
 * kcache, vcache [B, heads, n, dim_head] (a head's keys are contiguous: the windowed read streams); shift1, shift2 [B, 2, d/2];
 * gn_hist [B, n, hid/2].  Sequence b keeps its prime before start[b]: position p+1 is sampled (seq[b][p+1] += id, quirk Q5)
 * iff p+1 >= start[b].  grid_bar (one uint32) must be zero on entry; att_count ([B * heads] int32) is reserved (the attention
 * merges no longer use a global counter).  Limits: B <= 64, dim_head a power of two in [8, 64], window <= 512, V <= 512,
 * feature widths <= 8192. */
typedef struct progen_decode_run_t {
  int32_t n, d, heads, dim_head, inner, window, hid, V, depth, wdtype, shift_tokens, top_k;
  int32_t B, pos0, nsteps, _pad;
  const float* embed;          /* [V, d] */
  const float* lnf_scale;      /* [d] */
  const void* whead_t;         /* [V, d] */
  const float* bhead;          /* [V] */
  const float* rot_sin;        /* [n, dim_head/2] */
  const float* rot_cos;
  const progen_decode_layer_t* layers;   /* device */
  int32_t* seq;                /* [B, n] token ids; sampled ids are ADDED in place */
  const int32_t* start;        /* [B] first sampled position of each sequence */
  const float* noise;          /* [B, n, V] gumbel noise, or NULL for the greedy limit */
  float* logits_all;           /* [B, n, V] every step's logits (may be NULL) */
  float* x;                    /* [B, d] residual stream */
  float* q;                    /* [B, inner] */
  float* att;                  /* [B, inner] */
  float* att_part;             /* [B, heads, ceil(2*window/32), dim_head + 4] partial (max, sum, -, -, out) per 32-key slice */
  int32_t* att_count;          /* [B, heads] reserved (non-null) */
  float* u;                    /* [B, hid] */
  float* sg;                   /* [8, B, hid/2] partial spatial gates (up to 8 splits of the history range) */
  float* pj;                   /* [B, hid/2] */
  float* logits;               /* [B, V] */
  uint32_t* grid_bar;          /* grid barrier counter */
  long long* prof;             /* optional [2][160][2] clock64 at entry / exit of every grid barrier of the launch's last
                                  step, for CTA 0 and the last CTA, then [160][8] marks inside CTA 0's phases (NULL: off) */
} progen_decode_run_t;

int progen_decode_run(const progen_decode_run_t* run, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PROGEN_B200_H */
