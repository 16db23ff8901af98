/*
 * deer_b200.h -- C ABI of libdeer_b200.so (hand-written sm_100a CUDA for the DEER hot path).
 *
 * The reference (kalgeee/Uncertainty-Aware-Multimodal-Emotion-Recognition) is pure PyTorch and has NO
 * FFI/operator interface (SURVEY.md section 8b); its boundary is the Python class/dict API, which the
 * host package mirrors.  This header is the boundary a maintainer would bind instead of the stock ATen
 * calls; every entry point cites the reference call site it replaces (paths relative to the reference
 * repository root).  INTEGRATION.md shows the ctypes stub.
 *
 * Conventions
 *   - plain pointers and sizes only; all pointers are DEVICE pointers unless stated; fp32 row-major.
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous on it and never synchronise,
 *     never allocate and never free (graph-capture safe).  Scratch memory is caller-provided.
 *   - return 0 on success; <0 on error: -1 invalid argument, -2 unsupported shape, -(1000+e) CUDA error e.
 *     deer_last_error() returns a thread-local description.
 *   - ld* are leading dimensions in ELEMENTS.
 */
#ifndef DEER_B200_H
#define DEER_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define DEER_OK 0
#define DEER_ERR_INVALID (-1)
#define DEER_ERR_UNSUPPORTED (-2)

/* activation codes for fused epilogues */
#define DEER_ACT_NONE 0
#define DEER_ACT_RELU 1
#define DEER_ACT_TANH 2
#define DEER_ACT_SIGMOID 3

/* GEMM engines */
#define DEER_GEMM_AUTO 0   /* tcgen05 when the shape/alignment allows it, SIMT otherwise */
#define DEER_GEMM_SIMT 1   /* fp32 CUDA-core tiles (exact fp32; small or unaligned shapes) */
#define DEER_GEMM_TF32 2   /* tcgen05.mma kind::tf32, fp32 accumulate in TMEM, TMA-fed */
#define DEER_GEMM_TF32X3 5 /* error-compensated 3xTF32 tensor-core tiles (fp32-grade accuracy at every M): the engine of
                              the post-pooling fusion / head chain, see deer_gemm_x3 */
/* LSTM recurrence engines (deer_lstm_fwd/bwd `engine`): DEER_GEMM_SIMT = exact-fp32 stepwise; DEER_GEMM_AUTO/TF32 =
 * round-1 8-CTA TF32 persistent forward kernel when H == 256 (stepwise otherwise; backward always stepwise);
 * 3 = stepwise with TF32 step GEMMs; 4 = same as AUTO.  These natural-layout entry points are the on-device reference;
 * the production path is deer_lstm_cluster_fwd/bwd below. */
#define DEER_LSTM_STEPWISE_TF32 3
#define DEER_LSTM_PERSISTENT_V1 4

int deer_version(void);
/* which engine the dispatchers picked, counted per call since process start (the parity tests assert that the
 * benchmarked dispatch -- tcgen05 for the time-batched contractions -- is the one they exercised) */
#define DEER_ENGINE_SIMT 1       /* exact-fp32 CUDA-core tiles */
#define DEER_ENGINE_TF32 2       /* tcgen05 kind::tf32, 128x128 tiles */
#define DEER_ENGINE_TF32_PAIR 3  /* tcgen05 kind::tf32, cta_group::2 256x256 tiles */
#define DEER_ENGINE_H16 4        /* tcgen05 kind::f16 (deer_gemm_h16) */
#define DEER_ENGINE_TF32X3 5     /* error-compensated 3xTF32 tensor-core tiles (fp32-grade accuracy) */
#define DEER_ENGINE_H16_SPLIT 6  /* tcgen05 kind::f16 on FP16 hi/lo operand pairs, 3 passes (deer_gemm_h16_split) */
long long deer_gemm_engine_count(int engine);
const char* deer_last_error(void);
/* number of kernels launched by this library since process start (bench.py `gpu_launches`) */
long long deer_launch_count(void);
/* timeline probe: a one-thread kernel that writes %globaltimer (ns) to slots[index] when the stream reaches it; capturable
 * into CUDA graphs, so the phases of a replayed step can be timed on every stream (tools/step_timeline.py) */
int deer_timestamp(unsigned long long* slots, int index, void* stream);
/* process-wide tuning switches (testing / ablation) */
#define DEER_OPT_TMA_TF32_ROUND 1 /* 1 (default): TMA loads fp32 operands as TFLOAT32 (rounded); 0: raw fp32 bits */
#define DEER_OPT_LSTM_TS 2        /* 1 (default): resident recurrent weights in TMEM (tcgen05.mma A from TMEM); 0: in smem */
#define DEER_OPT_LSTM_TILE 3      /* 0 (default): auto; 16 or 32: batch columns per cluster of the persistent LSTM */
#define DEER_OPT_SMALL_GEMM 4      /* 2 (default): cp.async-pipelined exact-fp32 small-problem GEMM; 1: register-staged one */
#define DEER_OPT_H16_PAIR 5        /* 1 (default): 16-bit GEMM on cta_group::2 CTA pairs (256x256 tiles); 0: single-CTA kernel */
#define DEER_OPT_TF32_PAIR 6       /* 1 (default): large TF32 GEMMs on the CTA-pair kernel (256x256 tiles); 0: 128x128-tile kernel */
#define DEER_OPT_NIG_PIPELINE 8    /* 1 (default): software-pipelined operand loads in the two NIG loss passes (80 registers, 4 blocks/SM); 0: load -> compute trips (64 registers, 5 blocks/SM) */
#define DEER_OPT_LSTM_DUAL 9       /* 1 (default): inference LSTM at 32 batch columns per CTA = two interleaved 16-column sub-tiles (own warps, shared resident weights); 0: one monolithic 32-column tile; 2: experiment - also the TRAINING forward of a one-wave batch as dual sub-tiles on half the SMs (measured slower: 4.66 -> 5.39 ms, the audio stream is the critical path) */
#define DEER_OPT_LSTM_COLSPLIT 10  /* 1: forward LSTM on 16-column tiles with 16 compute warps (two column halves per tile; same results, measured no faster: the step is instruction-issue bound); 0 (default): 8 compute warps */
#define DEER_OPT_LSTM_KEEP16 11    /* 1 (default): the activated gates / cell states the LSTM forward keeps for BPTT (`gact`, `c_blk`) are FP16 (half the bytes of the recurrence's dominant store / load stream); 0: fp32.  Both kernels read the option, so it must not change between a forward and its backward */
#define DEER_OPT_LSTM_STASYNC 12   /* 1: the forward recurrence all-gathers h with per-lane st.async stores (16 bytes, completion counted on the peer's mbarrier) straight into the peers' B-operand tiles; 0 (default; measured equal or faster in every configuration): one bulk copy (cp.async.bulk.shared::cluster) per warp and destination */
#define DEER_OPT_LSTM_HALFSPLIT 13 /* 1: forward recurrence on 16-column tiles as TWO independent 8-column halves per CTA (own compute warps, accumulators, B-operand tiles and barriers; shared resident weights and MMA warp): one half's DSMEM exchange flies while the other half's gates are computed (the kernel alone: 1.46 -> 1.33 us/step; the whole step: slower, so off); 0 (default): one 16-column recurrence per CTA */
#define DEER_OPT_LSTM_CARVEOUT 14  /* 1 (default): the persistent LSTM kernels request the maximum shared-memory carve-out, so that a <= 100 KB GEMM CTA of a concurrent stream can share the SM with a recurrence CTA (must be set before the first LSTM launch of the process: the attribute is applied once per kernel) */
#define DEER_OPT_LSTM_XIN 15       /* 1 (default): the first LSTM layer's input projection (In <= 128) runs INSIDE the forward recurrence kernel (deer_lstm_cluster_fwd_xin): no pre-activation tensor; 3: only in the 16-column-tile kernel (the dual-sub-tile inference kernel keeps the GEMM); 0: projection GEMM + deer_lstm_cluster_fwd_pre16 */
#define DEER_OPT_PDL 7             /* 1: launch kernels with programmatic stream serialization (PDL); 0 (default, faster as measured) */
int deer_set_option(int option, int value);
/* debugging aid: device buffer of >= 32 int64 that receives a clock64() trace of four steps of the persistent LSTM
 * kernels' block 0 (NULL disables; tools/lstm_probe.py --prof) */
int deer_lstm_set_profile_buffer(long long* device_buf);

/* ---- dense contractions: every nn.Linear on the path (encoders.py:93-107,443-475,597-625;
 *      fusion.py:98-103,201-219,286-304; deer.py:48-56,215-222; complete_project.py:61-417), the
 *      time-batched LSTM input projections (encoders.py:82,380) and the Conv1d taps (encoders.py:450-459).
 *      C[b] = act(opA(A[b]) * opB(B[b]) + bias[b] + beta * C[b])      (beta in {0,1}; beta=1 chains K-blocks of a
 *      concatenated input -- Linear(cat[a,b]) = a W1^T + b W2^T -- and accumulates weight gradients)
 *      opA(A) is M x K: transA=0 -> A stored [M,K] (lda>=K); transA=1 -> A stored [K,M] (lda>=M).
 *      opB(B) is K x N: transB=0 -> B stored [K,N] (ldb>=N); transB=1 -> B stored [N,K] (ldb>=K)  (nn.Linear weight).
 *      batch>=1 with element strides sA/sB/sC/sBias (may be negative or zero). bias may be NULL. */
/*      Sliding-window operands: a leading dimension SMALLER than the row length describes overlapping rows (row i starts
 *      ld elements after row i-1).  Accepted on the TMA engines only (CTA-pair kernels): A with transA = 0, B with
 *      transB = 0, and C with beta = 1 (overlapping output rows are accumulated with TMA reduce-add).  Other shapes
 *      return DEER_ERR_UNSUPPORTED. */
int deer_gemm(const float* A, long long lda, int transA, const float* B, long long ldb, int transB,
              float* C, long long ldc, int M, int N, int K, const float* bias, int act, float beta,
              int batch, long long sA, long long sB, long long sC, long long sBias, int engine, void* stream);

/* ---- 16-bit-operand engine for the time-batched LSTM contractions (csrc/gemm_h16.cu): same contract as deer_gemm
 *      (batch = 1) but A and B are both FP16 (a_bf16 = b_bf16 = 0) or both BF16 (= 1) matrices; accumulation and C
 *      are fp32.  16-bit OUTPUT: pass C = NULL and C16 (FP16, or BF16 with c16_bf16 = 1; row pitch ldc16 elements, a
 *      multiple of 8): the result is rounded once, after bias/activation, and only 2 bytes per element are written
 *      (CTA-pair kernel only: M > 128, beta = 0).  Passing both C and C16 returns DEER_ERR_UNSUPPORTED.
 *      All pointers 16-byte aligned; lda/ldb multiples of 8 elements, ldc a multiple of 4. */
int deer_gemm_h16(const void* A, long long lda, int transA, int a_bf16, const void* B, long long ldb, int transB,
                  int b_bf16, float* C, long long ldc, void* C16, long long ldc16, int c16_bf16, int M, int N, int K,
                  const float* bias, int act, float beta, void* stream);
/*      debugging aid: >= 8 int64 device counters (block 0): cycles waiting on empty / tmem_empty / full / tmem_full and
 *      cycles spent in the epilogue (NULL disables) */
int deer_gemm_h16_set_profile_buffer(long long* device_buf);
/*      fp32 [rows, cols] (pitch ld_src) -> 16-bit [rows, cols_pad] (pitch ld_dst), columns >= cols zero-filled */
int deer_cast16(const float* src, long long ld_src, void* dst, long long ld_dst, long long rows, int cols, int cols_pad,
                int bf16, void* stream);

/* ---- activation backward + bias gradient (autograd of the Linear+act blocks above).
 *      dz = dy * act'(y) (dz may alias dy; dz may be NULL when act==NONE); dbias[n] += sum_m dz[m,n] if dbias. */
int deer_bias_act_bwd(const float* dy, long long ld_dy, const float* y, long long ld_y, float* dz, long long ld_dz,
                      float* dbias, int M, int N, int act, void* stream);

/* ---- nn.LayerNorm (encoders.py:106,474,624; fusion.py:102,218,303; complete_project.py:70,88,329,340) */
int deer_layernorm_fwd(const float* x, const float* gamma, const float* beta, float* y, float* mean, float* rstd,
                       int M, int N, float eps, void* stream);
int deer_layernorm_bwd(const float* dy, const float* x, const float* gamma, const float* mean, const float* rstd,
                       float* dx, float* dgamma, float* dbeta, int M, int N, void* stream);

/* ---- nn.Dropout with a counter-based generator (Philox-4x32-10 keyed by seed, indexed by element).
 *      y = x * keep/(1-p); the same call regenerates the mask for backward. x may alias y.
 *      step_ptr (device, may be NULL): a 64-bit step counter mixed into the Philox counter so that a captured
 *      CUDA graph draws a fresh mask on every replay. */
int deer_dropout(const float* x, float* y, long long n, float p, unsigned long long seed, unsigned long long offset,
                 const unsigned long long* step_ptr, void* stream);
/*      the same mask (same seed / offset / step) applied while casting to the 16-bit GEMM operands of the next LSTM layer
 *      (nn.LSTM inter-layer dropout, encoders.py:82-89): y_fp16 and/or y_bf16 [n], n % 4 == 0; p == 0 is a plain cast */
/*      keep_mask (may be NULL; needs n % 128 == 0): uint32 [n/32], bit j of word w = element 32 w + j survived -- read
 *      back by deer_gemm_h16_dropmask in backward instead of a Philox pass over the input gradient */
int deer_dropout_cast16(const float* x, void* y_fp16, void* y_bf16, long long n, float p, unsigned long long seed,
                        unsigned long long offset, const unsigned long long* step_ptr, void* keep_mask, void* stream);

/* ---- attention pooling over time (encoders.py:93-98,383-384; :462-467,543-544; :597-602,738-746).
 *      rowdot: s[m] = sum_j h[m,j]*w[j] + b[0]   (the Linear(D/2 -> 1) scorer head) */
int deer_rowdot_fwd(const float* h, const float* w, const float* b, float* s, long long M, int N, void* stream);
int deer_rowdot_bwd(const float* ds, const float* h, const float* w, float* dh, float* dw, float* db,
                    long long M, int N, void* stream);
/*      backward of the whole scorer head s = w2 . tanh(z) + b2 in one pass over hidden = tanh(z) [M,N]:
 *      dz = ds w2 (1 - hidden^2) (may alias hidden), dw2 += sum_m ds hidden, db1 += sum_m dz, db2 += sum_m ds;
 *      dz_row_scale (may be NULL): the STORED row m of dz is multiplied by dz_row_scale[m] (premasked scorer input) */
int deer_scorer_bwd(const float* ds, const float* hidden, const float* w2, float* dz, float* dw2, float* db1, float* db2,
                    const float* dz_row_scale, long long M, int N, void* stream);
/*      pool: p = softmax_t(s[b,:]); if mask: p = p*mask / (sum_t p*mask + 1e-10); out[b,:] = sum_t p[b,t] * x[b,t,:]
 *      x element (b,t,d) at x[b*xs_b + t*xs_t + d]; s element (b,t) at s[b*ss_b + t*ss_t]; mask [B,T] contiguous or NULL;
 *      if premask, the pooled rows are mask[b,t] * x[b,t,:] (text path, encoders.py:733-735: the masked embeddings are
 *      never materialised; the scorer sees them through deer_cast_split16's row_scale). wts [B,T] out. */
int deer_attn_pool_fwd(const float* x, long long xs_b, long long xs_t, const float* s, long long ss_b, long long ss_t,
                       const float* mask, float* out, float* wts, int B, int T, int D, int premask, void* stream);
/*      dx (b,t,d) = wts*dout (same strides as x, overwritten or accumulated per `accumulate`; NULL when x needs no
 *      gradient: only ds is produced), ds (same strides as s) */
int deer_attn_pool_bwd(const float* dout, const float* x, long long xs_b, long long xs_t, const float* s, long long ss_b,
                       long long ss_t, const float* mask, const float* wts, float* dx, float* ds, int B, int T, int D,
                       int accumulate, int premask, void* stream);
/*      pooling over each sample's own frames t < L_b = clamp(lengths[b], 1, T) (lengths [B] int32 / int64 per lengths_i64,
 *      device memory): softmax and weighted sum over those only; padded rows of x and s are never read, wts is 0 there.
 *      Backward (wts as written by the forward): ds is 0 at padded rows, and dx (NULL: not produced) is OVERWRITTEN --
 *      w_t dout at valid rows, 0 at padded rows. */
int deer_attn_pool_len_fwd(const float* x, long long xs_b, long long xs_t, const float* s, long long ss_b, long long ss_t,
                           const void* lengths, int lengths_i64, float* out, float* wts, int B, int T, int D,
                           void* stream);
int deer_attn_pool_len_bwd(const float* dout, const float* x, long long xs_b, long long xs_t, long long ss_b,
                           long long ss_t, const void* lengths, int lengths_i64, const float* wts, float* dx, float* ds,
                           int B, int T, int D, void* stream);

/* ---- layout helpers */
/* y[t,b,:] = x[b,t,:] (batch-first -> time-major) and the inverse */
int deer_permute_bt(const float* x, float* y, int B, int T, int D, void* stream);
/*      [B,T,D] fp32 -> time-major 16-bit rows [T*B, Dp] (Dp >= D even, columns D.. zero): FP16 (y_fp16) and / or BF16 (y_bf16)
 *      copies in one pass -- the first nn.LSTM layer's projection operand and its weight-gradient operand
 *      (encoders.py:82-89,380: `self.lstm(enhanced_features)` on a batch_first input) */
int deer_permute_bt_cast16(const float* x, void* y_fp16, void* y_bf16, int B, int T, int D, int Dp, void* stream);
/*      the same with per-utterance lengths: rows of frames t >= clamp(lengths[b], 1, T) are written as zeros and their input
 *      is never read (NaN / Inf padding stays out of the LSTM projection and of dW_ih).  x is [B,T,D], or already
 *      time-major [T,B,D] when x_time_major != 0.  lengths [B] int32 / int64 (lengths_i64) in device memory. */
int deer_permute_bt_cast16_len(const float* x, void* y_fp16, void* y_bf16, const void* lengths, int lengths_i64, int B,
                               int T, int D, int Dp, int x_time_major, void* stream);
/* y[m,:] = x[m,:] * mask[m]  (text mask, encoders.py:734-735); backward is the same call on dy */
int deer_rowscale(const float* x, const float* mask, float* y, long long M, int D, void* stream);
/* Conv1d(k=3,pad=1) lowering on channels-last x [B,T,C]: col [B*T, 3C], tap k holds x[b,t+k-1,:] (zero outside) */
int deer_im2col3(const float* x, float* col, int B, int T, int C, void* stream);
int deer_col2im3(const float* dcol, float* dx, int B, int T, int C, void* stream);
/*      sliding-window form of the same convolution (no im2col matrix): padded copy
 *        xp = [lead zero rows][sample 0: T rows][zero row][sample 1: T rows][zero row]...[tail zero rows]   ([.,C], C % 4 == 0)
 *      with lead = 1 the rows of the k=3 im2col matrix are the OVERLAPPING windows xp[q .. q+3) (3C contiguous floats,
 *      row pitch C): deer_gemm accepts lda < K / ldb < N / ldc < N (with beta = 1: atomic accumulation) for such views.
 *      dir 0: x [B,T,C] -> xp;  dir 1: xp -> x (drops the pad rows). */
int deer_rows_pad(const float* src, float* dst, int B, int T, int C, int lead, int tail, int dir, void* stream);
/*      the same copy with the video encoder's neighbouring passes folded in (encoders.py:450-459, nn.Dropout -> nn.Conv1d):
 *      dir 0: optional inverted dropout of x (the Philox stream of deer_dropout over the flat index of x: identical masks),
 *      padded fp32 copy, and (hi / lo non-NULL, C % 8 == 0) its FP16 hi / lo split in the same geometry -- the A operand of
 *      deer_gemm_h16_split; dir 1: un-pad dx_p and apply the same mask (the backward of dropout o pad). */
int deer_rows_pad_fused(const float* src, float* dst, void* hi, void* lo, int B, int T, int C, int lead, int tail, int dir,
                        float drop_p, unsigned long long seed, unsigned long long offset, const unsigned long long* step_ptr,
                        void* stream);
/*      backward entry of the same convolution: dy [B,T,C] -> dy_big [B*(T+1), C] (a zero row behind every sample) and the
 *      bias gradient colsum[c] += sum over rows of dy[., c] (nn.Conv1d.bias, encoders.py:450-459) in ONE pass over dy */
int deer_rows_pad_colsum(const float* src, float* dst, float* colsum, int B, int T, int C, void* stream);
/* w [Cout,Cin,3] (nn.Conv1d layout) <-> wk [Cout,3,Cin]; dir=0 pack, dir=1 unpack with accumulate into w */
int deer_conv3_weight_pack(const float* w, float* wk, int Cout, int Cin, int dir, void* stream);

/* ---- nn.BatchNorm1d + ReLU on channels-last rows x [M,C] (encoders.py:452,457).
 *      training: batch statistics (biased variance) and running-stat update (momentum, unbiased variance);
 *      eval: running statistics.  stats [2,C] scratch (mean, biased var). */
int deer_bn_stats(const float* x, float* stats, long long M, int C, void* stream);
int deer_bn_update_running(const float* stats, float* running_mean, float* running_var,
                           long long* num_batches_tracked /* int64 counter or NULL */, long long M, int C,
                           float momentum, void* stream);
int deer_bn_relu_fwd(const float* x, const float* mean, const float* var, const float* gamma, const float* beta,
                     float* y, long long M, int C, float eps, void* stream);
/*      training-mode backward (through the batch statistics) when batch_stats!=0, else plain affine backward.
 *      scratch [2,C] floats, zeroed by the call. dgamma/dbeta accumulate. */
int deer_bn_relu_bwd(const float* dy, const float* x, const float* y, const float* mean, const float* var,
                     const float* gamma, float* dx, float* dgamma, float* dbeta, float* scratch, long long M, int C,
                     float eps, int batch_stats, void* stream);

/* ---- 2-token multi-head self attention core (fusion.py:293-298,328-332): qkv [B,2,3E] packed (q|k|v) after in_proj,
 *      ctx [B,2,E] before out_proj, attw [B,2,2] head-averaged weights. */
/*      ctx_mean [B,E] = mean over the two tokens of ctx (fusion.py:335 commutes with the linear out_proj); either of
 *      ctx / ctx_mean may be NULL.  Backward takes the matching upstream gradients (either may be NULL). */
int deer_mha2_fwd(const float* qkv, float* ctx, float* ctx_mean, float* attw, float* probs, int B, int E, int heads,
                  void* stream);
int deer_mha2_bwd(const float* dctx, const float* dctx_mean, const float* dattw, const float* qkv, const float* probs,
                  float* dqkv, int B, int E, int heads, void* stream);

/* ---- bidirectional LSTM layer recurrence (encoders.py:82-89,380), time-major.
 *      gates [T,B,2,4H]: on entry the input projection x_t W_ih^T + b_ih + b_hh for both directions (dir 0 forward in
 *      time, dir 1 reverse), on exit the post-activation gates i,f,g,o (kept for backward).
 *      w_hh_fwd / w_hh_rev [4H,H] each (weight_hh_l{k}, weight_hh_l{k}_reverse); h_out [T,B,2H] (dir 0 in [0,H), dir 1 in [H,2H)); c_out [T,B,2,H] cell states or NULL
 *      (inference: not kept; c_work [B,2,H] scratch then required). */
int deer_lstm_fwd(float* gates, const float* w_hh_fwd, const float* w_hh_rev, float* h_out, float* c_out, float* c_work,
                  int T, int B, int H, int engine, void* stream);
/*      backward: dh_out [T,B,2H] upstream gradient; gates (post-activation) is overwritten by the pre-activation
 *      gradients dgates [T,B,2,4H]; dh_work,dc_work [B,2,H] scratch. dW_hh, dW_ih, db and dx are then plain GEMMs /
 *      column sums over dgates done by the caller. */
int deer_lstm_bwd(float* gates, const float* w_hh_fwd, const float* w_hh_rev, const float* c_all, const float* dh_out,
                  float* dh_work, float* dc_work, int T, int B, int H, int engine, void* stream);

/* ---- persistent cluster kernels for the same layer (production path, H == 256; csrc/lstm_cluster.cu).
 *      Layouts: pre_il / dpre_il are GATE-INTERLEAVED [T,B,2,H,4] (column 4*unit+gate): run the input projection with
 *      row-interleaved W_ih and bias (deer_gate_rows_interleave), and un-interleave the weight gradients computed from
 *      dpre_il.  gact (activated gates) and c_blk (cell states) are opaque workspaces private to the fwd/bwd pair:
 *      T*2*Bp*4H and T*2*Bp*H ELEMENTS with Bp = B rounded up to a multiple of 32 -- FP16 elements by default, fp32 with
 *      DEER_OPT_LSTM_KEEP16 = 0; NULL for inference.
 *      db_il [2,H,4] accumulates (atomics) the bias gradient = column sums of dpre_il; may be NULL. */
int deer_lstm_cluster_tile(int B);  /* batch columns per 4-CTA cluster the kernels will use for batch B (16 or 32) */
/*      h_f16 / h_bf16 (forward) and dpre_bf16 (backward): optional 16-bit shadow copies of h [T,B,2H] and dpre_il
 *      [T,B,2,H,4] written by the same kernels as operands for deer_gemm_h16 (NULL to skip). */
int deer_lstm_cluster_fwd(const float* pre_il, const float* w_hh_fwd, const float* w_hh_rev, float* h_out, void* gact,
                          void* c_blk, void* h_f16, void* h_bf16, int T, int B, int H, void* stream);
/*      the same forward reading FP16 pre-activations [T,B,2,H,4] (deer_gemm_h16 with a 16-bit output) */
int deer_lstm_cluster_fwd_pre16(const void* pre_il_f16, const float* w_hh_fwd, const float* w_hh_rev, float* h_out,
                                void* gact, void* c_blk, void* h_f16, void* h_bf16, int T, int B, int H,
                                void* stream);
/*      forward recurrence WITH the layer's input projection inside (first nn.LSTM layer, encoders.py:82-89,380: In = 84):
 *      gates_t = W_ih x_t + (b_ih + b_hh) + W_hh h_{t-1}.  x_f16: time-major FP16 rows [T*B, xk] (xk % 8 == 0, xk <= 128, zero
 *      padded: deer_permute_bt_cast16); w_ih_il_f16 [2*4H, xk]: both directions' gate-interleaved FP16 W_ih and bias_il
 *      [2*4H] their gate-interleaved b_ih + b_hh (deer_lstm_prep).  Each CTA keeps its 256 rows of W_ih in TMEM beside W_hh and
 *      issues W_ih x_t one step ahead into double-buffered TMEM accumulators, so the [T,B,2,4H] pre-activation tensor (a
 *      315 MB write + read per layer at B = 256) never exists.  deer_lstm_cluster_xin_mode: 0 = no such variant for this
 *      batch / keep / xk (training batches beyond one wave of 16-column tiles, B > 256: use the projection GEMM +
 *      deer_lstm_cluster_fwd_pre16), 1 = 16-column tiles, 2 = the no-keep dual-sub-tile kernel with one MMA warp per sub-tile.
 *      Outputs as deer_lstm_cluster_fwd. */
int deer_lstm_cluster_xin_mode(int B, int keep, int xk);
int deer_lstm_cluster_fwd_xin(const void* x_f16, int xk, const void* w_ih_il_f16, const float* bias_il, const float* w_hh_fwd,
                              const float* w_hh_rev, float* h_out, void* gact, void* c_blk, void* h_f16, void* h_bf16, int T,
                              int B, int H, void* stream);

/*      dpre_il (fp32) may be NULL when dpre_bf16 is given: only the 16-bit gradient is written */
int deer_lstm_cluster_bwd(const void* gact, const void* c_blk, const float* dh_out, const float* w_hh_fwd,
                          const float* w_hh_rev, float* dpre_il, float* db_il, void* dpre_bf16, int T, int B, int H,
                          void* stream);
/*      one-pass operand preparation of an LSTM layer for the cluster kernels + 16-bit GEMM: W_ih of both directions
 *      (nn.LSTM order, fp32 [4H,In]) -> gate-interleaved FP16/BF16 [2*4H, Kp] (Kp >= In even, zero-padded), and (b_il may
 *      be NULL) b_ih + b_hh -> gate-interleaved fp32 [2*4H];  and the reverse for the gradients: gate-interleaved
 *      dW_ih [2,4H,In], dW_hh [2,4H,H], db [2,4H] accumulated (+=) into the eight natural-order targets. */
int deer_lstm_prep(const float* w_ih_fwd, const float* w_ih_rev, const float* b_ih_fwd, const float* b_hh_fwd,
                   const float* b_ih_rev, const float* b_hh_rev, void* w16, float* b_il, int H, int In, int Kp, int bf16,
                   void* stream);
int deer_lstm_unprep(const float* dwi_il, const float* dwh_il, const float* db_il, float* dw_ih_fwd, float* dw_ih_rev,
                     float* dw_hh_fwd, float* dw_hh_rev, float* db_ih_fwd, float* db_hh_fwd, float* db_ih_rev,
                     float* db_hh_rev, int H, int In, void* stream);
/*      rows g*H+u of src [4H,K] -> rows 4u+g of dst (inverse=0) or back (inverse=1); accumulate!=0 adds into dst */
int deer_gate_rows_interleave(const float* src, float* dst, int H, int K, int inverse, int accumulate, void* stream);
/*      per-utterance lengths (nn.LSTM on pack_padded_sequence(x, lengths, batch_first=True, enforce_sorted=False)) on the
 *      unchanged cluster kernels: between the input projection and the forward recurrence, the i, f and o gates of every
 *      padded row t >= L_b of pre_il [T,B,2,H,4] (FP16 if pre_fp16, else fp32; 16-byte aligned) are set to -65504.  The
 *      kernels' sigmoid then gives 2^-60: the state is ~0 at every padded step (the reverse direction starts at L_b - 1 from
 *      zero, padded outputs <= 2^-83 ~ 1e-25), and with FP16 kept state (DEER_OPT_LSTM_KEEP16 = 1) BPTT produces dpre = 0 exactly
 *      there, provided dh_out is finite at padded rows.  lengths [B] int32 (lengths_i64 = 0) or int64 (1), device memory,
 *      clamped to [1, T] by the kernel.  Work scales with the number of padded rows. */
int deer_lstm_mask_pre(void* pre_il, int pre_fp16, const void* lengths, int lengths_i64, int T, int B, int H,
                       void* stream);

/* ---- NIG head transform (deer.py:90-98; complete_project.py:399-407). evidence [N,4] -> 7 arrays [N] */
int deer_nig_head_fwd(const float* evidence, float* mu, float* nu, float* alpha, float* beta, float* aleatoric,
                      float* epistemic, float* total, long long N, void* stream);
int deer_nig_head_bwd(const float* evidence, const float* dmu, const float* dnu, const float* dalpha,
                      const float* dbeta, const float* daleatoric, const float* depistemic, const float* dtotal,
                      float* devidence, long long N, void* stream);

/* ---- DEER loss (losses.py:72-348): two phases so the ECE bin statistics and batch means are exact.
 *      Inputs either raw evidence [B,D,4] (from_evidence=1: the softplus head is fused) or the four NIG arrays [B,D].
 *      stats [D, DEER_LOSS_NSTAT] must be zero on entry of phase 1; between the phases a data-parallel caller may
 *      all-reduce `stats` (sum) and pass the GLOBAL batch size to phase 2 for exact global-batch semantics.
 *      phase 2 writes losses[D*5+2] = per dim (total,nll,reg,kl,ece), cross_dim, total and the gradient
 *      (d total / d evidence [B,D,4], or d/d(gamma,nu,alpha,beta) [B,D] x4) scaled by grad_scale. */
#define DEER_LOSS_NSTAT 40
int deer_nig_loss_stats(const float* evidence, const float* gamma, const float* nu, const float* alpha,
                        const float* beta, const float* targets, const float* bin_edges, float* stats,
                        float* nig_out /* [7,B,D] or NULL */, long long B, int D, int from_evidence, float eps,
                        void* stream);
int deer_nig_loss_finish(const float* evidence, const float* gamma, const float* nu, const float* alpha,
                         const float* beta, const float* targets, const float* bin_edges, const float* stats,
                         const float* task_weights /* [D] or NULL */, float reg_w, float kl_w, float ece_w,
                         float cross_w, float eps, long long B_local, long long B_global, int D, int from_evidence,
                         float grad_scale, float* losses, float* d_out /* [B,D,4] */, void* stream);
/*      Amini-style variant, deer.py:111-195 (L3): stats-free single pass + mean; losses[5] */
int deer_amini_loss(const float* mu, const float* nu, const float* alpha, const float* beta, const float* targets,
                    float evidence_w, float kl_w, long long N, float* losses, float* dparams /* [4,N] or NULL */,
                    float* scratch /* [8] zeroed by call */, void* stream);

/* ---- trainer step (training.py:121-150,219,224): global grad norm, clip, AdamW over flat buffers */
int deer_sumsq(const float* x, long long n, float* out /* accumulates */, void* stream);
/*      clip coefficient = min(1, max_norm / (sqrt(*sumsq * inv_world^2...) + 1e-6)) computed on device from *sumsq */
/*      step_dev (device int64, may be NULL): when given the update uses step = *step_dev + 1 and `step` is ignored;
 *      lr_dev (device float, may be NULL): when given the learning rate is lr * *lr_dev.  Both exist so that a
 *      CUDA-graph capture of the training step stays valid across steps and LR-schedule changes. */
/* x[0..n) = 0 and (y non-NULL) y[0..ny) = 0: the once-per-step clear of the flat gradient buffer and of the
 * gradient-norm accumulator (replaces optimizer.zero_grad(), training.py:215); step_increment: *step += 1 on the device
 * (graph-replayable step counter read by deer_adamw and the dropout kernels) */
int deer_fill_zero(float* x, long long n, float* y, long long ny, void* stream);
int deer_step_increment(long long* step, void* stream);
int deer_adamw(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1, float beta2,
               float eps, float weight_decay, int step, const float* sumsq, float max_norm, float grad_scale,
               const long long* step_dev, const float* lr_dev, void* stream);

/* ---- C = opA(A) opB(B) + w (x) v per sample: the TF32 CTA-pair GEMM (M > 256, N >= 128, N % 4 == 0, K >= 64; beta = 0) with a
 * rank-1-per-sample row term in its epilogue: row m of C is sample b, step t of an [nb, nt] (batch-major) or [nt, nb]
 * (time_major) grid and receives w[b, t] * v[b, :] (w [nb, nt], v [nb, N]).  Replaces the pair "attention pooling writes its
 * input gradient, the scorer's input-gradient GEMM accumulates onto it" (encoders.py:93-98,383-384 in backward): dx is written
 * once instead of written, read and written. */
int deer_gemm_rowterm(const float* A, long long lda, int transA, const float* B, long long ldb, int transB, float* C,
                      long long ldc, int M, int N, int K, const float* w, const float* v, int nb, int nt, int time_major,
                      void* stream);

/* ---- C = dropout'(A B): the 16-bit GEMM (CTA-pair kernel: M > 128, N % 32 == 0, fp32 C, beta = 0) whose epilogue applies
 * the keep mask of an inverted dropout over C (deer_dropout_cast16's keep_mask, row pitch N/32 words) and its 1/(1-p)
 * scale: nn.LSTM's inter-layer dropout in backward (encoders.py:82-89) -- dx of layer l+1 is masked while it is written,
 * instead of a read-modify-write pass over [T*B, 2H] fp32. */
int deer_gemm_h16_dropmask(const void* A, long long lda, int transA, int a_bf16, const void* B, long long ldb, int transB,
                           int b_bf16, float* C, long long ldc, int M, int N, int K, const void* keep_mask, float scale,
                           void* stream);

/* ---- split-precision GEMM of the time-batched FORWARD contractions (scorers encoders.py:93-98,462-467,597-602, video
 * spatial_projection :443-447, Conv1d taps :450-459): every fp32 operand travels as a pair of FP16 matrices
 * x = hi + lo (deer_cast_split16: hi = fp16(x), lo = fp16(x - hi), 22 significant bits) and the CTA-pair tcgen05 kernel makes
 * three passes over K accumulating A_hi B_hi + A_lo B_hi + A_hi B_lo in its fp32 TMEM accumulator: fp32-grade products
 * at the cost of a TF32 GEMM (3 MMAs at twice the tensor rate).  Why: a TF32 forward (2^-11 operand rounding) perturbs
 * the encoder outputs by ~3e-4, which flips ~1e-4 of the downstream ReLU masks and costs the GRADIENT ~4e-2 relative
 * (cosine 0.998 per tensor); the backward contractions themselves are insensitive and stay on TF32 / BF16.
 *   C = act(opA(A) opB(B) + bias), fp32 out, beta = 0; M > 128, even N; lda < K (overlapping rows) allowed. */
int deer_gemm_h16_split(const void* A_hi, const void* A_lo, long long lda, int transA, const void* B_hi, const void* B_lo,
                        long long ldb, int transB, float* C, long long ldc, int M, int N, int K, const float* bias, int act,
                        void* stream);
/*   row_scale (may be NULL): row r of src is multiplied by row_scale[r] before the split -- the text encoder's
 *   `token_embeddings * attention_mask` (encoders.py:733-735) without materialising the masked copy */
int deer_cast_split16(const float* src, long long ld_src, const float* row_scale, void* hi, void* lo, long long ld_dst,
                      long long rows, int cols, int cols_pad, void* stream);

/* ---- fused 3xTF32 GEMM of the post-pooling chain: replaces the addmm + relu + dropout (+ their backward:
 * threshold_backward, dropout mask multiply, bias-gradient sum) ATen calls of nn.Linear / nn.ReLU / nn.Dropout stacks in
 * fusion.py:188-343 (AudioVisualFusion / TrimodalFusion / output_projection), deer.py:30-108,198-266 (DEERLayer,
 * MultiDimensionalDEER), encoders.py:101-107,470-475,608-625 (output projections) and complete_project.py:61-588.
 *   C[b] = dropout( act( opA(A_eff[b]) opB(B[b]) + bias[b] + beta*C[b] ) ),   A_eff = A (.) gatefn(gate)
 * gate (optional, same layout as A with leading dimension ldgate): gate_mode 1 = (gate > 0 ? gate_scale : 0) -- the
 * backward of ReLU (+ inverted dropout, gate_scale = 1/(1-p)) from the layer's saved output; 2 = (1-gate^2)*gate_scale
 * (tanh'); 3 = gate(1-gate)*gate_scale (sigmoid').  colsum (optional, transA only): colsum[b][m] += sum_k A_eff[k,m],
 * the bias gradient of dW = dz^T x.  Dropout: inverted, Philox stream of deer_dropout keyed by (seed, *drop_step) over the
 * flat index row*drop_ld + b*drop_batch_stride + drop_col0 + col (drop_ld = 0 means ldc).  batch > 1: operand b at pointer + b*stride. */
typedef struct {
  const float* A; const float* B; float* C; const float* bias; const float* gate; float* colsum;
  const unsigned long long* drop_step;
  long long lda, ldb, ldc, ldgate;
  long long sA, sB, sC, sBias, sGate, sColsum;
  unsigned long long drop_seed, drop_offset;
  long long drop_ld, drop_batch_stride;
  int drop_col0;
  int M, N, K, batch;
  int transA, transB, act;
  float beta, drop_p;
  int gate_mode;
  float gate_scale;
  int splitk;   /* internal (cross-CTA split-K factor chosen by the dispatcher); ignored on input */
} deer_gemm_x3_args;
int deer_gemm_x3(const deer_gemm_x3_args* args, void* stream);

/* ---- persistent chain kernel: the whole post-pooling part of a step (HierarchicalMultimodalFusion.forward
 * fusion.py:119-171 with AudioVisualFusion :188-271 and TrimodalFusion :274-343, then MultiDimensionalDEER.forward
 * deer.py:233-266; and their autograd) as ONE launch per direction.  The caller passes a PROGRAM: ops grouped into
 * dependency levels; one CTA per SM deals the tiles of a level round-robin and a grid-wide barrier separates levels.
 * Op kinds: 0 GEMM (`g` = deer_gemm_x3 arguments, 32x32 tiles: tiles = ceil(M/32)*ceil(N/32)*batch; operands 16-byte
 * aligned, pitches multiples of 4); 1 LayerNorm forward (g.A = x, g.B = gamma, g.bias = beta, g.C = y, g.gate = mean out,
 * g.colsum = rstd out, g.beta = eps; tiles = ceil(M/8)); 2 LayerNorm backward (g.A = dy, g.B = x, g.bias = gamma,
 * g.gate = mean, g.colsum = rstd, g.C = dx (g.beta = 1: +=), dgamma / dbeta accumulators as pointers in g.drop_seed /
 * g.drop_offset; tiles = ceil(M/32)); 3 / 4 two-token attention core forward / backward (see csrc/chain.cu; g.N = E,
 * g.K = heads; tiles = M); 5 y (+)= x (g.A, g.C, g.beta; tiles = ceil(M/32)).  `barrier`: a zero-initialised device
 * counter; `error` (optional): set to 1 by the device-side watchdog if a barrier times out. */
#define DEER_CHAIN_MAX_OPS 72
#define DEER_CHAIN_MAX_LEVELS 48
typedef struct {
  int kind, tiles, tiles_n, pad_;
  deer_gemm_x3_args g;
} deer_chain_op;
typedef struct {
  int nops, nlevels;
  unsigned int* barrier;
  int* error;
  int level_begin[DEER_CHAIN_MAX_LEVELS + 1];
  deer_chain_op ops[DEER_CHAIN_MAX_OPS];
} deer_chain_program;
int deer_chain_run(const deer_chain_program* program, void* stream);
int deer_chain_max_ops(void);
int deer_chain_max_levels(void);

/* ---- generic elementwise helpers used by the pooled model (complete_project.py:282-293,364,439-459) */
/* y = a*x1 + b*x2 (x2 may be NULL) */
int deer_axpby(const float* x1, const float* x2, float* y, long long n, float a, float b, void* stream);
/* out[m,:] = w[m*ldw]*s[m,:] + (1-u[m*ldu])*c[m,:]   and its backward */
int deer_mix_fwd(const float* w, long long ldw, const float* u, long long ldu, const float* s, const float* c, float* out,
                 long long M, int N, void* stream);
int deer_mix_bwd(const float* dout, const float* w, long long ldw, const float* u, long long ldu, const float* s,
                 const float* c, float* dw, long long lddw, float* du, long long lddu, float* ds, float* dc, long long M,
                 int N, void* stream);
/* out = g*a + (1-g)*b and backward */
int deer_gate_fwd(const float* g, const float* a, const float* b, float* out, long long n, void* stream);
int deer_gate_bwd(const float* dout, const float* g, const float* a, const float* b, float* dg, float* da, float* db,
                  long long n, void* stream);
/* y[m,n] = x[m,n] / t[n] (temperature scaling, complete_project.py:449); backward: dx = dy/t, dt[n] += -sum_m dy x / t^2 */
int deer_coldiv_fwd(const float* x, const float* t, float* y, long long M, int N, void* stream);
int deer_coldiv_bwd(const float* dy, const float* x, const float* t, float* dx, float* dt /* accumulates, may be NULL */,
                    long long M, int N, void* stream);
/* row softmax over N<=32 columns and backward */
int deer_softmax_rows_fwd(const float* x, float* y, long long M, int N, void* stream);
int deer_softmax_rows_bwd(const float* dy, const float* y, float* dx, long long M, int N, void* stream);

/* ---- text-side integer features: EnhancedTextEncoder.extract_linguistic_features (encoders.py:648-699).
 *      input_ids / attention_mask [B,T] int64 (a token is valid when its mask is non-zero), features [B,10] fp32:
 *      {n/max_length, unique/n, n/(max id + 1), max multiplicity, frac ids in [999,1030], frac ids in [100,999], 0,0,0,0};
 *      all-zero row for a sample with no valid token.  Replaces the reference's O(B) Python loop; bit-exact. T <= 1024. */
int deer_linguistic_features(const long long* input_ids, const long long* attention_mask, float* features, int B, int T,
                             int max_length, void* stream);

/* ---- validation metrics (src/utils/metrics.py), device-side reductions
 *      moments[d][8] (fp64, zeroed by the call) = {n, sum t, sum p, sum t^2, sum p^2, sum t*p, sum |t-p|, sum (t-p)^2}
 *      over the rows where neither value is NaN; CCC (:59-103), MAE (:105-114), RMSE (:116-125) and Cohen's d
 *      (:190-211) are closed forms of these. pred/target contiguous [N,D], D in {1,2,3,4,6,8}. */
#define DEER_METRICS_NMOM 8
int deer_metrics_moments(const float* pred, const float* target, long long N, int D, double* moments, void* stream);
/*      uncertainty_calibration_error (:214-279) in three device stages; the host only turns 2*(n_bins+1) order
 *      statistics into quantile edges (numpy's linear interpolation) and the bin sums into the final scalar.
 *      prepare: err_mean[b] = mean_d |pred-target|, keys[b] = order-preserving code of mean_d uncert (0xffffffff for a
 *               dropped sample: NaN error, NaN/inf uncertainty, :245), *n_valid = kept samples (zeroed by the call)
 *      select : values[r] = the ranks_host[r]-th smallest kept uncertainty mean (0-based, exact; 8-bit radix select,
 *               4 passes over `keys`); ranks_host is a HOST array, R <= DEER_UCE_MAX_RANKS
 *      bins   : bin_sums[3][n_bins] (fp64, zeroed by the call) = {count, sum (1-u), sum (1-err)} over edges[j] <= u <
 *               edges[j+1]; edges is a DEVICE array of n_bins+1 fp64 */
#define DEER_UCE_MAX_RANKS 24
#define DEER_UCE_MAX_BINS 64
#define DEER_UCE_WORKSPACE_BYTES 65536
int deer_uce_prepare(const float* pred, const float* target, const float* uncert, long long N, int D, float* err_mean,
                     unsigned* keys, unsigned long long* n_valid, void* stream);
int deer_uce_select(const unsigned* keys, long long N, const long long* ranks_host, int R, float* values,
                    void* workspace, long long workspace_bytes, void* stream);
int deer_uce_bins(const unsigned* keys, const float* err_mean, long long N, int n_bins, const double* edges,
                  double* bin_sums, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DEER_B200_H */
