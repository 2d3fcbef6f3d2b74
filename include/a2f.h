/*
 * a2f.h -- C-ABI of liba2f_sm100.so: the B200 (sm_100a) audio->mesh hot path of
 * xtliu97/audio2face-pytorch (reference checked out at /root/reference, cited below as ref:<file>:<line>).
 *
 * The reference has no FFI layer: its boundary is the Python nn.Module contract of
 * ref:src/model/lightning_model.py:50-73,111-117 (get_model / forward(x, one_hot, template)).  The drop-in
 * Python modules of this repo (audio2face-pytorch_b200/modules.py) keep that contract and call the entry points
 * below through ctypes; INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer owned by the caller (PyTorch allocates), unless the name ends in _host;
 *  - nothing is allocated or freed inside the library; scratch space is passed in as `workspace`
 *    (size from the matching *_workspace_bytes call);
 *  - every call is asynchronous on `stream` (a cudaStream_t passed as void*; NULL = legacy default stream);
 *  - return value: A2F_OK or a negative a2f status; a2f_last_error() gives the message of the calling thread;
 *  - there is NO CPU fallback: on a device that is not sm_100 every compute call returns A2F_EARCH.
 *  - matrices are row-major; "[N,K]" weights are exactly torch's nn.Linear.weight layout.
 */
#ifndef A2F_H_
#define A2F_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define A2F_VERSION 100

#define A2F_OK 0
#define A2F_EINVAL (-1) /* bad shape / alignment / argument */
#define A2F_EARCH (-2)  /* device is not sm_100 */
#define A2F_ECUDA (-3)  /* CUDA runtime error, message kept in a2f_last_error() */

#define A2F_F32 0
#define A2F_BF16 1
#define A2F_I16 2   /* int16 PCM: a2f_audio_fragments input only */

#define A2F_ACT_NONE 0
#define A2F_ACT_RELU 1
#define A2F_ACT_GELU 2 /* exact erf GELU (HF activations "gelu" == torch F.gelu) */
#define A2F_ACT_TANH 3

#define A2F_BACKEND_SIMT_F32 0 /* true fp32 FMA path: the 1e-5 parity path */
#define A2F_BACKEND_TCGEN05 1  /* bf16 operands via TMA, fp32 accumulate in TMEM */

int a2f_version(void);
const char* a2f_status_string(int status);
const char* a2f_last_error(void);
/* A2F_OK when the current CUDA device is compute capability 10.x, else A2F_EARCH / A2F_ECUDA. */
int a2f_device_check(void);
/* number of kernels this library has launched from the calling process since load (bench.py's gpu_launches). */
long long a2f_launch_count(void);

/* ------------------------------------------------------------------------------------------------------------
 * Generic fused GEMM:  C[m,n] = act( sum_k A[m,k] * W[n,k] + bias[n] ) + resid[m,n] + tmpl[m / rows_per_tmpl, n]
 * Replaces every nn.Linear / F.linear on the path (ref:src/model/voca.py:30-36, ref:src/model/audio2face.py:49-55,
 * ref:src/model/faceformer.py:112,129, HF modeling_wav2vec2.py:422-434,466-573) and, through the A-row addressing
 * below, the stride-2 Conv1d stack of the wav2vec2 feature encoder as an implicit GEMM
 * (HF modeling_wav2vec2.py:254-272) with activations kept channels-last.
 *
 * A-row addressing: logical row m -> (b, r) = (m / rows_per_batch, m % rows_per_batch);
 *   element (m,k) lives at A + b*a_batch_stride + r*a_row_stride + k   (strides in elements).
 *   Plain matrix: rows_per_batch = M, a_row_stride = lda.  Conv1d(k taps, stride s) over channels-last [B,L,C]:
 *   K = k*C, a_row_stride = s*C, a_batch_stride = L*C, rows_per_batch = L_out  (rows overlap, nothing is copied).
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct a2f_gemm_args {
    int M, N, K;
    const void* A;
    int a_dtype; /* A2F_F32 (SIMT backend) or A2F_BF16 (either backend) */
    long long a_row_stride, a_batch_stride;
    int rows_per_batch;
    const void* W; /* [N,K], same dtype as A */
    long long ldw;
    const float* bias; /* [N] or NULL */
    int act;
    const void* resid; /* [M,N] added after the activation, or NULL */
    int resid_dtype;
    long long ldr;
    const float* tmpl; /* [ceil(M/rows_per_tmpl), N] fp32 added last (template mesh), or NULL */
    int rows_per_tmpl;
    void* C;
    int c_dtype;
    long long ldc;
    long long c_batch_stride; /* elements between the output blocks of consecutive batches; 0 = dense
                                 (rows_per_batch*ldc).  Lets a conv layer write straight into the zero-padded
                                 layout its successor reads (Audio2Mesh). */
    /* ---- backward-pass extensions (all zero = forward behaviour) ---- */
    int a_rows;               /* rows that exist in A per batch (0 = rows_per_batch); a logical row that maps outside
                                 [0, a_rows) reads as zeros */
    int n_seg;                /* 0/1: K is one run per row.  2..4: K = n_seg runs of K/n_seg elements; run s of logical
                                 row r is A[b, r + seg_row_off[s], seg_col_off[s] .. +K/n_seg).  The data gradient of a
                                 stride-2 Conv1d gathers its taps this way (no col2im scatter). */
    int seg_row_off[4];
    int seg_col_off[4];
    long long r_batch_stride; /* elements between the resid blocks of consecutive batches (0 = rows_per_batch*ldr) */
    int resid_mode;           /* A2F_RESID_ADD (default), or A2F_RESID_DACT: resid holds the forward PRE-activation z and
                                 the result is multiplied by act'(z) (act = the forward activation; bias is ignored):
                                 fuses the activation backward into the data-gradient GEMM */
    void* C2;                 /* optional second output (tcgen05 CTA-pair kernel, 16-byte aligned bf16/fp32 like C, no resid / tmpl):
                               * C receives the PRE-activation z = A W^T + bias, C2 receives act(z) -- the forward of a training
                               * step keeps z for the activation backward and feeds act(z) to the next GEMM, in one pass */
    long long ldc2;           /* row stride of C2 in elements (batch stride: c_batch_stride scaled by ldc2 / ldc) */
} a2f_gemm_args;

#define A2F_RESID_ADD 0
#define A2F_RESID_DACT 1

int a2f_gemm(const a2f_gemm_args* args, int backend, void* stream);

/* Weight gradient:  dW[n, s*K + k] += sum_m dY[m, n] * X[m -> (b, r + x_row_off[s]), x_col_off[s] + k],  s < n_seg
 * (the transposed-operand GEMM of every nn.Linear / Conv1d backward on the path; rows of X outside [0, x_rows) read as
 * zero).  dY: [M, N] rows addressed like A above; X likewise; dW: fp32 [N, n_seg*K] with row stride ldw, ACCUMULATED
 * into (callers zero it once per step: it is the .grad buffer).  tcgen05 backend: bf16 dY / X read in place through
 * MN-major UMMA descriptors (no transposed copies), split-K over the CTAs, fp32 TMA reduce-add into dW.
 * SIMT backend: fp32 or bf16 operands, fp32 atomics. */
typedef struct a2f_wgrad_args {
    int M, N, K;
    int dtype; /* of dY and X */
    const void* dY;
    long long dy_row_stride, dy_batch_stride;
    const void* X;
    long long x_row_stride, x_batch_stride;
    int rows_per_batch; /* logical rows (of dY) per batch */
    int x_rows;         /* rows of X that exist per batch (0 = rows_per_batch).  All x_rows rows must be READABLE and
                           FINITE over the columns the segments touch: rows past rows_per_batch meet zero-filled dY rows
                           inside the MMA, and 0 * NaN = NaN.  (Stride-2 conv over an odd-length input: the last
                           2*C-wide row of the last batch runs C elements past the tensor -- keep one zeroed spare row.) */
    int n_seg;          /* 0/1 = one segment; 2..4 = table below; > 4 needs x_row_step (linear table) */
    int x_row_off[4];
    int x_col_off[4];
    float* dW;
    long long ldw;
    int x_row_step;     /* != 0: segment s reads rows r + x_row_off[0] + s*x_row_step, columns x_col_off[0].. (the 128
                           taps of the positional conv); the table entries 1..3 are ignored */
} a2f_wgrad_args;
int a2f_gemm_wgrad(const a2f_wgrad_args* args, int backend, void* stream);

/* GEMM with the post-LayerNorm of the wav2vec2 encoder layer fused into its epilogue (tcgen05 back end, bf16):
 *   out[m,:] = LayerNorm(A[m,:] W^T + bias + resid[m,:]) * gamma + beta          (eps inside the square root)
 * = `h = layer_norm(h + out_proj(attn))` and `h = final_layer_norm(h + output_dense(ffn))` of HF
 * modeling_wav2vec2.py:576-609, which ref:src/model/wav2vec.py:174-180 runs 12 times per forward.  One thread-block
 * cluster of N/256 CTA pairs holds a whole 256-row block; row statistics travel through distributed shared memory and
 * the pre-LayerNorm sum stays in tensor memory (fp32, never rounded).  A [M,K], W [N,K], resid / out [M,N] bf16 with row
 * strides lda / ldw / ldr / ldo (elements, multiples of 8); N in {256, 512, 768}; bias may be NULL.
 * pre_out (may be NULL): training -- also store the pre-LayerNorm sum (bf16 [M,N], row stride ldp), the input of
 * a2f_layernorm_bwd. */
int a2f_gemm_ln(const void* A, long long lda, const void* W, long long ldw, const float* bias, const void* resid,
                long long ldr, const float* gamma, const float* beta, float eps, void* out, long long ldo, void* pre_out,
                long long ldp, int M, int N, int K, void* stream);

/* Everything of a post-LN encoder layer that is local to a block of rows, in ONE kernel (tcgen05 back end, bf16;
 * HF modeling_wav2vec2.py:551-609 through ref:src/model/wav2vec.py:174-180):
 *   h1    = LayerNorm(h_in + att Wo^T + bo) * ln1_g + ln1_b          skipped when att == NULL (h1 is then an input)
 *   f     = gelu(h1 W1^T + b1)                                         scratch [M,F], stays in L2
 *   h_out = LayerNorm(h1 + f W2^T + b2) * ln2_g + ln2_b
 *   qkv   = h_out Wq^T + bq                                            the NEXT layer's in-projection; skipped when wq == NULL
 * so that an encoder layer is two launches: the attention and this.  Same cluster layout as a2f_gemm_ln (N/256 CTA
 * pairs per 256-row block); all GEMMs of a row block share one smem ring and the TMEM double buffer, phase outputs are
 * handed over inside the cluster through L2 with cluster-scope mbarriers.  Results are bit-identical to a2f_gemm_ln,
 * a2f_gemm (GELU), a2f_gemm_ln, a2f_gemm run one after the other.
 * All matrices bf16, row strides in elements (multiples of 8), bases 16-byte aligned; N in {256,512,768}; F in {N..4N};
 * NQ in {N,2N,3N}; gelu = the tanh form the bf16 back end uses everywhere.  h1, f, h_out must be distinct buffers. */
typedef struct a2f_encoder_block_args {
    int M, N, F;
    const void* att; long long ld_att;      /* [M,N] attention output (heads merged); NULL = no attention-output phase */
    const void* wo; long long ld_wo;        /* [N,N] */
    const float* bo;
    const void* h_in; long long ld_hin;     /* [M,N] layer input (residual of the attention block) */
    const float* ln1_g; const float* ln1_b;
    void* h1; long long ld_h1;              /* [M,N] out (in when att == NULL) */
    const void* w1; long long ld_w1;        /* [F,N] */
    const float* b1;
    void* f; long long ld_f;                /* [M,F] scratch */
    const void* w2; long long ld_w2;        /* [N,F] */
    const float* b2;
    const float* ln2_g; const float* ln2_b;
    void* h_out; long long ld_hout;         /* [M,N] out */
    const void* wq; long long ld_wq;        /* [NQ,N]; NULL = no in-projection phase */
    const float* bq;
    int NQ;
    void* qkv; long long ld_qkv;            /* [M,NQ] out */
    float eps;
} a2f_encoder_block_args;
int a2f_encoder_block(const a2f_encoder_block_args* args, void* stream);


/* ------------------------------------------------------------------------------------------------------------
 * wav2vec2 positional conv embedding (HF modeling_wav2vec2.py:326-379,690-693 via ref:src/model/wav2vec.py:174):
 *   out[b,t,:] = h[b,t,:] + gelu( grouped_conv1d_k128_pad64_g16(h)[b,t,:] + bias )      (last conv step dropped)
 * h, out: channels-last [B,T,768].  Wp: packed weight produced by a2f_pack_posconv_weight:
 *   SIMT backend     kpad = 48: fp32 [16 groups][48 out][128 taps][48 in]
 *   tcgen05 backend  kpad = 8:  bf16 [16 groups][128 taps][6 chunks][48 out][8 in] -- per tap the shared-memory image of
 *                    the UMMA B operand (K-major, no swizzle), streamed by 1-D bulk copies (csrc/posconv_tc.cu); bf16 in/out
 *   (kpad = 64, bf16 [16][48][128][64 zero-padded]: the generic-GEMM path kept behind a2f_debug_set_umma_field(9, 1))
 * ---------------------------------------------------------------------------------------------------------- */
int a2f_posconv(const void* h, int h_dtype, const void* Wp, const float* bias, void* out, int out_dtype, int B, int T,
                int backend, void* stream);
/* weight_norm fold g*v/||v|| (norm over dims (0,1) per tap; HF weight_norm(dim=2)) + regroup.
 * g: [128] (original0), v: [768,48,128] (original1) fp32.  out dtype fp32 (kpad=48) or bf16 (kpad=8 / 64). */
int a2f_pack_posconv_weight(const float* g, const float* v, void* out, int out_dtype, int kpad,
                            float* norm_scratch /* [128] device floats */, void* stream);
/* Conv1d weight [Cout,Cin,taps] fp32 -> implicit-GEMM W [Cout, taps*Cin] (k = tap*Cin + cin), fp32 or bf16 */
int a2f_pack_conv1d_weight(const float* w, void* out, int out_dtype, int cout, int cin, int taps, void* stream);
/* elementwise cast fp32 -> bf16 (n elements) */
int a2f_cast_f32_to_bf16(const float* in, void* out, long long n, void* stream);
int a2f_cast_bf16_to_f32(const void* in, float* out, long long n, void* stream);
/* Error-compensated split for the tensor-core vertex head (K11): fp32 [rows,K] (row stride ld_in) -> bf16 [rows,3K],
 * activations as [hi | lo | hi], weights (is_weight=1) as [hi | hi | lo], hi = bf16(x), lo = bf16(x - hi): one bf16
 * GEMM with K' = 3K then evaluates a*w to ~2^-16 relative error with fp32 accumulation. */
int a2f_split_bf16x3(const float* in, long long ld_in, void* out, long long rows, int K, int is_weight, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * wav2vec2 front end.
 *  a2f_audio_stats: per-utterance mean and 1/sqrt(var+1e-7) (population variance) of raw audio [B,N]
 *     (the Wav2Vec2Processor zero-mean/unit-variance step the reference runs in numpy on the host,
 *      ref:src/model/faceformer.py:142-144 -> HF feature_extraction_wav2vec2.py:78-98). stats: [B,2] fp32.
 *  a2f_conv0_gn_gelu: normalise + Conv1d(1->512,k10,s5,no bias) + GroupNorm(512 groups, eps 1e-5, affine) + GELU
 *     (HF modeling_wav2vec2.py:302-323).  out: channels-last [B,L0,512], L0 = (N-10)/5+1.
 *     workspace: a2f_conv0_workspace_bytes(B,N).
 *  a2f_interp_ln: linear_interpolation(align_corners=True) S->T frames (ref:src/model/wav2vec.py:76-84,126-128)
 *     followed by LayerNorm(C, eps) of the feature projection (HF modeling_wav2vec2.py:429-431).
 *     in [B,S,C] -> out [B,T,C].
 * ---------------------------------------------------------------------------------------------------------- */
int a2f_audio_stats(const float* audio, int B, long long N, float* stats, void* stream);
size_t a2f_conv0_workspace_bytes(int B, long long N);
int a2f_conv0_gn_gelu(const float* audio, const float* stats, const float* w /*[512,10]*/, const float* gamma,
                      const float* beta, void* out, int out_dtype, int B, long long N, void* workspace,
                      size_t workspace_bytes, void* stream);
/* a2f_audio_stats + a2f_conv0_gn_gelu from ONE pass over the raw audio (inference): the moments of the normalised audio follow
 * algebraically from raw lag sums / products and sum x, sum x^2 (fp64); stats_out [B,2] (mean, rstd) is WRITTEN.  One launch
 * and one pass less in the dependent chain in front of conv0. */
size_t a2f_conv0_auto_workspace_bytes(int B, long long N);
int a2f_conv0_gn_gelu_auto(const float* audio, float* stats_out, const float* w /*[512,10]*/, const float* gamma,
                           const float* beta, void* out, int out_dtype, int B, long long N, void* workspace,
                           size_t workspace_bytes, void* stream);
int a2f_interp_ln(const void* in, int in_dtype, const float* gamma, const float* beta, float eps, void* out,
                  int out_dtype, int B, int S, int T, int C, void* stream);
/* LayerNorm over the last dim (C <= 4096, C % 4 == 0): out = (x-mean)*rstd*gamma+beta, stats in fp32.
 * Optional second output out2 (e.g. fp32 master + bf16 GEMM operand in one pass). */
int a2f_layernorm(const void* x, int x_dtype, const float* gamma, const float* beta, float eps, void* out,
                  int out_dtype, void* out2, int out2_dtype, long long rows, int C, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Encoder self-attention (HF modeling_wav2vec2.py:438-549): softmax(Q K^T * scale) V, no mask, never
 * materialising the [T,T] probabilities.  qkv: [B,T,3*H*D] (q | k | v blocks, each head-major), out: [B,T,H*D].
 * D must be 64.  fp32 in/out -> SIMT fp32 kernel; bf16 in/out -> tensor-core kernel.
 * ---------------------------------------------------------------------------------------------------------- */
int a2f_mha_fwd(const void* qkv, void* out, int dtype, int B, int T, int H, int D, float scale, void* stream);
/* same, also writing the row log-sum-exp of the scaled scores, lse [B,H,T] fp32 (needed by the backward) */
int a2f_mha_fwd_lse(const void* qkv, void* out, float* lse, int dtype, int B, int T, int H, int D, float scale,
                    void* stream);
/* training forward: additionally out_f32 [B,T,H*D] (optional, bf16 path only) = the output BEFORE rounding to bf16.
 * The backward's delta_i = sum_d dO_id O_id term cancels against dO V^T to within the spread of the value rows; when
 * the tokens are nearly alike (random init, late layers) the bf16 rounding of O would dominate dQ / dK. */
int a2f_mha_fwd_train(const void* qkv, void* out, float* lse, float* out_f32, int dtype, int B, int T, int H, int D,
                      float scale, void* stream);
/* backward: dqkv [B,T,3*H*D] (dq | dk | dv) from dout [B,T,H*D]; the probabilities are recomputed from q, k and lse,
 * never stored.  workspace: B*H*T floats.  bf16: two mma.sync passes (query-major dQ, key-major dK/dV), no atomics. */
int a2f_mha_bwd(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv, int dtype, int B, int T,
                int H, int D, float scale, void* workspace, size_t workspace_bytes, void* stream);
/* same; out_f32 (optional) = a2f_mha_fwd_train's un-rounded output, used for delta instead of `out` */
int a2f_mha_bwd_train(const void* qkv, const void* out, const float* out_f32, const void* dout, const float* lse,
                      void* dqkv, int dtype, int B, int T, int H, int D, float scale, void* workspace,
                      size_t workspace_bytes, void* stream);
/* training with attention dropout (site 8 * layer + A2F_DROP_ATTN_PROB, see "Encoder dropout" below): out = (P o Z/(1-p)) V,
 * lse stays that of the undropped softmax; Z over the logical tensor [B, H, T, Tp], Tp = ceil(T/8)*8 (padding the key
 * axis keeps an 8-key group inside one query row).  The backward regenerates Z in registers (dV = (P o Z/(1-p))^T dO,
 * dP = (dO V^T) o Z/(1-p), dS = P o (dP - delta), delta = rowsum(dO o O) of the dropped O).  A NULL dropout pointer,
 * p == 0 or a NULL seed_offset_dev is the call without the suffix. */
struct a2f_dropout_args;
int a2f_mha_fwd_train_dropout(const void* qkv, void* out, float* lse, float* out_f32, int dtype, int B, int T, int H, int D,
                              float scale, const struct a2f_dropout_args* dropout, void* stream);
int a2f_mha_bwd_train_dropout(const void* qkv, const void* out, const float* out_f32, const void* dout, const float* lse,
                              void* dqkv, int dtype, int B, int T, int H, int D, float scale,
                              const struct a2f_dropout_args* dropout, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * FaceFormer autoregressive decoder (ref:src/model/faceformer.py:154-185; torch nn.TransformerDecoderLayer
 * post-norm, d=64, 4 heads, ffn 128) as ONE persistent kernel, one CTA per utterance, KV-cached O(T) decode:
 *   e_0 = style;  d_i = DecLayer(PPE(e_0..e_i), mem)[i];  e_{i+1} = Wc d_i + bc + style
 * with Wc = vertice_map.weight @ vertice_map_r.weight, bc = vertice_map.weight @ vertice_map_r.bias +
 * vertice_map.bias (a2f_pack_feedback) -- algebraically the reference's 64->15069->64 feedback.
 * The ALiBi-style bias -slope_h*floor((i-j)/period) (ref:faceformer.py:22-54) and the diagonal memory mask
 * (ref:faceformer.py:58-66, which reduces cross-attention to out_proj(v_proj(mem_i))) are generated in-register.
 * Output D: [B,T,64] fp32 decoder states; the vertices follow from a2f_gemm with the template epilogue.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct a2f_decoder_weights {
    const float* sa_in_w;  /* [192,64] self_attn.in_proj_weight */
    const float* sa_in_b;  /* [192] */
    const float* sa_out_w; /* [64,64] */
    const float* sa_out_b; /* [64] */
    const float* ca_in_w;  /* [192,64] multihead_attn.in_proj_weight (only rows 128:192 are live) */
    const float* ca_in_b;  /* [192] */
    const float* ca_out_w; /* [64,64] */
    const float* ca_out_b; /* [64] */
    const float* lin1_w;   /* [128,64] */
    const float* lin1_b;   /* [128] */
    const float* lin2_w;   /* [64,128] */
    const float* lin2_b;   /* [64] */
    const float* n1_w;     /* norm1..3 weight/bias [64] */
    const float* n1_b;
    const float* n2_w;
    const float* n2_b;
    const float* n3_w;
    const float* n3_b;
    const float* fb_w;  /* [64,64] Wc from a2f_pack_feedback */
    const float* fb_b;  /* [64] bc */
    const float* obj_w; /* [64,n_onehot] obj_vector.weight (no bias) */
    const float* pe;    /* [period,64] first period rows of PPE.pe */
    const float* fold_w;  /* [192,64]      self_attn.in_proj_weight @ Wc          (a2f_pack_decoder_fold) */
    const float* fold_pe; /* [period,192]  pe[pos] @ self_attn.in_proj_weight^T   (a2f_pack_decoder_fold) */
} a2f_decoder_weights;

size_t a2f_decoder_workspace_bytes(int B, int T);
int a2f_decoder_rollout(const a2f_decoder_weights* w, const float* memory /*[B,T,64]*/, const float* one_hot
                        /*[B,n_onehot]*/, int n_onehot, int period, float* D /*[B,T,64]*/, int B, int T,
                        void* workspace, size_t workspace_bytes, void* stream);
/* Training variant: identical result, additionally stores the per-step activations the backward pass needs into
 * `saves` (fp32; field f is a dense [B,T,width_f] block starting at float offset B*T*a2f_decoder_save_offset(f);
 * total size B*T*a2f_decoder_save_offset(A2F_DEC_NFIELDS) floats).  The first 2*B*T*64 floats of `workspace` hold
 * v_proj(memory) and the cross-attention vectors afterwards (read by a2f_decoder_rollout_bwd's caller). */
#define A2F_DEC_X 0      /* decoder input e_i + pe          64 */
#define A2F_DEC_Q 1      /* scaled query                    64 */
#define A2F_DEC_K 2      /*                                 64 */
#define A2F_DEC_V 3      /*                                 64 */
#define A2F_DEC_CTX 4    /* attention output (heads concat) 64 */
#define A2F_DEC_Y1PRE 5  /* x + self_attn (LN1 input)       64 */
#define A2F_DEC_Y2PRE 6  /* LN1 out + cross-attn (LN2 in)   64 */
#define A2F_DEC_Y2 7     /* LN2 output                      64 */
#define A2F_DEC_HID 8    /* relu(linear1)                  128 */
#define A2F_DEC_Y3PRE 9  /* LN3 input                       64 */
#define A2F_DEC_LSE 10   /* self-attn log-sum-exp per head   4 */
#define A2F_DEC_NFIELDS 11
int a2f_decoder_save_offset(int field);
int a2f_decoder_rollout_train(const a2f_decoder_weights* w, const float* memory, const float* one_hot, int n_onehot,
                              int period, float* D, int B, int T, void* workspace, size_t workspace_bytes, float* saves,
                              void* stream);

/* a2f_decoder_rollout with the cross-attention vectors already computed: ca [B,T,64] = out_proj(v_proj(memory)).  Because
 * memory = audio_feature_map(h) is itself linear, a caller can fold the three Linear layers into ONE [64, 768] GEMM from the
 * encoder states (modules.Faceformer does, for inference); the two 64x64 SIMT GEMM launches of a2f_decoder_rollout
 * disappear.  Same workspace contract. */
int a2f_decoder_rollout_ca(const a2f_decoder_weights* w, const float* ca, const float* one_hot, int n_onehot, int period,
                           float* D, int B, int T, void* workspace, size_t workspace_bytes, void* stream);

/* Inference rollout that hands its result to the vertex head WHILE it runs (one CTA per utterance: 116 of the 148 SMs of a
 * B200 are idle during a 32-utterance rollout).  Besides D, every finished frame i is written as the head's bf16 operand
 * (hi | lo | hi of a2f_split_bf16x3, 192 columns) to row i * B + b of z3_frame_major, then frames_done[i] is incremented
 * with release semantics, once per utterance.  z3_frame_major: a2f_vertex_head_stream_rows(B, T) rows x 192 bf16;
 * frames_done: T zeroed counters.  Always the single-CTA-per-utterance kernel. */
int a2f_decoder_rollout_stream(const a2f_decoder_weights* w, const float* ca, const float* one_hot, int n_onehot, int period,
                               float* D, int B, int T, void* workspace, size_t workspace_bytes, void* z3_frame_major,
                               unsigned* frames_done, void* stream);
/* The consumer: out[b, t, :] = W3 z3[t * B + b, :] + bias + tmpl[b, :] for B in {32, 64, 128} utterances (ref:
 * src/model/faceformer.py:181-188), launched on a SECOND stream at the same time as a2f_decoder_rollout_stream.  The
 * tcgen05 vertex-head kernel processes groups of 128 / B frames in frame order; the producer warp of a tile waits
 * (ld.acquire.gpu) until frames_done of the group's last frame has reached B.  The grid is capped at #SMs - reserve_sms
 * so that the rollout's CTAs are resident whatever order the two kernels start in (reserve_sms >= B).  Same bits as
 * a2f_gemm on the utterance-major operand. */
int a2f_vertex_head_stream_rows(int B, int T);   /* rows of z3_frame_major (0 = this B is not supported) */
int a2f_vertex_head_stream(const void* z3_frame_major, const void* w3, int K3, const float* bias, const float* tmpl, int B, int T,
                           int V3, float* out, const unsigned* frames_done, int reserve_sms, void* stream);

/* Backward through the rollout (BPTT; the reference trains by free rollout, ref:src/model/faceformer.py:154-185, so
 * gradients flow through the fed-back embeddings).  One persistent CTA per utterance walks the frames in reverse.
 * gD: [B,T,64] dL/dd_i from the vertex head.  grads (fp32): field f is a dense [B,T,width_f] block at float offset
 * B*T*a2f_decoder_grad_offset(f); after the [B,T,*] blocks follow DSTYLE [B,64].  The per-step vectors are turned into
 * weight gradients by batched a2f_gemm_wgrad / a2f_colsum calls (the sequential kernel carries no outer products).
 * workspace: a2f_decoder_bwd_workspace_bytes(B,T), zero-filled by the call. */
#define A2F_DECG_GD 0    /* dL/dd_i total (LN3 output grad)        64 */
#define A2F_DECG_G3 1    /* dL/d(LN3 input)                        64 */
#define A2F_DECG_GHID 2  /* dL/d(linear1 pre-activation)          128 */
#define A2F_DECG_GY2 3   /* dL/d(LN2 output)                       64 */
#define A2F_DECG_G2 4    /* dL/d(LN2 input) = dL/d(cross-attn)     64 */
#define A2F_DECG_G1 5    /* dL/d(LN1 input) = dL/d(self-attn out)  64 */
#define A2F_DECG_GQKV 6  /* dL/d(in_proj output) (raw q | k | v)  192 */
#define A2F_DECG_DEFB 7  /* dL/de_i for i >= 1 (row 0 zero)        64 */
#define A2F_DECG_NFIELDS 8
int a2f_decoder_grad_offset(int field);
size_t a2f_decoder_bwd_workspace_bytes(int B, int T);
int a2f_decoder_rollout_bwd(const a2f_decoder_weights* w, const float* saves, const float* gD, int period, float* grads,
                            int B, int T, void* workspace, size_t workspace_bytes, void* stream);
/* dgamma[64] += sum_rows dy * xhat(x), dbeta[64] += sum_rows dy  for a LayerNorm(64) with saved input x */
int a2f_ln64_param_grad(const float* dy, const float* x, long long rows, float* dgamma, float* dbeta, void* stream);

/* Wc[64,64], bc[64] from vertice_map {weight [64,V3], bias [64]} and vertice_map_r {weight [V3,64], bias [V3]};
 * accumulation in fp64. */
int a2f_pack_feedback(const float* vm_w, const float* vm_b, const float* vmr_w, const float* vmr_b, int V3, float* Wc,
                      float* bc, void* stream);
/* The cross-attention of the decoder layer under the diagonal memory mask (ref:src/model/faceformer.py:58-66,168-179)
 * is out_proj(v_proj(audio_feature_map(h))).  Folds the three Linear layers (fp64) into one operand for a2f_gemm:
 *   W[64,Kin] = wo wv wa,  b[64] = wo (wv ba + bv) + bo
 * wv / bv: rows 128..191 of multihead_attn.in_proj_{weight,bias}; wo / bo: multihead_attn.out_proj; wa [64,Kin] / ba:
 * audio_feature_map.  W is written as fp32 or bf16 (w_dtype). */
/* The feedback e_{i+1} = Wc d_i + bc + style (+ pe_{i+1}) and the self-attention in-projection of token i+1 are two Linear
 * layers in a row; the rollout kernels apply them as ONE matvec from d_i.  This packs its operands (fp64 accumulation):
 *   fold_w[192,64] = sa_in_w @ Wc,   fold_pe[pos,192] = sa_in_w @ pe[pos]  for pos < period.
 * Call after a2f_pack_feedback (Wc must be current) whenever self_attn.in_proj_weight, vertice_map(_r) or PPE change. */
/* debug: device buffer of 13 uint64 (or NULL to switch off) that receives, from thread 0 of CTA 0 of every following
 * single-CTA rollout launch, the clock cycles it spent in 12 sections of the step loop ([12] = number of steps; the sections
 * are listed in tools/decoder_phases.py).  Launches a separate instantiation of the kernel: production code is unaffected. */
int a2f_debug_set_decoder_timing(void* dev_ptr);
int a2f_pack_decoder_fold(const float* sa_in_w, const float* wc, const float* pe, int period, float* fold_w, float* fold_pe,
                          void* stream);
int a2f_pack_cross_attention(const float* wv, const float* bv, const float* wo, const float* bo, const float* wa,
                             const float* ba, int Kin, void* W, int w_dtype, float* b, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * VOCA trunk (ref:src/model/voca.py:19-46): one-hot tiling + 4 x (Conv2d(3x1,s2,p1)+ReLU) + concat(one_hot[:8])
 * + Linear 72->72 -> Linear 72->128 -> tanh -> Linear 128->50, fused in one kernel (one warp-group per window).
 * x: [B,29,16], one_hot: [B,n_onehot] (first 8 used), z: [B,ldz] fp32 or bf16 with the 50 live columns first and
 * columns 50..ldz-1 zeroed (ldz = 64 feeds the vertex-head GEMM with K padded to a UMMA-friendly 64).
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct a2f_voca_weights {
    const float* conv_w[4]; /* time_conv.{0,2,4,6}.weight [32,37,3,1] [32,32,3,1] [64,32,3,1] [64,64,3,1] */
    const float* conv_b[4];
    const float* fc_w[3]; /* decoder.{0,1,3}.weight [72,72] [128,72] [50,128] */
    const float* fc_b[3];
} a2f_voca_weights;
int a2f_voca_trunk(const a2f_voca_weights* w, const float* x, const float* one_hot, int n_onehot, void* z, int z_dtype,
                   int ldz, int B, void* stream);

/* the same im2col with plain fp32 rows [rows, kpad] (SIMT parity path; Song2Face's k=5 / k=3 convolutions) */
int a2f_im2col1d(const float* x, long long outer, long long outer_stride, int ld, int C, int L, int taps, int stride, int pad,
                 const float* scale, const float* shift, int kpad, float* out, void* stream);
/* ---- Song2Face (ref:src/model/song2face.py:5-72) specific pieces; its convolutions, projections, MLP and head reuse
 * a2f_im2col1d(_split) + a2f_gemm, a2f_a2m_mlp and the vertex-head GEMM ---- */
/* y[b, c, r] = x[b, r, c]  (fp32): conv output [B, H, C] -> the [B, steps = C, features = H] tensor the LSTM reads */
int a2f_transpose_batched(const float* x, float* y, int B, int R, int C, void* stream);
/* single-layer batch_first LSTM recurrence (torch.nn.LSTM gate order i, f, g, o; h0 = c0 = 0):
 *   gates_t = xp[b, t, :] + W_hh h_{t-1},  xp = x W_ih^T + b_ih + b_hh precomputed for all steps ([B, T, 4*hidden]),
 *   whh_t = W_hh transposed to [hidden, 4*hidden], whh_n = W_hh as stored [4*hidden, hidden];  hout [B, T, hidden];
 *   hidden must be 256.  From 4 sequences on an 8-CTA thread-block cluster keeps W_hh (whh_n) in shared memory for the whole
 *   sequence and exchanges h_t through distributed shared memory; smaller batches stream whh_t from L2 every step. */
int a2f_lstm_recurrence(const float* xp, const float* whh_t, const float* whh_n, float* hout, int B, int T, int hidden,
                        void* stream);
/* out[b, i, t] = bilinear resize (align_corners = False) of h[b, t, :] from `hidden` to out_h samples: ref song2face.py:65-66
 * F.interpolate(x.unsqueeze(3), size=(32, 1)) written channels-last [B, out_h, T] for the regression convs */
int a2f_song2face_resize(const float* h, int B, int T, int hidden, int out_h, float* out, void* stream);
/* ---- Song2Face training step (model.train(); conv_training.py).  All fp32, hidden must be 256, any B >= 1 (8-CTA
 * clusters of 8 sequences; a partly filled cluster ignores the missing sequences). ----
 * a2f_lstm_recurrence_train: the recurrence of a2f_lstm_recurrence on the cluster kernel for every B, whh_n = W_hh
 *   [4*hidden, hidden]; hout [B, T, hidden] as there (bit-identical from B = 4 on, where inference runs the same kernel),
 *   and per step the post-activation gates [B, T, 4*hidden] (i, f, g, o = sigmoid, sigmoid, tanh, sigmoid) and the cell
 *   state c_t [B, T, hidden] that a2f_lstm_bptt reads. */
int a2f_lstm_recurrence_train(const float* xp, const float* whh_n, float* hout, float* gates, float* cell, int B, int T, int hidden,
                              void* stream);
/* a2f_lstm_bptt: backpropagation through time of that LSTM.  dh_out [B, T, hidden] = dL/dh_t from above the layer;
 *   gates / cell as saved by a2f_lstm_recurrence_train; -> dgates [B, T, 4*hidden] = dL/d(pre-activation gates), i.e.
 *   dL/dxp.  For t = T-1 .. 0 with dh = dh_out_t + W_hh^T da_{t+1}, dc carried from t+1, c_{-1} = 0:
 *     tc = tanh(c_t); dc += dh o (1 - tc^2); da = (dc g i(1-i), dc c_{t-1} f(1-f), dc i (1-g^2), dh tc o(1-o)); dc <- dc f.
 *   The weight, bias and input gradients follow from dgates by GEMMs.  Deterministic (no atomics). */
int a2f_lstm_bptt(const float* dh_out, const float* gates, const float* cell, const float* whh_n, float* dgates, int B, int T,
                  int hidden, void* stream);
/* a2f_col2im1d: adjoint of a2f_im2col1d with the same argument list (x becomes the output dx, out the input dcol):
 *   dx[o*outer_stride + l*ld + c] = sum over (lo, tap) with lo*stride - pad + tap = l of dcol[o*L_out + lo, tap*C + c]
 *   (times scale[c] when scale != NULL; shift does not enter the adjoint).  Every element l < L, c < C of dx is written
 *   (gathered, deterministic); columns c >= C of a row are left untouched. */
int a2f_col2im1d(float* dx, long long outer, long long outer_stride, int ld, int C, int L, int taps, int stride, int pad,
                 const float* scale, const float* shift, int kpad, const float* dcol, void* stream);
/* a2f_song2face_resize_bwd: adjoint of a2f_song2face_resize: dout [B, out_h, T] -> dh [B, T, hidden], every column written
 *   (zeros where no output sample reads a hidden unit); gathered, deterministic. */
int a2f_song2face_resize_bwd(const float* dout, int B, int T, int hidden, int out_h, float* dh, void* stream);
/* fused output MLP of Audio2Mesh (ref:src/model/audio2face.py:49-55 minus the vertex head):
 *   z[r, :n2] = W2 tanh(W1 (W0 [feat[r, :k_feat] ; extra[r, :k_extra]] + b0) + b1) + b2,  z[r, n2:ldz] = 0
 * all fp32, row-major weights [n_out, n_in]; every width <= 512. */
int a2f_a2m_mlp(const float* feat, int ld_feat, int k_feat, const float* extra, int k_extra, const float* w0, const float* b0,
                int n0, const float* w1, const float* b1, int n1, const float* w2, const float* b2, int n2, float* z, int ldz,
                int B, void* stream);
/* explicit im2col of a 1-D convolution over the middle axis of a channels-last fp32 activation x[o*outer_stride + l*ld + c]
 * (o < outer, l < L, c < C) into the error-compensated bf16 split consumed by the tcgen05 GEMM:
 *   out[(o*L_out + lo), s*kpad + tap*C + c], s = 0,1,2 = hi | lo | hi of  affine(x[o, lo*stride - pad + tap, c])  (0 outside
 *   [0,L) and for k >= taps*C), L_out = (L + 2*pad - taps)/stride + 1; affine = x*scale[c] + shift[c] when scale != NULL
 *   (an eval-mode BatchNorm that precedes the conv, ref:src/model/audio2face.py:41-46).  Audio2Mesh trunk, precision "bf16". */
int a2f_im2col1d_split(const float* x, long long outer, long long outer_stride, int ld, int C, int L, int taps, int stride,
                        int pad, const float* scale, const float* shift, int kpad, void* out, void* stream);
/* ------------------------------------------------------------------------------------------------------------
 * Audio2Mesh (ref:src/model/audio2face.py:5-69).  The ten convolutions are a2f_gemm calls over channels-last
 * activations with one zero row/column of left padding ([B,64,W+1,C] for the analysis net, [B,H+1,256] for the
 * articulation net); these two helpers build the first padded activation and apply the BatchNorms that precede a conv.
 *  a2f_a2m_assemble: x [B,52,32] + tiled one_hot (emb[r][c] = one_hot[(32r+c) % n_onehot], ref audio2face.py:59)
 *                    -> out [B,64,33] fp32, column 0 zero.
 *  a2f_channel_affine: in place x[b, r, c] = x*scale[c] + shift[c] for r < rows_per_batch (element (b,r,c) at
 *                    x + b*batch_stride + r*ld + c).
 * ---------------------------------------------------------------------------------------------------------- */
int a2f_a2m_assemble(const float* x, const float* one_hot, int n_onehot, float* out, int B, void* stream);
int a2f_channel_affine(void* x, int dtype, const float* scale, const float* shift, int C, long long rows_per_batch,
                       long long ld, long long batch_stride, long long batches, void* stream);

/* Training step of the convolutional models (train-mode BatchNorm2d = batch statistics, ref audio2face.py:13-47 under
 * Lightning's training_step).  Layout of every tensor below: element (b, r, c) at base + b*batch_stride + r*ld + c,
 * b < batches, r < rows_per_batch, c < C; callers pass `base` advanced past the left zero padding.
 *  a2f_voca_assemble: x [B,29,16] + tiled one-hot (ref voca.py:40-45) -> out [B,17,37] channels-last, row 0 zero.
 *  a2f_bn_train_stats: per-channel batch mean / rstd (biased variance, fp64 sums) -> mean_rstd [2C]; the fused
 *      scale = gamma*rstd, shift = beta - mean*scale -> scale_shift [2C]; running_mean / running_var (optional)
 *      updated with `momentum` and the unbiased variance, as torch.nn.BatchNorm2d does.  workspace: 2*C doubles.
 *  a2f_affine_act: out = act(in*scale[c] + shift[c]) (scale/shift NULL = identity); in and out may alias.
 *  a2f_bn_train_bwd: dz = d/dz of y = gamma*(z-mean)*rstd + beta given dy (masked by y_relu > 0 when a ReLU followed,
 *      y_relu NULL otherwise); dgamma / dbeta accumulate.  workspace: 2*C doubles.
 *  An eval-mode ("frozen") BatchNorm inside a training step (model.train(), the layer in eval()) normalises with its
 *  running statistics, leaves them unchanged, and its mean / rstd are constants of the step:
 *  a2f_bn_frozen_stats: mean_rstd = {running_mean, 1/sqrt(running_var + eps)} and scale_shift as a2f_bn_train_stats
 *      writes them; reads the running statistics only.
 *  a2f_bn_frozen_bwd: dz = gamma*rstd*dy_eff (dy_eff = dy masked by y_relu > 0 as above), dgamma += sum dy_eff*xhat,
 *      dbeta += sum dy_eff.  Same arguments as a2f_bn_train_bwd, mean_rstd from a2f_bn_frozen_stats.
 *      workspace: 2*C doubles. */
int a2f_voca_assemble(const float* x, const float* one_hot, int n_onehot, float* out, int B, void* stream);
int a2f_bn_train_stats(const float* x, int C, long long rows_per_batch, long long ld, long long batch_stride,
                       long long batches, const float* gamma, const float* beta, float eps, float momentum,
                       float* running_mean, float* running_var, float* mean_rstd, float* scale_shift, void* workspace,
                       size_t workspace_bytes, void* stream);
int a2f_affine_act(const float* in, float* out, const float* scale, const float* shift, int act, int C,
                   long long rows_per_batch, long long ld_in, long long bs_in, long long ld_out, long long bs_out,
                   long long batches, void* stream);
int a2f_bn_train_bwd(const float* dy, const float* y_relu, const float* z, const float* mean_rstd, const float* gamma, int C,
                     long long rows_per_batch, long long ld, long long batch_stride, long long batches, float* dz,
                     float* dgamma, float* dbeta, void* workspace, size_t workspace_bytes, void* stream);
int a2f_bn_frozen_stats(const float* gamma, const float* beta, float eps, const float* running_mean,
                        const float* running_var, int C, float* mean_rstd, float* scale_shift, void* stream);
int a2f_bn_frozen_bwd(const float* dy, const float* y_relu, const float* z, const float* mean_rstd, const float* gamma, int C,
                      long long rows_per_batch, long long ld, long long batch_stride, long long batches, float* dz,
                      float* dgamma, float* dbeta, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Losses (ref:src/loss/loss.py:24-55; FaceFormerLoss :4-17 is the same with bs = T after dropping an odd last
 * frame -- done by the caller through `rows`).  pred, gt: [rows, V3] fp32, rows even.
 *   rec = mean_{row,v} sum_xyz (p-g)^2 ; vel = same on non-overlapping row pairs (2k,2k+1) ; loss = k_rec*rec+k_vel*vel
 * out3 = {loss, rec, vel} fp32 (zeroed inside).  Optional grad: dpred = d loss / d pred * gscale (one pass).
 * ---------------------------------------------------------------------------------------------------------- */
size_t a2f_voca_loss_workspace_bytes(void);
int a2f_voca_loss_fwd(const float* pred, const float* gt, long long rows, int V3, float k_rec, float k_vel,
                      float* out3, void* workspace, size_t workspace_bytes, void* stream);
int a2f_voca_loss_bwd(const float* pred, const float* gt, long long rows, int V3, float k_rec, float k_vel,
                      const float* gscale /* device scalar d(out)/d(loss), or NULL = 1 */, float* dpred,
                      void* stream);

/* Vertex head with the losses fused into its epilogue (tensor-core path; north_star: "vertex-offset regression Linear ...
 * fused with the template add and the reconstruction/velocity losses", ref:src/model/faceformer.py:181-188 +
 * ref:src/loss/loss.py:29-55):
 *     y = z W^T + bias + tmpl[m / rows_per_tmpl];   out3 = {loss, rec, vel} of (y, gt) as a2f_voca_loss_fwd defines them;
 *     dy[m, :V3] = d loss / d y  (bf16, row stride ld_dy >= V3; columns >= V3 are left untouched: keep them zero)
 * z3 [rows, K3] / w3 [V3, K3]: the error-compensated bf16 splits of a2f_split_bf16x3 (K3 = 3 x 64).  gt [rows, V3] fp32 is
 * read once; y is stored (fp32 [rows, V3]) only when pred != NULL.  rows even (pairs of consecutive frames).  Deterministic:
 * per-warp fp64 partials in the workspace, summed in a fixed order. */
size_t a2f_vertex_head_loss_workspace_bytes(void);
int a2f_vertex_head_loss(const void* z3, const void* w3, int K3, const float* bias, const float* tmpl, int rows_per_tmpl,
                         const float* gt, long long rows, int V3, float k_rec, float k_vel, float* pred, void* dy_bf16,
                         long long ld_dy, float* out3, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Training step (BASELINE.json configs[3]): the backward pass of the path above.  The reference gets it from
 * torch.autograd over ref:src/model/faceformer.py:139-188 + HF Wav2Vec2Model inside Lightning's training_step
 * (ref:src/model/lightning_model.py:150-161); here every backward op is an explicit kernel.  Gradient outputs that are
 * parameter gradients (dgamma, dbeta, dbias, dw, dW, dv, dg ...) are ACCUMULATED into (+=), like autograd's .grad.
 * ---------------------------------------------------------------------------------------------------------- */
/* y = act(z) + resid (resid optional, dtype of y) / dz = dy * act'(z), n elements (GELU / ReLU / tanh of the forward
 * epilogues, kept as separate passes in training because the backward needs the pre-activation z). */
int a2f_act_fwd(const void* z, int z_dtype, const void* resid, void* y, int y_dtype, long long n, int act, void* stream);
int a2f_act_bwd(const void* dy, int dy_dtype, const void* z, int z_dtype, void* dz, int dz_dtype, long long n, int act,
                void* stream);
/* out[r, 0:cols] = in[r, 0:cols] converted, out[r, cols:ld_out] = 0 (bf16 operand of a backward GEMM from fp32 rows
 * whose length is not a multiple of 8, e.g. the 15069-wide vertex gradient). */
int a2f_cast_rows(const void* in, int in_dtype, long long ld_in, void* out, int out_dtype, long long ld_out, long long rows,
                  int cols, void* stream);
/* out[c*ldo + r] = in[r*ld_r + c*ld_c], r < R, c < C: W^T operands of the data-gradient GEMMs (Linear: ld_c = 1;
 * one tap of a Conv1d weight [co,ci,taps]: ld_r = ci*taps, ld_c = taps). */
int a2f_transpose_cast(const float* in, long long ld_r, long long ld_c, int R, int C, void* out, int out_dtype,
                       long long ldo, void* stream);
/* Many strided 2-D fp32 -> fp32/bf16 copies in one launch: for every job, dst[r*ldo_r + c*ldo_c] = src[r*ld_r + c*ld_c],
 * r < R, c < C.  `jobs_dev` is a DEVICE array of n_jobs entries whose `tile0` fields hold the exclusive prefix sum of
 * ceil(R/32)*ceil(C/32) (total_tiles = the full sum).  Re-derives every packed operand of a training step (bf16 casts,
 * transposed data-gradient operands, implicit-GEMM conv layouts, fused QKV) after the optimizer touched the fp32 masters
 * (the reference has no counterpart: torch.autocast re-casts weights op by op, SURVEY.md 5). */
typedef struct a2f_copy_job {
    const float* src;
    void* dst;
    long long ld_r, ld_c;      /* source strides of the logical [R, C] matrix, in elements */
    long long ldo_r, ldo_c;    /* destination strides, in elements */
    int R, C;
    int dst_dtype;             /* A2F_F32 or A2F_BF16 */
    int tile0;                 /* first 32x32 tile of this job within the launch */
} a2f_copy_job;
int a2f_strided_copy_jobs(const a2f_copy_job* jobs_dev, int n_jobs, int total_tiles, void* stream);
/* out[i0*so0+i1*so1+i2*so2] += in[i0*si0+i1*si1+i2*si2] over an n0 x n1 x n2 index space (fp32): adds a weight gradient
 * computed in the implicit-GEMM layout [co][tap][ci] into the parameter's own [co][ci][tap] .grad buffer. */
int a2f_add_strided3(const float* in, float* out, int n0, int n1, int n2, long long si0, long long si1, long long si2,
                     long long so0, long long so1, long long so2, void* stream);
/* bias gradient: out[n] += sum_m x[m*ld + n] */
int a2f_colsum(const void* x, int dtype, long long ld, long long rows, int cols, float* out, void* stream);
/* three bias gradients from one pass over a fused [rows, 3*seg_cols] gradient (q | k | v): out_i[n] += sum_m x[m*ld + i*seg_cols + n] */
int a2f_colsum3(const void* x, int dtype, long long ld, long long rows, int seg_cols, float* out0, float* out1, float* out2,
                void* stream);
/* SpecAugment time masking (training only), replaces `hidden_states[mask_time_indices] = masked_spec_embed` of
 * ref:src/model/wav2vec.py:149-162.  h / dh: [rows, cols] activations (fp32 or bf16) modified in place; mask: one byte
 * per row, non-zero = masked (the host draws it with the reference's numpy sequence, spec_augment.py); embed /
 * dembed: fp32 [cols].  bwd: dembed[c] += sum_{masked r} dh[r,c], then dh[masked rows] = 0. */
int a2f_spec_mask_fwd(void* h, int dtype, const unsigned char* mask, const float* embed, long long rows, int cols,
                      void* stream);
int a2f_spec_mask_bwd(void* dh, int dtype, const unsigned char* mask, float* dembed, long long rows, int cols,
                      void* stream);
/* Encoder dropout (training forward of the wav2vec2 encoder; HF modeling_wav2vec2.py train-mode dropout).
 *
 * RNG contract -- a keep mask depends only on (seed, offset, site, element index), never on the kernel, tile,
 * precision or launch that applies it, so a reference implementation can regenerate it exactly:
 *   generator  Philox4x32-10 (Random123 constants); key = the 64-bit seed (low word first);
 *              counter = (g lo, g hi, site, offset), where g is a 64-bit group index
 *   values     one call yields eight 16-bit values: half-word i (i = 0..7) is word i/2 of the output, low half first
 *   element e  of a site uses call g = e / 8 and half-word e % 8; it is KEPT iff that value >= round(p * 65536) and
 *              then scaled by 1 / (1 - p) (fp32); dropped elements become 0
 *   e          the row-major linear index in the site's logical tensor: [B*T, 768] for the hidden sites, [B*T, 3072]
 *              for the FFN activation, [B, 12, T, Tp] with Tp = ceil(T/8)*8 for the attention probabilities
 *   site       8 * layer + kind for the per-layer sites (kind: A2F_DROP_ATTN_PROB, A2F_DROP_ATTN_OUT, A2F_DROP_FFN_ACT,
 *              A2F_DROP_FFN_OUT); A2F_DROP_FEAT_PROJ and A2F_DROP_ENC_IN for the two sites in front of the layers
 *   seed/offset read from DEVICE memory: seed_offset_dev points at two 64-bit integers {seed, offset}; the low 32 bits
 *              of offset are used.  A training forward snapshots them for its backward and then advances the offset,
 *              so a replayed CUDA graph draws fresh masks each step.
 * A NULL args pointer, a NULL seed_offset_dev or p == 0 means "no dropout". */
typedef struct a2f_dropout_args {
    float p;                      /* drop probability in [0, 1) */
    unsigned site;                /* see the site numbering above */
    const void* seed_offset_dev;  /* {unsigned long long seed, unsigned long long offset} in device memory, or NULL */
} a2f_dropout_args;

#define A2F_DROP_ATTN_PROB 0   /* logical tensor [B, H, T, Tp], a2f_mha_fwd_train_dropout / a2f_mha_bwd_train_dropout */
#define A2F_DROP_ATTN_OUT 1
#define A2F_DROP_FFN_ACT 2
#define A2F_DROP_FFN_OUT 3
#define A2F_DROP_FEAT_PROJ 96
#define A2F_DROP_ENC_IN 97

/* the keep mask of one site over the first n elements of its logical tensor: mask[e] = 1 (kept) or 0 (dropped) */
int a2f_dropout_mask(const a2f_dropout_args* args, long long n, unsigned char* mask, void* stream);
/* y[e] = drop(x[e]) (+ resid[e] when resid is not NULL) over n elements (n % 8 == 0, 16-byte aligned, x / resid / y of
 * one dtype, A2F_F32 or A2F_BF16; y may alias x or resid).  The backward of a site is the same call on the gradient. */
int a2f_dropout_apply(const void* x, const void* resid, void* y, int dtype, long long n, const a2f_dropout_args* args,
                      void* stream);
/* LayerNorm backward over the last dim (C = 512 or 768): x is the saved LayerNorm INPUT.  dgamma / dbeta accumulate
 * (either may be NULL); dbias (optional) accumulates the column sums of dx = the bias gradient of the Linear that
 * produced x.  dx may be NULL (then dbias must be NULL): parameter gradients only, the input gradient is not computed. */
int a2f_layernorm_bwd(const void* dy, int dy_dtype, const void* x, int x_dtype, const float* gamma, float eps, void* dx,
                      int dx_dtype, float* dgamma, float* dbeta, float* dbias, long long rows, int C, void* stream);
/* backward of a2f_interp_ln: `in` [B,S,C] is the saved input, dy [B,T,C]; din [B,S,C] fp32 is ACCUMULATED into.
 * din may be NULL: dgamma / dbeta only, the input gradient is not computed. */
int a2f_interp_ln_bwd(const void* in, int in_dtype, const void* dy, int dy_dtype, const float* gamma, float eps,
                      float* din, float* dgamma, float* dbeta, int B, int S, int T, int C, void* stream);
/* backward of a2f_conv0_gn_gelu given da = dL/d(output) [B,L0,512]; gn_stats = the [B,512] (mean, rstd) float2 block
 * the forward left in its workspace (offset a2f_conv0_gn_offset(B,N) bytes).  dw [512,10], dgamma, dbeta accumulate. */
size_t a2f_conv0_gn_offset(int B, long long N);
size_t a2f_conv0_bwd_workspace_bytes(int B);
int a2f_conv0_bwd(const float* audio, const float* stats, const float* w, const float* gamma, const float* beta,
                  const void* gn_stats, const void* da, int da_dtype, int B, long long N, float* dw, float* dgamma,
                  float* dbeta, void* workspace, size_t workspace_bytes, void* stream);
/* weight_norm backward of the positional conv: dWp = gradient wrt the effective weight in the packed fp32 layout
 * [16][48][128][48] (what a2f_posconv_wgrad writes); dv [768,48,128] and dg [128] accumulate. workspace: 256 doubles. */
int a2f_weight_norm_bwd(const float* dWp, const float* v, const float* g, float* dv, float* dg, void* workspace,
                        size_t workspace_bytes, void* stream);
/* data-gradient weight of the positional conv (taps flipped, in/out swapped inside each group); norm[128] as filled by
 * a2f_pack_posconv_weight. */
int a2f_pack_posconv_dgrad_weight(const float* g, const float* v, void* out, int out_dtype, int kpad, float* norm,
                                  void* stream);
/* dh = dout + grouped_conv_transpose(dpc): input gradient of a2f_posconv (dpc = dout * gelu'(conv pre-activation)). */
int a2f_posconv_dgrad(const void* dpc, int dtype, const void* Wd, const void* dout, void* dh, int B, int T, int backend,
                      void* stream);
/* conv pre-activation only (training forward): pc = grouped_conv(h) + bias, no GELU / residual. */
int a2f_posconv_pre(const void* h, int h_dtype, const void* Wp, const float* bias, void* pc, int B, int T, int backend,
                    void* stream);
/* dWp[g][co][tap][ci] += sum_{b,t} dpc[b,t,g*48+co] * h[b,t+tap-64,g*48+ci]   (fp32 [16][48][128][48]) */
int a2f_posconv_wgrad(const void* dpc, const void* h, int dtype, float* dWp, int B, int T, int backend, void* stream);
/* fused Adam step with L2 weight decay on flat fp32 buffers (torch.optim.Adam semantics as configured at
 * ref:src/model/lightning_model.py:209-213); the gradient is multiplied by grad_scale first (1/world_size). */
int a2f_adam_step(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1, float beta2, float eps,
                  float weight_decay, int step, float grad_scale, void* stream);
/* same step with the gradient read as bf16: the flat gradient as it comes off a bf16 all-reduce (data-parallel training,
 * trainer.FlatBuffers wire="bf16": half the bytes on NVLink; masters, moments and the update stay fp32). */
int a2f_adam_step_bf16g(float* p, const void* g_bf16, float* m, float* v, long long n, float lr, float beta1, float beta2,
                        float eps, float weight_decay, int step, float grad_scale, void* stream);
/* same step with the step count t (>= 1) read from DEVICE memory, so that the launch can sit in a captured CUDA graph that is
 * replayed for every optimisation step (the caller increments *step_dev on the stream before this call); g_dtype A2F_F32 or
 * A2F_BF16. */
int a2f_adam_step_dev(float* p, const void* g, int g_dtype, float* m, float* v, long long n, float lr, float beta1, float beta2,
                      float eps, float weight_decay, const int* step_dev, float grad_scale, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * MFCC feature extractor (SURVEY.md 8(f) rank 1; replaces ref:src/model/extractor.py:10-60 = torchaudio.transforms.MFCC
 * + transpose + bilinear resize, which runs as ~8 library kernels in the reference).  The DFT itself is a2f_gemm of the
 * frame matrix with a window-folded (cos | sin) basis [2*n_freq (+pad), K]; these three entry points are the rest.
 * ---------------------------------------------------------------------------------------------------------- */
/* audio [B,N] fp32 -> frame matrix, F = 1 + N/hop rows per clip (centre=True, reflect padding n_fft/2):
 *   A[b*F+t, k] = audio_reflect[b, t*hop + (n_fft-win)/2 - n_fft/2 + k], k < win; zero for win <= k < kpad.
 * a_dtype A2F_F32: [B*F, kpad] fp32; A2F_BF16: [B*F, 3*kpad] error-compensated split [hi | lo | hi] (pair it with the
 * basis split [hi | hi | lo] of a2f_split_bf16x3).  Also resets *gmax_slot (the batch-global dB maximum) to -inf. */
int a2f_mfcc_frames(const float* audio, int B, int N, int win, int hop, int n_fft, int kpad, void* A, int a_dtype,
                    float* gmax_slot, void* stream);
/* spec [M, ld_spec] fp32 rows (Re[0..n_freq) | Im[0..n_freq)) -> db [M, n_mels] = 10*log10(max(|X|^2 @ fb, 1e-10));
 * fb [n_freq, n_mels] (torchaudio MelScale.fb), band [n_mels][2] = [first, last+1) frequency bin of each band's support;
 * *gmax_slot accumulates the maximum over everything written (torchaudio amplitude_to_DB on a 3-D batch: one cut-off). */
int a2f_mfcc_mel_db(const float* spec, int ld_spec, int M, int n_freq, const float* fb, const int* band, int n_mels,
                    float* db, float* gmax_slot, void* stream);
/* out [B, out_dim, n_mfcc] = bilinear_resize_time( max(db, gmax - top_db) @ dct ), dct [n_mels, n_mfcc] (ortho DCT-II);
 * resize = torch.nn.functional.interpolate(mode="bilinear", align_corners=False) from F to out_dim rows. */
int a2f_mfcc_dct_resize(const float* db, const float* gmax_slot, float top_db, const float* dct, int B, int F, int n_mels,
                        int n_mfcc, int out_dim, float* out, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Audio preparation (SURVEY.md 8(f) rank 3): what the reference's CPU DataLoader does before the extractor / model.
 * ---------------------------------------------------------------------------------------------------------- */
/* ref:src/dataset/vocaset.py:408-430 get_audio_fragment for frames first_frame .. first_frame+n_frames-1 of one clip:
 *   out[f, k] = pad_audio[(first_frame+f)*sample_rate/fps + k], k < 2*n_pad,
 *   pad_audio = [zeros(n_pad + shift), audio, zeros(2*n_pad)], n_pad = int(sample_rate*length/2).
 * audio_dtype A2F_F32, or A2F_I16 (scaled by 1/32768 = ref:vocaset.py:64-69 normalize_audio).  A2F_EINVAL when the last
 * fragment would end past the padded clip (the reference returns None there). */
int a2f_audio_fragments(const void* audio, int audio_dtype, long long n_samples, int first_frame, int n_frames, int sample_rate,
                        int fps, int n_pad, int shift, float* out, void* stream);
/* torchaudio.functional.resample as used at ref:src/dataset/vocaset.py:279-283 and ref:src/model/extractor.py:88:
 *   out[b, i*nnew + p] = sum_{k<kw} kernel[p][k] * xpad[b, i*orig + k],  xpad = x zero-padded by (width, width+orig),
 * orig/nnew = the two rates divided by their gcd, kernel [nnew][kw = 2*width + orig] the windowed-sinc filter bank,
 * target_len = ceil(nnew*N/orig) outputs per waveform. */
int a2f_resample_sinc(const float* x, int B, long long N, int orig, int nnew, const float* kernel, int kw, int width, float* out,
                      long long target_len, void* stream);
/* out[b, i, j] = bilinear resize (align_corners = False) of the map M_b[c, t] = h[b, t, c] (h channels-last [B, T, C], fp32 or
 * bf16) to out_h x out_w: ref:src/model/extractor.py:92-96 (Wav2VecExtractor: transpose(1,2) + F.interpolate(size=(out_dim,
 * n_feature), mode="bilinear")) in one pass. */
int a2f_bilinear_cl(const void* h, int h_dtype, int B, int T, int C, int out_h, int out_w, float* out, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Host-buffer entry points (what a non-PyTorch caller binds; also bench.py's e2e leg): pinned or pageable HOST
 * pointers in, HOST pointers out; H2D, compute and D2H are all enqueued on `stream`, then the stream is synchronised.
 * `dev_scratch` is a caller-owned DEVICE buffer of at least *_scratch_bytes.
 * ---------------------------------------------------------------------------------------------------------- */
/* debug/bring-up knobs of the tcgen05 path (tests only). field: 0=LBO enc, 1=SBO enc, 2=version, 3=layout type */
int a2f_debug_set_umma_field(int field, unsigned value);
/* debug: when non-NULL, every tcgen05 GEMM CTA writes 8 %globaltimer stamps (entry, setup done, first operands landed,
 * first tile issued, first accumulator complete, first epilogue issued, all epilogues issued, stores drained) to
 * dev_ptr[blockIdx.x*8 ..]; NULL switches it off. */
int a2f_debug_set_timeline(void* dev_ptr);

#ifdef __cplusplus
}
#endif
#endif /* A2F_H_ */
