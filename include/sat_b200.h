/* sat_b200.h -- C ABI of libsat_b200.so: the B200 (sm_100a) implementation of the
 * Show-Attend-and-Tell per-timestep decoder hot path.
 *
 * The reference (Lukeasargen/Show-Attend-and-Tell-Pytorch-Lightning) is pure Python and has
 * no FFI; the "interface" each entry point replaces is therefore a span of the reference's
 * model.py / util.py, cited per function below.  The Python host (sat_b200/model.py) mirrors
 * the reference's module/LightningModule API on top of these calls via ctypes.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer into caller-owned memory (torch tensors in practice);
 *    nothing is allocated, freed or retained by the library;
 *  - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, no host sync;
 *  - return 0 on success, SAT_ERR_INVALID (<0) for a bad argument / unsupported shape,
 *    >0 for a cudaError_t; sat_last_error() gives a thread-local message;
 *  - results are deterministic (no floating-point atomics);
 *  - dtype is the operand/storage type of activations and packed weights (SAT_F32 or
 *    SAT_BF16); accumulation, cell state, softmax, losses are always fp32;
 *  - shapes: B caption rows (= Bi images * ncap), L locations, D encoder_dim, A attention_dim,
 *    E embed_dim, H decoder_dim, V vocab, T decoder steps.  The kernels work on STORAGE dims D, A, E, H, V that are
 *    multiples of 8 (16-byte vectors, TMA rows); a module with other sizes (V = words above min_count + 4, 100/300-d GloVe
 *    embeddings ...) is zero-padded by sat_pack_weights: SatDims carries both the storage dims and the module's true dims
 *    (D0 .. V0).  Zero weights keep every padded lane exactly zero through forward and backward; padded vocabulary
 *    entries carry a bias of -inf, the cross-entropy / top-k kernels never select them, parameter gradients are written
 *    with the true shapes.
 *  - "gate-interleaved": row 4*j+g of a packed LSTM weight is row g*H+j of the torch weight
 *    (g = 0..3 for i,f,g,o), so the four gates of hidden unit j are adjacent output columns.
 */
#ifndef SAT_B200_H_
#define SAT_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SAT_F32 0
#define SAT_BF16 1
#define SAT_ERR_INVALID (-1)

#define SAT_ABI_VERSION 4
#define SAT_MAX_LAYERS 4      /* decoder_layers (nn.LSTM num_layers, model.py:175-180) supported by the kernels */

typedef struct SatDims {
  int32_t B, Bi, ncap;
  int32_t L, D, A, E, H, V, T;
  int32_t dtype;      /* SAT_F32 | SAT_BF16 */
  int32_t exact;      /* 1: libm-accurate tanh/exp (fp32 parity mode); 0: MUFU approximations */
  int32_t use_tc;     /* 1: tcgen05 tensor-core GEMMs where the shape allows (bf16 only); 0: SIMT FFMA GEMMs */
  int32_t plain_output; /* 1: DeepOutput with deep=False (model.py:128-129: x = W_ho h', no tanh / embedding / context); 0: deep */
  int32_t D0, A0, E0, H0, V0; /* true sizes of the reference module (<= the storage dims above; 0 = same as storage) */
  int32_t layers;     /* decoder_layers: stacked LSTM layers (0 or 1 = one layer).  Layer 0 takes [embedding ; beta*z], layer l > 0 the new
                         hidden state of layer l-1 (no dropout between layers); attention, beta gate and the output layer read the TOP
                         layer's state (model.py:300-327,538-547) */
} SatDims;

/* Packed decoder weights (device).  "s" = storage dtype of SatDims.dtype. */
typedef struct SatWeights {
  const void* Wa;      /* [A,D] s      attention.encoder_att.weight               model.py:90  */
  const void* Whcat;   /* [A+D+4H+E,H] s: attention.decoder_att.weight | beta.0.weight |
                          lstm.weight_hh_l0 (gate-interleaved) | output.hidden.weight           */
  const float* bhcat;  /* [A+D+4H+E]:   0 | beta.0.bias | 0 | 0                                 */
  const void* Wihz;    /* [4H,D] s     lstm.weight_ih_l0[:, E:], gate-interleaved               */
  const void* Wihe;    /* [4H,E] s     lstm.weight_ih_l0[:, :E], gate-interleaved               */
  const float* bg;     /* [4H]         bias_ih_l0 + bias_hh_l0, gate-interleaved                */
  const void* Whozo;   /* [E,H+D] s    output.hidden.weight | output.context.weight             */
  const void* Wo;      /* [V,E] s      output.output.weight                                     */
  const float* bo;     /* [V] or NULL  output.output.bias (NULL when weight-tied)               */
  const float* wf;     /* [A]          attention.f_att.weight                                   */
  const void* Emb;     /* [V,E] s      embedding.weight                                         */
  const void* Wfact;   /* [E,D] s      init_lstm.factorize.weight                               */
  const float* bfact;  /* [E]                                                                   */
  const void* Winit;   /* [2*layers*H,E] s  init_lstm.init.weight                               */
  const float* binit;  /* [2*layers*H]                                                          */
  /* transposed copies, used by the backward pass only (may be NULL for inference) */
  const void* WoT;     /* [E,V] s */
  const void* WhozoT;  /* [H+D,E] s */
  const void* WihzT;   /* [D,4H] s */
  const void* WiheT;   /* [E,4H] s */
  const void* WhcatT;  /* [H,A+D+4H] s  (first three row blocks of Whcat, transposed) */
  const void* WaT;     /* [D,A] s */
  const void* WinitT;  /* [E,2*layers*H] s */
  const void* WfactT;  /* [D,E] s */
  /* stacked layers l = 1 .. layers-1 (index l-1): the layer's input is the new hidden state of the layer below */
  const void* Wl[SAT_MAX_LAYERS - 1];    /* [4H,2H] s   lstm.weight_ih_l{l} | lstm.weight_hh_l{l}, gate-interleaved rows   */
  const float* bgl[SAT_MAX_LAYERS - 1];  /* [4H]        bias_ih_l{l} + bias_hh_l{l}, gate-interleaved                       */
  const void* WlT[SAT_MAX_LAYERS - 1];   /* [2H,4H] s   transposed (backward)                                              */
} SatWeights;

/* fp32 master parameters under the reference's names (device pointers, contiguous, SURVEY.md §A.3). */
typedef struct SatMasterWeights {
  const float* embedding;    /* embedding.weight [V,E]                       */
  const float* fact_w;       /* init_lstm.factorize.weight [E,D]             */
  const float* fact_b;       /* init_lstm.factorize.bias [E]                 */
  const float* init_w;       /* init_lstm.init.weight [2*layers*H,E]        */
  const float* init_b;       /* init_lstm.init.bias [2*layers*H]            */
  const float* w_ih;         /* lstm.weight_ih_l0 [4H,E+D]                   */
  const float* w_hh;         /* lstm.weight_hh_l0 [4H,H]                     */
  const float* b_ih;         /* lstm.bias_ih_l0 [4H]                         */
  const float* b_hh;         /* lstm.bias_hh_l0 [4H]                         */
  const float* enc_att;      /* attention.encoder_att.weight [A,D]           */
  const float* dec_att;      /* attention.decoder_att.weight [A,H]           */
  const float* f_att;        /* attention.f_att.weight [1,A]                 */
  const float* beta_w;       /* beta.0.weight [D,H]                          */
  const float* beta_b;       /* beta.0.bias [D]                              */
  const float* out_hidden;   /* output.hidden.weight [E,H]                   */
  const float* out_context;  /* output.context.weight [E,D] or NULL (deep_output=False: destination stays zero) */
  const float* out_w;        /* output.output.weight [V,E]                   */
  const float* out_b;        /* output.output.bias [V] or NULL (weight tying) */
  const float* w_ih_l[SAT_MAX_LAYERS - 1];   /* lstm.weight_ih_l{l} [4H,H], l = 1 ..   (NULL beyond decoder_layers) */
  const float* w_hh_l[SAT_MAX_LAYERS - 1];   /* lstm.weight_hh_l{l} [4H,H]  */
  const float* b_ih_l[SAT_MAX_LAYERS - 1];   /* lstm.bias_ih_l{l} [4H]      */
  const float* b_hh_l[SAT_MAX_LAYERS - 1];   /* lstm.bias_hh_l{l} [4H]      */
} SatMasterWeights;

/* Buffers of one teacher-forced training step.  fwd = written by sat_train_forward and read by
 * sat_train_backward; bwd = written by sat_train_backward. */
typedef struct SatTrainBuffers {
  /* inputs */
  const void* ann;       /* [Bi,L,D] s   annotations: channels-last view of get_encoder's [Bi,D,h,w] (model.py:483) */
  const int32_t* caps;   /* [B,T+1]      encoded captions, column 0 = <START>                     */
  const int32_t* lens;   /* [B]          number of targets per caption (model.py:492)             */
  const int32_t* sampled; /* HOST pointer, [T] flags or NULL: step t feeds back argmax_v logits[t-1] instead of the ground-truth
                            word (scheduled sampling, model.py:518-523; the host draws torch.rand(1) per step > 2); on the fused
                            path a caption finished before step t-1 keeps its ground-truth word.  sat_train_vocab_path(d, 1) names the
                            vocabulary path, and so the buffers, such a call needs                                         */
  /* fwd */
  int32_t* tok;          /* [T,B]        previous-word ids actually fed at each step (ground truth or sampled)      */
  void* P;               /* [Bi,L,A] s   W_a * a, once per image (reference recomputes per step, model.py:100) */
  void* meanv;           /* [Bi,D] s     mean over locations (model.py:78)                        */
  void* f1;              /* [Bi,E] s     init_lstm.factorize output                               */
  float* init_out;       /* [Bi,2*layers*H]  init_lstm.init output before the [2*layers,B,H] reinterpretation */
  /* per-step buffers are TIME-MAJOR (row m = t*B + b): each step's slice is a contiguous GEMM
   * operand, and the whole-sequence projections are single GEMMs with M = T*B. */
  void* Xe;              /* [T,B,E] s    embedded previous words                                  */
  float* Gx;             /* [T,B,4H]     Xe * Wihe^T + bg                                          */
  void* Hs;              /* [layers,T+1,B,H] s  hidden state of every layer before step t at [l][t] ([l][0] = h0 of layer l) */
  float* Cs;             /* [layers,T+1,B,H]    cell state                                        */
  float* hp;             /* [B,A+D+4H]   per-step scratch: q | beta_pre | W_hh h                   */
  float* Q;              /* [T,B,A]      q_t = W_h h_t (saved for backward)                        */
  float* alphas;         /* [B,T,L]      attention weights (batch-major, the reference's return layout);
                                         zeros where t >= lens[b] (model.py:534)                   */
  void* Z;               /* [T,B,D] s    context z_t                                               */
  void* GZ;              /* [T,B,D] s    beta_t * z_t  (LSTM input)                                */
  void* Beta;            /* [T,B,D] s    beta_t                                                    */
  void* Gates;           /* [layers,T,B,4H] s   post-activation i,f,g,o (gate-interleaved)         */
  void* Xo;              /* [T,B,E] s    tanh(Xe + W_ho h' + W_zo z)                               */
  void* logits;          /* [T,B,V]      s, or fp32 when logits_f32 != 0; zeros where inactive.  May be NULL when ce_stats is
                                         given (fused path)                                        */
  void* dlogits;         /* [T,B,V] s    (softmax - target dist)/N_tok; may alias `logits` when the
                                         caller does not need the logits back; NULL = not wanted   */
  float* row_loss;       /* [T,B]        per-token loss (0 where inactive)                         */
  int32_t* row_argmax;   /* [T,B]        argmax_v logits (-1 where inactive)                       */
  float* S;              /* [B,L]        sum_t alphas                                              */
  float* out;            /* [8]          loss, cross-entropy part, doubly-stochastic part, accuracy, 1/N_tok, N_tok,
                                         [6] = 1 when a caption held a word id outside [0, V0) (such ids are fed as <PAD>) */
  /* fused vocabulary projection + cross entropy (tensor-core mode, logits == NULL): the [T,B,V] logits are never written;
   * the forward keeps per-tile soft-max statistics, the backward-enabled forward recomputes the tiles into dlogits */
  float* ce_stats;       /* [T*B, ceil(V/128), 4]  max, sum exp(x - max), sum x, arg-max per 128-column tile; NULL = unfused path */
  float* row_lse;        /* [T*B]        log-sum-exp of every token row                            */
  float* row_xt;         /* [T*B]        logit of the target word                                  */
  /* bwd */
  const float* gscale;   /* [1]          upstream d(loss) (device scalar)                          */
  const float* dalpha_ext; /* [B,T,L] or NULL: extra upstream grad wrt alphas (API path: train_batch's alphas
                                         used by a caller-side loss); the fused loss path leaves it NULL  */
  void* dpre;            /* [T,B,E] s    grad wrt deep-output pre-activation                       */
  float* dHZ;            /* [T,B,H+D]    dpre * [W_ho|W_zo]                                        */
  void* DY;              /* [T,B,A+D+4H] s: dq | dbeta_pre | dG (gate-interleaved)                 */
  float* dgz;            /* [16,B,D]     per-step scratch: split-K partials of dG * Wihz                   */
  float* dh;             /* [16,B,H]     running grad wrt h: split-K partials of the h-chain GEMM          */
  float* dc;             /* [layers,B,H] running grad wrt c of every layer                         */
  void* dGl;             /* [layers-1,T,B,4H] s  pre-activation gate grads of the stacked layers l >= 1 (NULL for one layer) */
  float* dxl;            /* [layers-1,16,B,2H]   split-K partials of dG_l * [W_ih_l | W_hh_l]: columns 0..H = grad wrt the
                                         layer's input (new state of layer l-1, same step), H..2H = grad wrt its own previous state */
  float* dhq;            /* [16,B,H]     layers > 1: split-K partials of [dq | dbeta_pre] * [W_h ; W_beta] (grad wrt the top state);
                                         `dh` then holds dG_0 * W_hh_l0 only                       */
  void* dZ;              /* [T,B,D] s    total grad wrt z_t (for d_ann)                            */
  float* dP;             /* [B,L,A]      accumulated grad wrt P                                    */
  void* dP16;            /* [B,L,A] s    copy of dP in the operand dtype, written at the last backward step (t = 0);
                                         feeds the tensor-core d_ann GEMM (may be NULL in fp32 mode)          */
  float* dwf_part;       /* [T,B,A]      per-(b,t) partial of d f_att.weight                       */
  float* de;             /* [T,B,L]      scaled softmax-backward term of each step; dP is rebuilt from it, Q and P
                                          after the time loop (NULL: the slower step-by-step accumulation is used)  */
  float* dXe;            /* [T,B,E]      grad wrt embedded words                                   */
  float* d_init_out;     /* [Bi,2*layers*H]                                                       */
  float* df1;            /* [Bi,E]                                                                */
  void* d_init_out16;    /* [Bi,2*layers*H] s  operand-dtype copies feeding the tensor-core init-path GEMMs (may be NULL: SIMT) */
  void* df116;           /* [Bi,E] s                                                              */
  float* dmean;          /* [Bi,D]                                                                */
  void* d_ann;           /* [B,L,D] s    grad wrt annotations, one slab per caption row (host sums the ncap rows of an image) */
  /* scalars */
  float label_smoothing;
  float att_gamma;
  float dropout_p;       /* nn.Dropout p of InitLSTM (model.py:74,78) and DeepOutput (model.py:117,130); 0 in eval mode */
  float emb_dropout_p;   /* embedding_dropout p (model.py:164,526)                                                     */
  uint64_t dropout_seed; /* masks are a pure function of (seed, stream, element index); draw a new seed every step      */
  int32_t logits_f32;    /* logits buffer is fp32 (API path: train_batch returns fp32 logits, model.py:504) */
  int32_t reserved;
} SatTrainBuffers;

/* Buffers of one batched greedy / beam decode (SAT.forward / SAT.caption, model.py:214-472, sample_method
 * "beam", no decoder noise).  All images advance together; R = n_img * k rows, the beams of image n are rows
 * n*k .. n*k+kcur[n]-1 (order-preserving compaction, like the reference's boolean indexing). */
typedef struct SatDecodeBuffers {
  const void* ann;       /* [n_img,L,D] s                                                        */
  void* P;               /* [n_img,L,A] s                                                        */
  void* meanv;           /* [n_img,D] s                                                          */
  void* f1;              /* [n_img,E] s                                                          */
  float* init_out;       /* [n_img,2*layers*H]                                                   */
  const float* GxV;      /* [V,4H]  Emb * Wihe^T + bg per vocabulary entry (sat_decode_prepare_weights) */
  void* h;               /* [layers,R,H] s   state entering the step                              */
  float* c;              /* [layers,R,H]                                                          */
  void* hn;              /* [layers,R,H] s   state after the LSTM update, before the beam reorder  */
  float* cn;             /* [layers,R,H]                                                          */
  float* hp;             /* [R,A+D+4H]                                                            */
  void* z;               /* [R,D] s                                                               */
  void* gz;              /* [R,D] s                                                               */
  void* xo;              /* [R,E] s                                                               */
  float* logits;         /* [R,V]  SAT_VOCAB_PATH_ROWS only, else NULL                           */
  float* alpha_all;      /* [S+1,R,L]  alpha of every step and row (histories hold row indices)    */
  float* topk_stats;     /* [R, ceil(V/128), 4] or NULL: the fused paths (sat_decode_vocab_path) keep per-tile soft-max statistics
                                         (greedy: and the best word) instead of writing the logits             */
  float* cand_val;       /* [R,kcap]   per-row candidates: score (log-prob + parent score)        */
  int32_t* cand_idx;     /* [R,kcap]   word                                                       */
  float* cand_key;       /* [R,kcap]   sampling key (multinomial sampler), NULL for beam search   */
  void* h_noisy;         /* [layers,R,H] s  h + noise, operand of the recurrent projections (decoder_noise != 0), else NULL */
  int32_t* tok_hist;     /* [2,R,S+1]  generated words per live beam (ping-pong)                   */
  int32_t* asrc_hist;    /* [2,R,S+1]  row of alpha_all[step] that belongs to the beam's ancestry  */
  float* top_scores;     /* [R]                                                                   */
  int32_t* cur_tok;      /* [R]        previous word of each beam                                 */
  int32_t* src_row;      /* [R]        row of hn/cn each new beam continues from                   */
  int32_t* alive;        /* [R]                                                                   */
  int32_t* kcur;         /* [n_img]    live beams per image                                       */
  int32_t* fin_tokens;   /* [n_img,k,S+1]  finished captions (START/END stripped), in finishing order */
  int32_t* fin_asrc;     /* [n_img,k,S+1]                                                         */
  int32_t* fin_len;      /* [n_img,k]                                                             */
  float* fin_score;      /* [n_img,k]  rescored (None / LN / WR / BAR, model.py:405-417)           */
  float* fin_ppl;        /* [n_img,k]  exp(-score/step) (model.py:425)                             */
  int32_t* fin_count;    /* [n_img]                                                               */
  const float* temps;    /* HOST pointer, [S+1]: temperature per step (model.py:292)              */
  int32_t* live_images;  /* [1] device counter of images that still have live beams (optional, NULL = off)                  */
  volatile int32_t* done_host; /* early-out (model.py:419,436: the reference stops an image's loop when its beams are used up):
                            a pinned, device-accessible HOST int32.  The kernel that retires the last live image stores `call_id`
                            there; the launch loop of sat_decode polls it before queueing the next step and stops when it matches.
                            Effective when the host, not the GPU, paces the loop (few images); NULL = always run S+1 steps */
  int32_t k, max_gen_length, rescore;   /* rescore: 0 none, 1 LN, 2 WR, 3 BAR                      */
  float reward;
  int32_t tokPAD, tokSTART, tokEND, tokUNK;
  /* sampling decoders (model.py:360-379) and decoder noise (model.py:322-324); all zero = plain beam search */
  int32_t sample_method; /* 0 "beam", 1 "multinomial" (kc draws without replacement from softmax(20*seq_scores/step)), 2 "topk"
                            (kc draws from the softmax(score/step) of every beam's sample_topk best words); Gumbel-top-k      */
  int32_t sample_topk;   /* candidates per beam of the "topk" sampler (<= 32)                      */
  int32_t kcap;          /* row pitch of cand_*: >= max(k, sample_topk); 0 = k                     */
  float decoder_noise;   /* base std-dev of the Gaussian noise added to h before the LSTM cell, scaled by 1/(step+1) */
  uint64_t sample_seed;  /* the sampling / noise draws are a pure function of (seed, step, row, word) */
  int32_t call_id;       /* non-zero tag of this call for done_host (distinguishes calls still in flight on the stream) */
  int32_t reserved1;
  /* fused beam / sampling candidates (sat_decode_vocab_path() == SAT_VOCAB_PATH_CAND; NULL otherwise): the vocabulary GEMM's
   * epilogue keeps per 128-column tile the soft-max statistics in topk_stats ([R, ceil(V/128), 4]: max and sum exp of x = logit / T)
   * and the tile's best kcap candidate words, in (key descending, word ascending) order, instead of writing the logits */
  float* tile_val;       /* [R, ceil(V/128), kcap]  x of the candidate; -inf in an empty slot                              */
  int32_t* tile_idx;     /* [R, ceil(V/128), kcap]  word; 0x7fffffff in an empty slot                                       */
  float* tile_key;       /* [R, ceil(V/128), kcap]  multinomial sampler: 20/step * x + Gumbel noise (the selection key), else NULL */
  float* topk_stats2;    /* [R, ceil(V/128), 2]     multinomial sampler: max and sum exp of 20/step * x over the unmasked words */
} SatDecodeBuffers;

int sat_version(void);
const char* sat_last_error(void);
/* sizeof() of the ABI structs as compiled, so the ctypes mirror can verify itself: 0 SatDims, 1 SatWeights, 2 SatTrainBuffers, 3 SatDecodeBuffers, 4 SatMasterWeights, 5 SatParamGrads */
int sat_abi_sizeof(int which);
/* number of kernels launched by this library in this process so far (bench.py's gpu_launches) */
unsigned long long sat_launch_count(void);

/* Converts the master parameters into every packed layout of `w` (whose pointers name caller-allocated buffers; NULL
 * destinations are skipped) with one kernel.  Replaces the implicit per-op layouts of the reference's nn.Modules
 * (model.py:158-199); run after every optimizer step. */
int sat_pack_weights(const SatDims* d, const SatMasterWeights* m, const SatWeights* w, void* stream);

/* Kernel timing for bench.py's roofline entry: while enabled, every launch of the selected kernel kind
 * (1 = attention step forward, 2 = attention step backward, 3 = vocabulary projection stage (GEMM, or the fused
 * statistics pass + row finalize + dlogits pass), 4 = gate GEMM + LSTM cell of the training forward) is bracketed by CUDA
 * events on its own stream.  sat_profile_end synchronises, returns the summed device time and count. */
int sat_profile_begin(int kind);
int sat_profile_end(float* total_ms, int* count);

/* C[M,N] (ldc) = A[M,K] (lda) * W[N,K]^T (ldw) + bias[N] (optional).  a/w dtype = dtype, C fp32 when
 * c_f32 != 0 else dtype.  The GEMM core shared by every projection below; exported for unit tests.
 * Replaces torch.nn.Linear call sites model.py:72-73,90-92,119-123,188. */
int sat_linear(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias, void* C, int64_t ldc,
               int32_t M, int32_t N, int32_t K, int32_t dtype, int32_t c_f32, int32_t use_tc, void* stream);

/* C[z][N1,N2] (fp32, ldc, one slab of N1*ldc floats per k split z < splitk) = sum over the z-th share of the Krows rows of
 * A[k,n1] * B[k,n2]: the "NT" GEMM core of the weight gradients dW = dY^T X (what autograd's mm_backward does for the
 * nn.Linear call sites model.py:72-73,90-92,119-123,188).  Exported for unit tests; sat_train_param_grads is the user. */
int sat_linear_nt(const void* A, int64_t lda, const void* B, int64_t ldb, float* C, int64_t ldc, int32_t Krows, int32_t N1, int32_t N2,
                  int32_t dtype, int32_t use_tc, int32_t splitk, void* stream);

/* Once per image: P = ann * Wa^T (model.py:100), mean over L (model.py:78), factorize/init Linear
 * layers (model.py:79) and the [B,2*layers*H] -> [2*layers,B,H] state reinterpretation (model.py:79-80) into
 * h0 [B,H] (s) / c0 [B,H] (fp32). */
int sat_prepare_images(const SatDims* d, const SatWeights* w, const void* ann, void* P, void* meanv, void* f1,
                       float* init_out, void* h0, float* c0, void* stream);

/* One decoder time step, attention part (SoftAttention.forward model.py:94-109 + beta gate
 * model.py:187-192,538-541), rows with t < lens[b] only.
 *   hp [B,ldhp] fp32 holds q (cols 0..A) and beta_pre (cols A..A+D) for this step.
 *   Writes alpha[b,:] (row stride ld_alpha), z, beta*z, beta (row strides ld_z). */
int sat_attention_step_fwd(const SatDims* d, const void* ann, const void* P, const float* wf, const float* hp,
                           int64_t ldhp, const int32_t* lens, int32_t t, float* alpha, int64_t ld_alpha, void* z,
                           void* gz, void* beta, int64_t ld_z, void* stream);

/* Whole teacher-forced forward + loss: SAT.train_batch (model.py:474-557) with epsilon = 1,
 * LabelSmoothing (util.py:105-112), doubly-stochastic term and accuracy (model.py:592-597). */
/* The dropout multiplier (0 or 1/(1-p)) the kernels apply to element `idx` of stream 1 (InitLSTM mean, idx = img*D+d),
 * 2 (embedded words, idx = (t*B+b)*E+e) or 3 (deep-output activations, idx = (t*B+b)*E+e).  Host-side mirror for tests. */
float sat_dropout_multiplier(float p, uint64_t seed, uint32_t stream, uint64_t idx);

/* int64 word ids / lengths (what the dataset's collate hands to SAT.train_batch, util.py:43-44) -> the int32 arrays
 * SatTrainBuffers.caps / .lens point to; one launch. */
int sat_cast_captions(const int64_t* caps64, const int64_t* lens64, int32_t* caps32, int32_t* lens32, int64_t n_caps, int64_t n_lens,
                      void* stream);

/* Encoder tail (SURVEY.md §8 f2; readme.md:118-121: nn.Upsample((s,s), mode="bilinear", align_corners=False) appended to the encoder
 * of model.py:16-63): bilinear resize of an NHWC map [n,h,w,D] to [n,H2,W2,D], i.e. straight into the [B,L,D] annotation array the
 * decoder kernels read -- fp32 interpolation of the stored values, one rounding to `dtype` (SAT_F32 / SAT_BF16).  _bwd is its
 * transpose in gather form (no atomics: deterministic), d_dst [n,H2,W2,D] -> d_src [n,h,w,D].  D % (16 / sizeof(dtype)) == 0. */
int sat_resize_nhwc_fwd(const void* src, void* dst, int32_t n, int32_t h, int32_t w, int32_t H2, int32_t W2, int32_t D, int32_t dtype,
                        void* stream);
int sat_resize_nhwc_bwd(const void* d_dst, void* d_src, int32_t n, int32_t h, int32_t w, int32_t H2, int32_t W2, int32_t D, int32_t dtype,
                        void* stream);

/* Which vocabulary stage sat_train_forward runs for these dims, teacher-forced (sampled = 0) or with scheduled-sampling steps
 * (sampled != 0), and so which buffers it reads: SAT_TRAIN_PATH_LOGITS = [T,B,V] `logits` + the shared-memory cross-entropy row
 * kernel (V <= 58,072), SAT_TRAIN_PATH_FUSED = `ce_stats` / `row_lse` / `row_xt` (+ `dlogits` with backward), no logits: the
 * vocabulary GEMM's epilogue keeps per-tile statistics, and a sampled step feeds back the arg-max read from them.  Teacher-forced:
 * FUSED wherever it can run (bf16 tensor cores; the caller may still keep the logits instead).  Sampled, bf16 tensor cores: FUSED
 * where a logits row does not fit the row kernel, or everywhere under SAT_TRAIN_FUSED_SS=1; LOGITS otherwise.  A caller that
 * wants the logits back (train_batch) passes `logits` and no `ce_stats`, and is held to the row kernel's limit.  < 0 (error
 * set) when no path takes the call (fp32, or bf16 without tensor cores, above the limit). */
#define SAT_TRAIN_PATH_LOGITS 0
#define SAT_TRAIN_PATH_FUSED 1
int sat_train_vocab_path(const SatDims* d, int32_t sampled);

int sat_train_forward(const SatDims* d, const SatWeights* w, SatTrainBuffers* b, void* stream);

/* Hand-written BPTT of sat_train_forward (what autograd derives from model.py:510-548): fills
 * dlogits-derived buffers, DY, dZ, dP, dwf_part, dXe, d_init_out, df1, dmean, d_ann.  The
 * reductions over (b,t) that produce the parameter gradients are sat_train_param_grads below. */
int sat_train_backward(const SatDims* d, const SatWeights* w, SatTrainBuffers* b, void* stream);

/* Destinations of the parameter gradients: fp32 device buffers with the reference's parameter shapes (true dims, contiguous;
 * SURVEY.md §A.3).  NULL = not wanted. */
typedef struct SatParamGrads {
  float* embedding;    /* embedding.weight [V0,E0]  (row pad_idx is zero: nn.Embedding(padding_idx), model.py:162)     */
  float* fact_w;       /* init_lstm.factorize.weight [E0,D0]   */
  float* fact_b;       /* init_lstm.factorize.bias [E0]        */
  float* init_w;       /* init_lstm.init.weight [2*layers*H0,E0] */
  float* init_b;       /* init_lstm.init.bias [2*layers*H0]   */
  float* w_ih;         /* lstm.weight_ih_l0 [4H0,E0+D0]        */
  float* w_hh;         /* lstm.weight_hh_l0 [4H0,H0]           */
  float* b_ih;         /* lstm.bias_ih_l0 [4H0]                */
  float* b_hh;         /* lstm.bias_hh_l0 [4H0]                */
  float* enc_att;      /* attention.encoder_att.weight [A0,D0] */
  float* dec_att;      /* attention.decoder_att.weight [A0,H0] */
  float* f_att;        /* attention.f_att.weight [1,A0]        */
  float* beta_w;       /* beta.0.weight [D0,H0]                */
  float* beta_b;       /* beta.0.bias [D0]                     */
  float* out_hidden;   /* output.hidden.weight [E0,H0]         */
  float* out_context;  /* output.context.weight [E0,D0] (deep output only) */
  float* out_w;        /* output.output.weight [V0,E0]; NULL when weight-tied */
  float* out_b;        /* output.output.bias [V0] or NULL      */
  float* w_ih_l[SAT_MAX_LAYERS - 1];   /* lstm.weight_ih_l{l} [4H0,H0], l = 1 .. decoder_layers-1 */
  float* w_hh_l[SAT_MAX_LAYERS - 1];   /* lstm.weight_hh_l{l} [4H0,H0] */
  float* b_ih_l[SAT_MAX_LAYERS - 1];   /* lstm.bias_ih_l{l} [4H0]      */
  float* b_hh_l[SAT_MAX_LAYERS - 1];   /* lstm.bias_hh_l{l} [4H0]      */
  int32_t pad_idx;     /* embedding row whose own gradient is zero, -1 = none */
  int32_t weight_tying;/* 1: output.output.weight IS embedding.weight (model.py:198-199): its gradient is added into `embedding` */
} SatParamGrads;

/* Bytes of scratch sat_train_param_grads needs for these dims (split-k partials, column-sum partials). */
int64_t sat_param_grads_workspace_bytes(const SatDims* d);

/* Parameter gradients of the step whose buffers `b` holds (after sat_train_forward + sat_train_backward): the reductions
 * over (t, b) that autograd performs for model.py:510-548 -- dW = dY^T X on the tensor cores (split-k, partials added in
 * fixed order), bias / f_att column sums, the embedding segment sum, gate de-interleave and un-padding -- all inside the
 * library and bit-reproducible from run to run (the reference trains with deterministic=True, train.py:271).
 * `workspace` is 256-byte aligned device memory of at least sat_param_grads_workspace_bytes(d) bytes. */
int sat_train_param_grads(const SatDims* d, const SatTrainBuffers* b, const SatParamGrads* g, void* workspace, int64_t workspace_bytes,
                          void* stream);

/* GxV[v,:] = Emb[v,:] * Wihe^T + bg for every vocabulary entry (once per set of weights). */
int sat_decode_prepare_weights(const SatDims* d, const SatWeights* w, float* GxV, void* stream);

/* Which vocabulary stage sat_decode runs for these dims, beam width and sample method (0 beam, 1 multinomial, 2 topk), and so
 * which buffers it reads: SAT_VOCAB_PATH_ROWS = [R,V] `logits` + the shared-memory row kernels (V <= 58,072; multinomial
 * V <= 29,032), SAT_VOCAB_PATH_GREEDY = `topk_stats` (greedy on the bf16 tensor-core path), SAT_VOCAB_PATH_CAND = `topk_stats`
 * + `tile_val` / `tile_idx` (+ `tile_key` / `topk_stats2` for the multinomial sampler): bf16 tensor-core decode where a logits
 * row does not fit the row kernels, or everywhere under SAT_VOCAB_TOPK=1.  < 0 (error set) when no path takes the call. */
#define SAT_VOCAB_PATH_ROWS 0
#define SAT_VOCAB_PATH_GREEDY 1
#define SAT_VOCAB_PATH_CAND 2
int sat_decode_vocab_path(const SatDims* d, int32_t k, int32_t sample_method, int32_t sample_topk);

/* Batched greedy (k = 1) / beam decode; d->B = n_img * k rows, d->Bi = n_img, d->ncap = k.  Runs
 * max_gen_length + 1 steps with device-side bookkeeping (no host sync); results are in the fin_* buffers. */
int sat_decode(const SatDims* d, const SatWeights* w, SatDecodeBuffers* b, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SAT_B200_H_ */
