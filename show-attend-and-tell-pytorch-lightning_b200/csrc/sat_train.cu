// Teacher-forced training step of the SAT decoder: forward + loss (sat_train_forward) and the
// hand-written BPTT (sat_train_backward), built from the fused kernels in sat_kernels.cuh and the
// GEMM cores (SIMT FFMA for fp32 parity, tcgen05 for bf16).
//
// Structure (B200-first, not a translation of model.py:510-548):
//  * everything that does not sit on the h/c recurrence is hoisted out of the time loop and run
//    as ONE GEMM over all T*B rows: W_a*a (once per image), the embedding half of the LSTM input
//    projection, the deep-output projection and the vocabulary projection + cross-entropy;
//  * the recurrent part of a step is three launches: h-projection GEMM (q | beta_pre | W_hh h),
//    fused attention kernel, gate GEMM with the LSTM cell in its epilogue;
//  * finished captions are predicated (t < lens[b]) instead of compacted, so there is no host
//    sync, no gather/scatter of state and no per-step reallocation;
//  * a scheduled-sampling step t (model.py:518-523) computes step t-1's output rows inside the loop: deep output, then
//    either the logits + row_argmax_kernel or, on the fused path, the VOCAB_STATS tiles + ss_feedback_kernel (no logits).
#include "sat_gemm.cuh"
#include "sat_attention_pipe.cuh"
#include "sat_kernels.cuh"
#include "sat_vocab_ce.cuh"

namespace {

template <typename TS>
static int prepare_images_impl(const SatDims& d, const SatWeights& w, const void* ann, void* P, void* meanv, void* f1,
                               float* init_out, void* h0, float* c0, int64_t lstride, cudaStream_t st, float drop_p = 0.0f,
                               uint64_t seed = 0) {
  // h0 / c0: state arrays of layer 0; layer l lives lstride elements further (training: (T+1)*B*H, single call: B*H)
  const int B = d.B, Bi = d.Bi, L = d.L, D = d.D, A = d.A, E = d.E, H = d.H;
  const int nl = d.layers > 1 ? d.layers : 1;
  const bool tc = d.use_tc != 0;
  // P = ann * Wa^T  ([Bi*L, D] x [A, D]^T)
  // first launch of a driver: no PDL attribute, so that operands written by the caller's preceding launch (the weight
  // pack kernel, the encoder) are complete and visible to every early (pre-wait) read of the kernels that follow
  SatNoPdlScope first_launch;
  SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(ann, D, D), (const TS*)w.Wa, D, Bi * L, A, EpiStore<TS>{(TS*)P, A, nullptr, nullptr, 0},
                           st)));
  // mean over locations, then the two Linear layers of InitLSTM (no nonlinearity between, model.py:79)
  const int NV = D / Vec16<TS>::N;
  mean_L_kernel<TS><<<dim3((NV + 31) / 32, Bi), 256, 0, st>>>((const TS*)ann, (TS*)meanv, L, D, drop_p, seed);
  SAT_COUNT_LAUNCH();
  SAT_LAUNCH_OK();
  SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(meanv, D, D), (const TS*)w.Wfact, D, Bi, E,
                           EpiStore<TS>{(TS*)f1, E, w.bfact, nullptr, 0}, st)));
  const int IO = 2 * nl * H;           // init_lstm.init output width (storage)
  SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(f1, E, E), (const TS*)w.Winit, E, Bi, IO,
                           EpiStore<float>{init_out, IO, w.binit, nullptr, 0}, st)));
  const int H0 = d.H0 ? d.H0 : H;      // the [B,2nH] -> [2n,B,H] reinterpretation works on the module's true decoder_dim
  if (H0 != H) {                        // padded state columns start (and stay) at zero
    for (int l = 0; l < nl; ++l) {
      SAT_CUDA(cudaMemsetAsync((TS*)h0 + l * lstride, 0, sizeof(TS) * (size_t)B * H, st));
      SAT_CUDA(cudaMemsetAsync(c0 + l * lstride, 0, sizeof(float) * (size_t)B * H, st));
    }
  }
  const int64_t n = 2 * (int64_t)nl * B * H0;
  init_state_kernel<TS><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(init_out, IO, (TS*)h0, c0, H, H, lstride, lstride, B, H0, d.ncap, nl);
  SAT_COUNT_LAUNCH();
  SAT_LAUNCH_OK();
  return 0;
}

constexpr size_t CE_SMEM_LIMIT = 227 * 1024;
size_t ce_smem_bytes(int V) { return sizeof(float) * (size_t)(V + 40); }      // ce_rows_kernel: one logits row + scratch

// Where the vocabulary stage of a training step runs (sat_train_vocab_path): 1 = fused (VOCAB_STATS / VOCAB_DLOGITS in the
// vocabulary GEMM's epilogue, no logits), 0 = logits + ce_rows_kernel.  Teacher-forced steps: the fused path wherever it can
// run (bf16 tensor cores), and the caller decides whether it keeps the logits instead.  Scheduled sampling: the unfused path
// while ce_rows_kernel holds a logits row, the fused one beyond that, or wherever it can run under SAT_TRAIN_FUSED_SS=1 (A/B
// timing, equivalence tests).  An error when the vocabulary fits neither.
int train_vocab_path(const SatDims& d, bool sampled) {
  const bool fused_ok = d.dtype == SAT_BF16 && d.use_tc != 0 && d.exact == 0;
  const bool rows_fit = ce_smem_bytes(d.V) <= CE_SMEM_LIMIT;
  static const int force_fused = getenv("SAT_TRAIN_FUSED_SS") ? atoi(getenv("SAT_TRAIN_FUSED_SS")) : 0;
  if (fused_ok && (!sampled || !rows_fit || force_fused != 0)) return SAT_TRAIN_PATH_FUSED;
  SAT_REQUIRE(rows_fit, "vocabulary of %d words needs %zu bytes of shared memory per row in the unfused cross-entropy kernel "
              "(limit 227 KB); training at this size needs the bf16 tensor-core path (bf16, use_tc, not exact)", d.V, ce_smem_bytes(d.V));
  return SAT_TRAIN_PATH_LOGITS;
}

template <typename TS, bool kExact>
int train_forward_impl(const SatDims& d, const SatWeights& w, SatTrainBuffers& b, cudaStream_t st) {
  const int B = d.B, Bi = d.Bi, L = d.L, D = d.D, A = d.A, E = d.E, H = d.H, V = d.V, T = d.T;
  const int NH3 = A + D + 4 * H;
  const int caplen = T + 1;
  const bool tc = d.use_tc != 0;
  const int V0 = d.V0 ? d.V0 : V;
  const TS* ann = (const TS*)b.ann;
  // fused vocabulary projection + cross entropy (tensor-core mode): the logits are never written
  const bool fuse_ce = b.ce_stats != nullptr && b.row_lse != nullptr && b.row_xt != nullptr && std::is_same<TS, bf16>::value && tc && !kExact &&
                       tc::operands_ok(gemm_a1(b.Xo, E, E), w.Wo, E);
  SAT_REQUIRE(fuse_ce || b.logits != nullptr, "sat_train_forward: logits buffer missing (only the fused tensor-core path can do without)");
  if (b.sampled != nullptr) {
    // scheduled sampling: sat_train_vocab_path decides; a caller that asks for the logits (train_batch) always gets them
    const int path = train_vocab_path(d, true);
    if (path < 0) return path;
    SAT_REQUIRE(!fuse_ce || path == SAT_TRAIN_PATH_FUSED, "sat_train_forward: fused vocabulary buffers given to a scheduled-sampling step whose "
                "vocabulary path is the unfused one (sat_train_vocab_path)");
  }
  SAT_REQUIRE(fuse_ce || ce_smem_bytes(V) <= CE_SMEM_LIMIT, "vocabulary of %d words needs %zu bytes of shared memory per row in the "
              "unfused cross-entropy kernel (limit 227 KB); training at this size needs the bf16 tensor-core path (bf16, use_tc, "
              "not exact) without kept logits", V, ce_smem_bytes(V));
  const int NTv = (V + 127) / 128;                        // 128-column vocabulary tiles per row (fused path)

  // ---- once per image ------------------------------------------------------------------------
  const int nl = d.layers > 1 ? d.layers : 1;
  const int64_t LS = (int64_t)(T + 1) * B * H;           // distance between the layers' state arrays in Hs / Cs
  const int64_t GS = (int64_t)T * B * 4 * H;             // ... in Gates
  TS* const Hs_top = (TS*)b.Hs + (nl - 1) * LS;          // attention, beta gate and the output layer read the top layer
  SAT_TRY((prepare_images_impl<TS>(d, w, b.ann, b.P, b.meanv, b.f1, b.init_out, b.Hs, b.Cs, LS, st, b.dropout_p, b.dropout_seed)));

  // ---- hoisted: embeddings of the (teacher-forced) previous words and their gate projection ---
  SAT_CUDA(cudaMemsetAsync(b.out, 0, 8 * sizeof(float), st));
  tok_init_kernel<<<(T * B + 255) / 256, 256, 0, st>>>(b.caps, b.tok, B, T, caplen, V0, b.out + 6);
  SAT_COUNT_LAUNCH();
  embed_gather_kernel<TS><<<T * B, 64, 0, st>>>((const TS*)w.Emb, b.tok, (TS*)b.Xe, E, 0, b.emb_dropout_p, b.dropout_seed);
  SAT_COUNT_LAUNCH();
  SAT_LAUNCH_OK();
  SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(b.Xe, E, E), (const TS*)w.Wihe, E, T * B, 4 * H,
                           EpiStore<float>{b.Gx, 4 * H, w.bg, nullptr, 0}, st)));

  // ---- recurrence ------------------------------------------------------------------------------
  const float scale = (float)(1.0 / sqrt((double)L));
  // The attention kernels re-read the same annotations at every step: when they fit the persisting part of the L2 they are
  // pinned there for the time loop (read from HBM once per step sequence instead of T times)
  struct L2Scope {
    L2Scope(const void* p, size_t n) {
      const size_t lim = sat_l2_persist_limit();
      if (lim > 0 && n > 0) { sat_l2_window().ptr = p; sat_l2_window().bytes = n < lim ? n : lim; sat_l2_window().hit_ratio = n <= lim ? 1.0f : (float)lim / (float)n; }
    }
    ~L2Scope() { sat_l2_window().ptr = nullptr; sat_l2_window().bytes = 0; }
  } l2scope(b.ann, sizeof(TS) * (size_t)Bi * L * D);
  for (int t = 0; t < T; ++t) {
    if (b.sampled != nullptr && t > 0 && b.sampled[t]) {
      // scheduled sampling (model.py:518-523): this step's input word is argmax_v logits[t-1]; compute the output of
      // step t-1 now (the hoisted whole-sequence GEMMs below recompute the same values), then re-embed and re-project.
      const int64_t o1 = (int64_t)(t - 1) * B;
      SAT_PROF(8, st);                                      // 8 = the extra work of a sampled step, deep output to Gx[t]
      SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a2((const TS*)Hs_top + (int64_t)t * B * H, H, H, (const TS*)b.Z + o1 * D, D, D), (const TS*)w.Whozo,
                               H + D, B, E, EpiTanhAdd<TS, kExact>{(const TS*)b.Xe + o1 * E, (TS*)b.Xo + o1 * E, E, nullptr, d.plain_output, b.dropout_p, b.dropout_seed, o1}, st)));
      if (fuse_ce) {
        // fused: the tile statistics of step t-1's rows (the hoisted pass rewrites them with the same values), then the
        // arg-max of each live row by the rule ce_finalize_kernel reports as row_argmax; no logits are written
        tc::VocabArgs va{};
        va.bias = w.bo; va.V0 = V0; va.NT = NTv; va.stats = reinterpret_cast<float4*>(b.ce_stats) + o1 * NTv;
        va.caps = b.caps; va.lens = b.lens; va.B = B; va.caplen = caplen; va.row0 = (int)o1; va.row_xt = b.row_xt + o1;
        SAT_TRY((tc::launch_vocab<tc::VOCAB_STATS>(gemm_a1((const TS*)b.Xo + o1 * E, E, E), (const bf16*)w.Wo, E, B, V, va, st)));
        SAT_CUDA(sat_launch_pdl(tc::ss_feedback_kernel, dim3((B + 7) / 8), dim3(256), 0, st, (const float4*)va.stats, NTv,
                                (const int32_t*)b.lens, B, t, V0, b.tok + (int64_t)t * B));
      } else if (b.logits_f32) {
        SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1((const TS*)b.Xo + o1 * E, E, E), (const TS*)w.Wo, E, B, V,
                                 EpiStore<float>{(float*)b.logits + o1 * V, V, w.bo, nullptr, 0}, st)));
        row_argmax_kernel<float><<<B, 256, 0, st>>>((const float*)b.logits + o1 * V, b.tok + (int64_t)t * B, V);
      } else {
        SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1((const TS*)b.Xo + o1 * E, E, E), (const TS*)w.Wo, E, B, V,
                                 EpiStore<TS>{(TS*)b.logits + o1 * V, V, w.bo, nullptr, 0}, st)));
        row_argmax_kernel<TS><<<B, 256, 0, st>>>((const TS*)b.logits + o1 * V, b.tok + (int64_t)t * B, V);
      }
      SAT_COUNT_LAUNCH();
      embed_gather_kernel<TS><<<B, 64, 0, st>>>((const TS*)w.Emb, b.tok + (int64_t)t * B, (TS*)b.Xe + (int64_t)t * B * E, E, (int64_t)t * B,
                                                b.emb_dropout_p, b.dropout_seed);
      SAT_COUNT_LAUNCH();
      SAT_LAUNCH_OK();
      SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1((const TS*)b.Xe + (int64_t)t * B * E, E, E), (const TS*)w.Wihe, E, B, 4 * H,
                               EpiStore<float>{b.Gx + (int64_t)t * B * 4 * H, 4 * H, w.bg, nullptr, 0}, st)));
      SAT_PROF(8, st);
    }
    const TS* h_t = (const TS*)b.Hs + (int64_t)t * B * H;            // layer 0
    const float* c_t = b.Cs + (int64_t)t * B * H;
    const TS* htop_t = Hs_top + (int64_t)t * B * H;
    if (nl == 1) {
      // hp = h_t * [W_h | W_beta | W_hh]^T + [0 | b_beta | 0]
      SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(h_t, H, H), (const TS*)w.Whcat, H, B, NH3,
                               EpiStore<float>{b.hp, NH3, w.bhcat, nullptr, 0}, st)));
    } else {
      // stacked layers: q | beta_pre from the top layer's state, the recurrent projection of layer 0 from its own
      SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(htop_t, H, H), (const TS*)w.Whcat, H, B, A + D,
                               EpiStore<float>{b.hp, NH3, w.bhcat, nullptr, 0}, st)));
      SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(h_t, H, H), (const TS*)w.Whcat + (int64_t)(A + D) * H, H, B, 4 * H,
                               EpiStore<float>{b.hp + A + D, NH3, nullptr, nullptr, 0}, st)));
    }
    TS* z_t = (TS*)b.Z + (int64_t)t * B * D;
    TS* gz_t = (TS*)b.GZ + (int64_t)t * B * D;
    TS* beta_t = (TS*)b.Beta + (int64_t)t * B * D;
    SAT_PROF(1, st);
    SAT_TRY((launch_attention_fwd<TS, kExact>(ann, (const TS*)b.P, w.wf, b.hp, NH3, b.lens, t, B, d.ncap, L, D, A, scale,
                                              b.alphas + (int64_t)t * L, (int64_t)T * L, b.Q + (int64_t)t * B * A, z_t, gz_t,
                                              beta_t, D, st)));
    SAT_PROF(1, st);
    // gates = gz * Wihz^T + Gx[t] + hp[:, A+D:]  -> LSTM cell -> h_{t+1}, c_{t+1}
    EpiLstm<TS, kExact> epi{b.Gx + (int64_t)t * B * 4 * H, 4 * H, b.hp + A + D, NH3, h_t, c_t,
                            (TS*)b.Hs + (int64_t)(t + 1) * B * H, b.Cs + (int64_t)(t + 1) * B * H, H, H,
                            (TS*)b.Gates + (int64_t)t * B * 4 * H, 4 * H, b.lens, t, nullptr};
    SAT_PROF(4, st);
    SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(gz_t, D, D), (const TS*)w.Wihz, D, B, 4 * H, epi, st)));
    SAT_PROF(4, st);
    for (int l = 1; l < nl; ++l) {
      // layer l: gates = [h'_{l-1} ; h_l] * [W_ih_l | W_hh_l]^T + b_l  (no dropout between layers, model.py:175-180)
      const TS* hin = (const TS*)b.Hs + (l - 1) * LS + (int64_t)(t + 1) * B * H;
      const TS* hl = (const TS*)b.Hs + l * LS + (int64_t)t * B * H;
      const float* cl = b.Cs + l * LS + (int64_t)t * B * H;
      EpiLstm<TS, kExact> epl{w.bgl[l - 1], 0, nullptr, 0, hl, cl, (TS*)b.Hs + l * LS + (int64_t)(t + 1) * B * H,
                              b.Cs + l * LS + (int64_t)(t + 1) * B * H, H, H, (TS*)b.Gates + l * GS + (int64_t)t * B * 4 * H, 4 * H, b.lens,
                              t, nullptr};
      SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a2(hin, H, H, hl, H, H), (const TS*)w.Wl[l - 1], 2 * H, B, 4 * H, epl, st)));
    }
  }

  // ---- hoisted: deep output (model.py:127) and vocabulary projection (model.py:130) over all T*B rows
  const TS* Hnext = (const TS*)Hs_top + (int64_t)B * H;   // h' of step t lives at Hs[top][t+1]
  SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a2(Hnext, H, H, b.Z, D, D), (const TS*)w.Whozo, H + D, T * B, E,
                           EpiTanhAdd<TS, kExact>{(const TS*)b.Xe, (TS*)b.Xo, E, nullptr, d.plain_output, b.dropout_p, b.dropout_seed, 0}, st)));
  ntok_kernel<<<1, 256, 0, st>>>(b.lens, B, b.out);
  SAT_COUNT_LAUNCH();
  SAT_PROF(3, st);
  if (fuse_ce) {
    // pass 1: per-tile soft-max statistics in the GEMM epilogue; finish per row; pass 2 (training only): recompute the tiles
    // into dlogits.  HBM traffic of the stage: one bf16 [T*B, V] write instead of write + read + write.
    tc::VocabArgs va{};
    va.bias = w.bo; va.V0 = V0; va.NT = NTv; va.stats = reinterpret_cast<float4*>(b.ce_stats);
    va.caps = b.caps; va.lens = b.lens; va.B = B; va.caplen = caplen; va.row_xt = b.row_xt; va.row_lse = b.row_lse;
    va.inv_ntok_p = b.out + 4; va.smoothing = b.label_smoothing; va.dlogits = (bf16*)b.dlogits; va.ldd = V;
    SAT_TRY((tc::launch_vocab<tc::VOCAB_STATS>(gemm_a1(b.Xo, E, E), (const bf16*)w.Wo, E, T * B, V, va, st)));
    SAT_CUDA(sat_launch_pdl(tc::ce_finalize_kernel, dim3((T * B + 7) / 8), dim3(256), 0, st, (const float4*)va.stats, va.NT,
                            (const float*)b.row_xt, b.lens, B, T * B, V0, b.label_smoothing, b.row_lse, b.row_loss, b.row_argmax));
    SAT_COUNT_LAUNCH();
    if (b.dlogits != nullptr) SAT_TRY((tc::launch_vocab<tc::VOCAB_DLOGITS>(gemm_a1(b.Xo, E, E), (const bf16*)w.Wo, E, T * B, V, va, st)));
    SAT_PROF(3, st);
  } else {
    if (b.logits_f32) {
      SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(b.Xo, E, E), (const TS*)w.Wo, E, T * B, V,
                               EpiStore<float>{(float*)b.logits, V, w.bo, nullptr, 0}, st)));
    } else {
      SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(b.Xo, E, E), (const TS*)w.Wo, E, T * B, V,
                               EpiStore<TS>{(TS*)b.logits, V, w.bo, nullptr, 0}, st)));
    }
    SAT_PROF(3, st);
    // ---- loss ----------------------------------------------------------------------------------
    const size_t ce_smem = ce_smem_bytes(V);              // within the limit: checked before the first launch
    if (b.logits_f32) {
      auto k = ce_rows_kernel<float, TS, kExact>;
      if (ce_smem > 48 * 1024) SAT_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ce_smem));
      k<<<T * B, 256, ce_smem, st>>>((float*)b.logits, (TS*)b.dlogits, b.caps, b.lens, b.out + 4, b.row_loss, b.row_argmax, B,
                                     V0, V, caplen, b.label_smoothing, 1);
    } else {
      auto k = ce_rows_kernel<TS, TS, kExact>;
      if (ce_smem > 48 * 1024) SAT_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ce_smem));
      k<<<T * B, 256, ce_smem, st>>>((TS*)b.logits, (TS*)b.dlogits, b.caps, b.lens, b.out + 4, b.row_loss, b.row_argmax, B, V0, V,
                                     caplen, b.label_smoothing, 1);
    }
    SAT_COUNT_LAUNCH();
    SAT_LAUNCH_OK();
  }
  // per-CTA partials of sum (1-S)^2 live in the (by now dead) hp scratch buffer
  const int nparts = (B * L + 255) / 256;
  SAT_REQUIRE((int64_t)nparts <= (int64_t)B * NH3, "reduction scratch too small");
  alpha_sum_kernel<<<nparts, 256, 0, st>>>(b.alphas, b.S, b.hp, B, T, L);
  SAT_COUNT_LAUNCH();
  loss_finalize_kernel<<<1, 1024, 0, st>>>(b.row_loss, b.row_argmax, b.caps, b.lens, b.hp, nparts, B, T, L, caplen, b.att_gamma, b.out);
  SAT_COUNT_LAUNCH();
  SAT_LAUNCH_OK();
  (void)Bi;
  return 0;
}

int check_dims(const SatDims* d) {
  SAT_REQUIRE(d != nullptr, "dims is NULL");
  SAT_REQUIRE(d->dtype == SAT_F32 || d->dtype == SAT_BF16, "unknown dtype %d", d->dtype);
  SAT_REQUIRE(d->B > 0 && d->Bi > 0 && d->ncap > 0 && d->B == d->Bi * d->ncap, "B=%d must equal Bi*ncap=%d*%d", d->B, d->Bi,
              d->ncap);
  SAT_REQUIRE(d->L > 0 && d->T >= 0, "bad L=%d T=%d", d->L, d->T);
  SAT_REQUIRE(d->layers >= 0 && d->layers <= SAT_MAX_LAYERS, "decoder_layers %d not in 1..%d", d->layers, SAT_MAX_LAYERS);
  SAT_REQUIRE(d->D % 8 == 0 && d->A % 8 == 0 && d->E % 8 == 0 && d->H % 8 == 0 && d->V % 8 == 0 && d->D > 0 && d->A > 0 &&
                  d->E > 0 && d->H > 0 && d->V > 0,
              "storage dims D=%d A=%d E=%d H=%d V=%d must be positive multiples of 8 (pad the module's dims: SatDims.D0 ..)", d->D, d->A,
              d->E, d->H, d->V);
  SAT_REQUIRE(d->D0 >= 0 && d->D0 <= d->D && d->A0 >= 0 && d->A0 <= d->A && d->E0 >= 0 && d->E0 <= d->E && d->H0 >= 0 && d->H0 <= d->H &&
                  d->V0 >= 0 && d->V0 <= d->V,
              "true dims D0=%d A0=%d E0=%d H0=%d V0=%d must not exceed the storage dims", d->D0, d->A0, d->E0, d->H0, d->V0);
  return 0;
}

}  // namespace

extern "C" {

int sat_linear(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias, void* C, int64_t ldc, int32_t M,
               int32_t N, int32_t K, int32_t dtype, int32_t c_f32, int32_t use_tc, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  SAT_REQUIRE(A && W && C, "sat_linear: NULL operand");
  const bool tc = use_tc != 0;
  if (dtype == SAT_F32) {
    SAT_REQUIRE(c_f32, "sat_linear: fp32 operands need an fp32 output");
    return gemm_tn<float, float>(false, gemm_a1(A, lda, K), (const float*)W, ldw, M, N,
                                 EpiStore<float>{(float*)C, ldc, bias, nullptr, 0}, st);
  } else if (dtype == SAT_BF16) {
    SatNoPdlScope no_pdl;             // W is the caller's: it may be the output of the launch just before this one
    const int rc = c_f32 ? gemm_tn<bf16, bf16>(tc, gemm_a1(A, lda, K), (const bf16*)W, ldw, M, N,
                                               EpiStore<float>{(float*)C, ldc, bias, nullptr, 0}, st)
                         : gemm_tn<bf16, bf16>(tc, gemm_a1(A, lda, K), (const bf16*)W, ldw, M, N,
                                               EpiStore<bf16>{(bf16*)C, ldc, bias, nullptr, 0}, st);
    return rc;
  }
  SAT_REQUIRE(false, "sat_linear: unknown dtype %d", dtype);
}

int sat_prepare_images(const SatDims* d, const SatWeights* w, const void* ann, void* P, void* meanv, void* f1, float* init_out,
                       void* h0, float* c0, void* stream) {
  SAT_TRY(check_dims(d));
  SAT_REQUIRE(w && ann && P && meanv && f1 && init_out && h0 && c0, "sat_prepare_images: NULL pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (d->dtype == SAT_F32) return prepare_images_impl<float>(*d, *w, ann, P, meanv, f1, init_out, h0, c0, (int64_t)d->B * d->H, st);
  return prepare_images_impl<bf16>(*d, *w, ann, P, meanv, f1, init_out, h0, c0, (int64_t)d->B * d->H, st);
}

int sat_attention_step_fwd(const SatDims* d, const void* ann, const void* P, const float* wf, const float* hp, int64_t ldhp,
                           const int32_t* lens, int32_t t, float* alpha, int64_t ld_alpha, void* z, void* gz, void* beta,
                           int64_t ld_z, void* stream) {
  SAT_TRY(check_dims(d));
  SAT_REQUIRE(ann && P && wf && hp && alpha && z && gz, "sat_attention_step_fwd: NULL pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const float scale = (float)(1.0 / sqrt((double)d->L));
  SatNoPdlScope no_pdl;               // ann / P are the caller's: they may be the output of the launch just before this one
#define SAT_LAUNCH_ATT(TS, EX)                                                                                          \
  SAT_TRY((launch_attention_fwd<TS, EX>((const TS*)ann, (const TS*)P, wf, hp, ldhp, lens, t, d->B, d->ncap, d->L, d->D, d->A, \
                                        scale, alpha, ld_alpha, nullptr, (TS*)z, (TS*)gz, (TS*)beta, ld_z, st)))
  if (d->dtype == SAT_F32) {
    if (d->exact) SAT_LAUNCH_ATT(float, true); else SAT_LAUNCH_ATT(float, false);
  } else {
    if (d->exact) SAT_LAUNCH_ATT(bf16, true); else SAT_LAUNCH_ATT(bf16, false);
  }
#undef SAT_LAUNCH_ATT
  return 0;
}

int sat_cast_captions(const int64_t* caps64, const int64_t* lens64, int32_t* caps32, int32_t* lens32, int64_t n_caps, int64_t n_lens,
                      void* stream) {
  SAT_REQUIRE(caps64 && lens64 && caps32 && lens32 && n_caps >= 0 && n_lens >= 0, "sat_cast_captions: bad argument");
  const int64_t n = n_caps + n_lens;
  if (n == 0) return 0;
  cast_captions_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(caps64, lens64, caps32, lens32, n_caps, n_lens);
  SAT_COUNT_LAUNCH();
  SAT_LAUNCH_OK();
  return 0;
}

int sat_train_vocab_path(const SatDims* d, int32_t sampled) {
  SAT_TRY(check_dims(d));
  return train_vocab_path(*d, sampled != 0);
}

int sat_train_forward(const SatDims* d, const SatWeights* w, SatTrainBuffers* b, void* stream) {
  SAT_TRY(check_dims(d));
  SAT_REQUIRE(w && b, "sat_train_forward: NULL struct");
  SAT_REQUIRE(d->T > 0, "sat_train_forward: T must be > 0");
  SAT_REQUIRE(b->ann && b->caps && b->lens && b->tok && b->P && b->meanv && b->f1 && b->init_out && b->Xe && b->Gx && b->Hs && b->Cs &&
                  b->hp && b->Q && b->alphas && b->Z && b->GZ && b->Beta && b->Gates && b->Xo && b->row_loss &&
                  b->row_argmax && b->S && b->out,
              "sat_train_forward: NULL forward buffer");
  cudaStream_t st = (cudaStream_t)stream;
  if (d->dtype == SAT_F32) {
    return d->exact ? train_forward_impl<float, true>(*d, *w, *b, st) : train_forward_impl<float, false>(*d, *w, *b, st);
  }
  return d->exact ? train_forward_impl<bf16, true>(*d, *w, *b, st) : train_forward_impl<bf16, false>(*d, *w, *b, st);
}

}  // extern "C"
