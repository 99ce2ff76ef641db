// Batched greedy / beam decode driver (SAT.forward, model.py:237-472): every image of the batch advances
// together, beams live in device memory, and one step is
//   h-projection GEMM -> fused attention -> gate GEMM + LSTM epilogue -> deep-output GEMM -> vocabulary GEMM
//   -> row top-k (log-softmax, masks, parent score) -> per-image beam update -> state gather
// with no host synchronisation (the reference loops over images one at a time and syncs several times a step).
#include "sat_decode_kernels.cuh"
#include "sat_gemm.cuh"
#include "sat_attention_pipe.cuh"
#include "sat_kernels.cuh"
#include "sat_vocab_ce.cuh"

namespace {

constexpr size_t SMEM_LIMIT = 227 * 1024;
size_t topk_smem_bytes(int V) { return sizeof(float) * (size_t)(V + 40); }          // row_topk_kernel / row_topk_thresh_kernel
size_t sample_smem_bytes(int V) { return sizeof(float) * (size_t)(2 * V + 40); }    // row_sample_kernel

// Where the vocabulary stage of a decode runs (sat_decode_vocab_path): the shared-memory row kernels when a logits row fits, the
// fused candidate lists of the vocabulary GEMM's epilogue otherwise (or always under SAT_VOCAB_TOPK=1, for A/B timing); greedy
// decode on the tensor cores always takes the fused arg-max.  One choice per call, so that every step reads the same buffers.
int vocab_path(const SatDims& d, int k, int sample) {
  const int V = d.V;
  const bool fused_ok = d.dtype == SAT_BF16 && d.use_tc != 0 && d.exact == 0;
  if (fused_ok && k == 1 && sample == SAT_SAMPLE_BEAM) return SAT_VOCAB_PATH_GREEDY;
  static const int force_cand = getenv("SAT_VOCAB_TOPK") ? atoi(getenv("SAT_VOCAB_TOPK")) : 0;
  const bool rows_fit = topk_smem_bytes(V) <= SMEM_LIMIT && (sample != SAT_SAMPLE_MULTINOMIAL || sample_smem_bytes(V) <= SMEM_LIMIT);
  if (fused_ok && (force_cand != 0 || !rows_fit)) return SAT_VOCAB_PATH_CAND;
  SAT_REQUIRE(topk_smem_bytes(V) <= SMEM_LIMIT, "vocabulary of %d words needs %zu bytes of shared memory per row in the top-k kernel "
              "(limit 227 KB); decoding at this size needs the bf16 tensor-core path (bf16, use_tc, not exact)", V, topk_smem_bytes(V));
  SAT_REQUIRE(rows_fit, "vocabulary of %d words is too large for the multinomial sampler's shared memory; decoding at this size needs "
              "the bf16 tensor-core path (bf16, use_tc, not exact)", V);
  return SAT_VOCAB_PATH_ROWS;
}

template <typename TS, bool kExact>
int decode_impl(const SatDims& d, const SatWeights& w, SatDecodeBuffers& b, cudaStream_t st) {
  const int R = d.B, n_img = d.Bi, k = d.ncap, L = d.L, D = d.D, A = d.A, E = d.E, H = d.H, V = d.V;
  const int S = b.max_gen_length;
  const int NH3 = A + D + 4 * H;
  const bool tc = d.use_tc != 0;
  const TS* ann = (const TS*)b.ann;

  // once per image: P = ann * Wa^T, mean, InitLSTM
  {
    // first launch of the driver: no PDL attribute, so that operands written by the caller's preceding launch (the weight
    // pack kernel, the encoder) are complete and visible to every early (pre-wait) read of the kernels that follow
    SatNoPdlScope first_launch;
    SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(ann, D, D), (const TS*)w.Wa, D, n_img * L, A,
                             EpiStore<TS>{(TS*)b.P, A, nullptr, nullptr, 0}, st)));
  }
  const int NV = D / Vec16<TS>::N;
  mean_L_kernel<TS><<<dim3((NV + 31) / 32, n_img), 256, 0, st>>>(ann, (TS*)b.meanv, L, D, 0.0f, 0ull);
  SAT_COUNT_LAUNCH();
  SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(b.meanv, D, D), (const TS*)w.Wfact, D, n_img, E,
                           EpiStore<TS>{(TS*)b.f1, E, w.bfact, nullptr, 0}, st)));
  const int nl = d.layers > 1 ? d.layers : 1;
  const int64_t RH = (int64_t)R * H;             // one layer of the state arrays
  SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(b.f1, E, E), (const TS*)w.Winit, E, n_img, 2 * nl * H,
                           EpiStore<float>{b.init_out, 2 * nl * H, w.binit, nullptr, 0}, st)));
  init_state_decode_kernel<TS><<<(unsigned)((nl * RH + 255) / 256), 256, 0, st>>>(b.init_out, 2 * nl * H, (TS*)b.h, b.c, n_img, k,
                                                                                  d.H0 ? d.H0 : H, H, nl);
  SAT_COUNT_LAUNCH();
  decode_init_kernel<<<(R + 255) / 256, 256, 0, st>>>(b.cur_tok, b.alive, b.top_scores, b.kcur, b.fin_count, b.fin_len, R, n_img, k,
                                                      b.tokSTART, b.live_images);
  SAT_COUNT_LAUNCH();
  SAT_LAUNCH_OK();

  const float scale = (float)(1.0 / sqrt((double)L));
  const size_t topk_smem = topk_smem_bytes(V);
  const int V0 = d.V0 ? d.V0 : V;
  const int path = vocab_path(d, k, b.sample_method);
  if (path < 0) return path;
  const bool fused_operands = tc::operands_ok(gemm_a1(b.xo, E, E), w.Wo, E);
  // greedy on the tensor cores: soft-max statistics and the best word come out of the vocabulary GEMM's epilogue
  const bool fuse_greedy = path == SAT_VOCAB_PATH_GREEDY && b.topk_stats != nullptr && fused_operands;
  // beam search / sampling above the row kernels' sizes: per-tile candidate lists come out of the epilogue
  const bool fuse_cand = path == SAT_VOCAB_PATH_CAND;
  SAT_REQUIRE(!fuse_cand || (fused_operands && b.topk_stats && b.tile_val && b.tile_idx &&
                             (b.sample_method != SAT_SAMPLE_MULTINOMIAL || (b.tile_key && b.topk_stats2))),
              "sat_decode: the fused candidate path needs aligned operands and the topk_stats / tile_* buffers");
  SAT_REQUIRE(fuse_greedy || fuse_cand || topk_smem <= SMEM_LIMIT, "vocabulary of %d words needs %zu bytes of shared memory per row in "
              "the top-k kernel (limit 227 KB)", V, topk_smem);
  SAT_REQUIRE(fuse_greedy || fuse_cand || b.logits != nullptr, "sat_decode: logits buffer missing");
  // candidate selection: threshold kernel (SAT_TOPK_MODE=0 forces the plain scan kernel for A/B runs)
  static const int topk_mode = getenv("SAT_TOPK_MODE") ? atoi(getenv("SAT_TOPK_MODE")) : 1;
  auto topk_k = (topk_mode == 0 || k == 1) ? row_topk_kernel : row_topk_thresh_kernel;      // greedy: one scan is already minimal
  if (!fuse_greedy && !fuse_cand && topk_smem > 48 * 1024) SAT_CUDA(cudaFuncSetAttribute(topk_k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)topk_smem));
  // sampling decoders (sample_method "multinomial" / "topk", model.py:360-379) and decoder noise (model.py:322-324)
  const int sample = b.sample_method;
  const int kcap = b.kcap > 0 ? b.kcap : k;
  const int kk_req = sample == SAT_SAMPLE_TOPK ? b.sample_topk : 0;
  const bool noisy = b.decoder_noise != 0.0f;
  SAT_REQUIRE(sample == SAT_SAMPLE_BEAM || (b.cand_key != nullptr || sample == SAT_SAMPLE_TOPK), "sat_decode: cand_key buffer missing");
  SAT_REQUIRE(!noisy || b.h_noisy != nullptr, "sat_decode: h_noisy buffer missing");
  const size_t samp_smem = sample_smem_bytes(V);
  if (sample == SAT_SAMPLE_MULTINOMIAL && !fuse_cand && samp_smem > 48 * 1024)
    SAT_CUDA(cudaFuncSetAttribute(row_sample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)samp_smem));
  BeamParams bp{k, V, S, b.tokEND, b.rescore, b.reward, S + 1, kcap, sample, b.sample_topk, b.sample_seed};
  const int64_t hist_sz = (int64_t)R * (S + 1);

  // k == 1 (greedy): a live row always continues from itself, so the post-LSTM state is used in place (buffer ping-pong)
  // instead of being gathered by source row
  void* h_cur = b.h; float* c_cur = b.c; void* h_nxt = b.hn; float* c_nxt = b.cn;
  for (int step = 0; step <= S; ++step) {
    // every image has used up its beams (model.py:419,436): the steps not yet queued would only run dead rows
    if (step > 0 && b.done_host != nullptr && b.live_images != nullptr && *b.done_host == b.call_id) break;
    const TS* h_top = (const TS*)h_cur + (nl - 1) * RH;      // attention, beta gate and the output layer read the top layer (model.py:299-300,327)
    if (!noisy && nl == 1) {
      SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(h_cur, H, H), (const TS*)w.Whcat, H, R, NH3, EpiStore<float>{b.hp, NH3, w.bhcat, nullptr, 0},
                               st)));
    } else {
      // decoder noise: attention and the beta gate read the clean state, the recurrent projections W_hh (h + noise) the noisy
      // one (every layer's state gets noise, model.py:324)
      if (noisy) {
        SAT_CUDA(sat_launch_pdl(noisy_state_kernel<TS>, dim3((unsigned)((nl * RH + 255) / 256)), dim3(256), 0, st, (const TS*)h_cur,
                                (TS*)b.h_noisy, nl * RH, b.decoder_noise / (float)(step + 1), b.sample_seed, step));
        SAT_COUNT_LAUNCH();
      }
      SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(h_top, H, H), (const TS*)w.Whcat, H, R, A + D, EpiStore<float>{b.hp, NH3, w.bhcat, nullptr, 0},
                               st)));
      SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(noisy ? (const TS*)b.h_noisy : (const TS*)h_cur, H, H), (const TS*)w.Whcat + (int64_t)(A + D) * H, H,
                               R, 4 * H, EpiStore<float>{b.hp + A + D, NH3, nullptr, nullptr, 0}, st)));
    }
    SAT_PROF(1, st);
    SAT_TRY((launch_attention_fwd<TS, kExact>(ann, (const TS*)b.P, w.wf, b.hp, NH3, b.alive, 0, R, k, L, D, A, scale,
                                              b.alpha_all + (int64_t)step * R * L, L, nullptr, (TS*)b.z, (TS*)b.gz,
                                              (TS*)nullptr, D, st, /*lens_dyn=*/1)));
    SAT_PROF(1, st);
    EpiLstm<TS, kExact> epi{b.GxV, 4 * H, b.hp + A + D, NH3, (const TS*)h_cur, c_cur, (TS*)h_nxt, c_nxt, H, H,
                            (TS*)nullptr, 0, b.alive, 0, b.cur_tok};
    SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(b.gz, D, D), (const TS*)w.Wihz, D, R, 4 * H, epi, st)));
    for (int l = 1; l < nl; ++l) {      // stacked layers: input = the new state of the layer below
      const TS* hl = (noisy ? (const TS*)b.h_noisy : (const TS*)h_cur) + l * RH;
      EpiLstm<TS, kExact> epl{w.bgl[l - 1], 0, nullptr, 0, (const TS*)h_cur + l * RH, c_cur + l * RH, (TS*)h_nxt + l * RH, c_nxt + l * RH, H, H,
                              (TS*)nullptr, 0, b.alive, 0, nullptr};
      SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a2((const TS*)h_nxt + (l - 1) * RH, H, H, hl, H, H), (const TS*)w.Wl[l - 1], 2 * H, R, 4 * H, epl, st)));
    }
    SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a2((const TS*)h_nxt + (nl - 1) * RH, H, H, b.z, D, D), (const TS*)w.Whozo, H + D, R, E,
                             EpiTanhAdd<TS, kExact>{(const TS*)w.Emb, (TS*)b.xo, E, b.cur_tok, d.plain_output, 0.0f, 0ull, 0}, st)));
    SAT_PROF(3, st);
    if (fuse_greedy) {
      tc::VocabArgs va{};
      va.bias = w.bo; va.V0 = V0; va.NT = (V + 127) / 128; va.stats = reinterpret_cast<float4*>(b.topk_stats);
      va.alive = b.alive; va.inv_temp = 1.0f / b.temps[step];
      va.tokPAD = b.tokPAD; va.tokSTART = b.tokSTART; va.tokEND = b.tokEND; va.tokUNK = b.tokUNK; va.step0 = step == 0;
      SAT_TRY((tc::launch_vocab<tc::VOCAB_GREEDY>(gemm_a1(b.xo, E, E), (const bf16*)w.Wo, E, R, V, va, st)));
      SAT_PROF(3, st);
      SAT_CUDA(sat_launch_pdl(tc::greedy_finalize_kernel, dim3((R + 7) / 8), dim3(256), 0, st, (const float4*)va.stats, va.NT,
                              (const int32_t*)b.alive, (const float*)b.top_scores, R, (int)(step == 0), b.cand_val, b.cand_idx));
      SAT_COUNT_LAUNCH();
    } else if (fuse_cand) {
      const bool samp = sample == SAT_SAMPLE_MULTINOMIAL && step > 0;
      tc::VocabArgs va{};
      va.bias = w.bo; va.V0 = V0; va.NT = (V + 127) / 128; va.stats = reinterpret_cast<float4*>(b.topk_stats);
      va.alive = b.alive; va.inv_temp = 1.0f / b.temps[step];
      va.tokPAD = b.tokPAD; va.tokSTART = b.tokSTART; va.tokEND = b.tokEND; va.tokUNK = b.tokUNK; va.step0 = step == 0;
      va.kcap = kcap; va.cand_x = b.tile_val; va.cand_col = b.tile_idx; va.cand_key = b.tile_key;
      va.stats2 = reinterpret_cast<float2*>(b.topk_stats2); va.sharp = 20.0f / (float)(step > 0 ? step : 1);
      va.seed = b.sample_seed; va.step = step;
      if (samp) SAT_TRY((tc::launch_vocab<tc::VOCAB_SAMPLE>(gemm_a1(b.xo, E, E), (const bf16*)w.Wo, E, R, V, va, st)));
      else SAT_TRY((tc::launch_vocab<tc::VOCAB_TOPK>(gemm_a1(b.xo, E, E), (const bf16*)w.Wo, E, R, V, va, st)));
      SAT_PROF(3, st);
      SAT_CUDA(sat_launch_pdl(samp ? tc::cand_finalize_kernel<true> : tc::cand_finalize_kernel<false>, dim3((R + 7) / 8), dim3(256), 0,
                              st, (const float4*)va.stats, (const float2*)va.stats2, (const float*)b.tile_val, (const float*)b.tile_key,
                              (const int32_t*)b.tile_idx, va.NT, kcap, (const float*)b.top_scores, (const int32_t*)b.kcur, k,
                              samp ? 0 : kk_req, R, (int)(step == 0), b.cand_key, b.cand_val, b.cand_idx));
      SAT_COUNT_LAUNCH();
    } else {
      SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(b.xo, E, E), (const TS*)w.Wo, E, R, V, EpiStore<float>{b.logits, V, w.bo, nullptr, 0}, st)));
      SAT_PROF(3, st);
      if (sample == SAT_SAMPLE_MULTINOMIAL && step > 0) {
        SAT_CUDA(sat_launch_pdl(row_sample_kernel, dim3(R), dim3(256), samp_smem, st, (const float*)b.logits, (const float*)b.top_scores,
                                (const int32_t*)b.kcur, k, kcap, V, step, b.temps[step], b.tokPAD, b.tokSTART, b.sample_seed, b.cand_key,
                                b.cand_val, b.cand_idx));
      } else {
        SAT_CUDA(sat_launch_pdl(topk_k, dim3(R), dim3(256), topk_smem, st, (const float*)b.logits, (const float*)b.top_scores,
                                (const int32_t*)b.kcur, k, kcap, kk_req, V, step, b.temps[step], b.tokPAD, b.tokSTART, b.tokEND, b.tokUNK,
                                b.cand_val, b.cand_idx));
      }
      SAT_COUNT_LAUNCH();
    }
    const int in = step & 1, out = in ^ 1;
    SAT_CUDA(sat_launch_pdl(beam_update_kernel, dim3(n_img), dim3(32), 0, st, bp, step, (const float*)b.cand_val, (const float*)b.cand_key,
                            (const int32_t*)b.cand_idx, b.kcur, b.top_scores, b.cur_tok, b.src_row, b.alive,
                            (const int32_t*)(b.tok_hist + in * hist_sz), (const int32_t*)(b.asrc_hist + in * hist_sz),
                            b.tok_hist + out * hist_sz, b.asrc_hist + out * hist_sz, b.fin_tokens, b.fin_asrc, b.fin_len, b.fin_score,
                            b.fin_ppl, b.fin_count, b.live_images, b.done_host, (int)b.call_id));
    SAT_COUNT_LAUNCH();
    if (k == 1) {
      void* th = h_cur; h_cur = h_nxt; h_nxt = th;
      float* tcp = c_cur; c_cur = c_nxt; c_nxt = tcp;
    } else {
      SAT_CUDA(sat_launch_pdl(gather_state_kernel<TS>, dim3((unsigned)((nl * RH + 255) / 256)), dim3(256), 0, st,
                              (const TS*)b.hn, (const float*)b.cn, (const int32_t*)b.src_row, (const int32_t*)b.alive, (TS*)b.h, b.c, R,
                              H, nl));
      SAT_COUNT_LAUNCH();
    }
  }
  return 0;
}

}  // namespace

extern "C" {

int sat_decode_prepare_weights(const SatDims* d, const SatWeights* w, float* GxV, void* stream) {
  SAT_REQUIRE(d && w && GxV && w->Emb && w->Wihe && w->bg, "sat_decode_prepare_weights: NULL pointer");
  cudaStream_t st = (cudaStream_t)stream;
  SatNoPdlScope no_pdl;               // the packed weights may be the output of the launch just before this one (sat_pack_weights)
  const bool tc = d->use_tc != 0;
  if (d->dtype == SAT_F32)
    return gemm_tn<float, float>(false, gemm_a1(w->Emb, d->E, d->E), (const float*)w->Wihe, d->E, d->V, 4 * d->H,
                                 EpiStore<float>{GxV, 4 * d->H, w->bg, nullptr, 0}, st);
  return gemm_tn<bf16, bf16>(tc, gemm_a1(w->Emb, d->E, d->E), (const bf16*)w->Wihe, d->E, d->V, 4 * d->H,
                             EpiStore<float>{GxV, 4 * d->H, w->bg, nullptr, 0}, st);
}

int sat_decode_vocab_path(const SatDims* d, int k, int sample_method, int sample_topk) {
  SAT_REQUIRE(d != nullptr, "sat_decode_vocab_path: NULL dims");
  SAT_REQUIRE(k >= 1 && k <= 32, "sat_decode_vocab_path: beam width %d outside 1..32", k);
  SAT_REQUIRE(sample_method >= 0 && sample_method <= 2, "sat_decode_vocab_path: unknown sample_method %d", sample_method);
  SAT_REQUIRE(sample_method != SAT_SAMPLE_TOPK || (sample_topk >= 1 && sample_topk <= 32),
              "sat_decode_vocab_path: the topk sampler needs 1 <= sample_topk <= 32");
  return vocab_path(*d, k, sample_method);
}

int sat_decode(const SatDims* d, const SatWeights* w, SatDecodeBuffers* b, void* stream) {
  SAT_REQUIRE(d && w && b, "sat_decode: NULL struct");
  SAT_REQUIRE(d->dtype == SAT_F32 || d->dtype == SAT_BF16, "unknown dtype %d", d->dtype);
  SAT_REQUIRE(d->B == d->Bi * d->ncap && d->ncap == b->k && b->k >= 1 && b->k <= 32, "sat_decode: rows %d != n_img %d * k %d (k <= 32)",
              d->B, d->Bi, b->k);
  SAT_REQUIRE(d->D % 8 == 0 && d->A % 8 == 0 && d->E % 8 == 0 && d->H % 8 == 0 && d->V % 8 == 0, "storage dims must be multiples of 8");
  SAT_REQUIRE(d->H0 >= 0 && d->H0 <= d->H && d->V0 >= 0 && d->V0 <= d->V, "true dims must not exceed the storage dims");
  SAT_REQUIRE(b->max_gen_length >= 1 && b->temps, "sat_decode: max_gen_length >= 1 and temps required");
  SAT_REQUIRE(b->sample_method >= 0 && b->sample_method <= 2, "sat_decode: unknown sample_method %d", b->sample_method);
  SAT_REQUIRE(b->sample_method != 2 || (b->sample_topk >= 1 && b->sample_topk <= 32 && b->kcap >= b->sample_topk && b->kcap >= b->k),
              "sat_decode: the topk sampler needs 1 <= sample_topk <= 32 and kcap >= max(k, sample_topk)");
  SAT_REQUIRE(b->kcap == 0 || b->kcap >= b->k, "sat_decode: kcap %d < k %d", b->kcap, b->k);
  SAT_REQUIRE(b->k + 4 <= (d->V0 ? d->V0 : d->V), "sat_decode: beam width %d too large for vocab %d", b->k, d->V0 ? d->V0 : d->V);
  SAT_REQUIRE(b->ann && b->P && b->meanv && b->f1 && b->init_out && b->GxV && b->h && b->c && b->hn && b->cn && b->hp && b->z &&
                  b->gz && b->xo && (b->logits || b->topk_stats) && b->alpha_all && b->cand_val && b->cand_idx && b->tok_hist && b->asrc_hist &&
                  b->top_scores && b->cur_tok && b->src_row && b->alive && b->kcur && b->fin_tokens && b->fin_asrc && b->fin_len &&
                  b->fin_score && b->fin_ppl && b->fin_count,
              "sat_decode: NULL buffer");
  cudaStream_t st = (cudaStream_t)stream;
  if (d->dtype == SAT_F32) return d->exact ? decode_impl<float, true>(*d, *w, *b, st) : decode_impl<float, false>(*d, *w, *b, st);
  return d->exact ? decode_impl<bf16, true>(*d, *w, *b, st) : decode_impl<bf16, false>(*d, *w, *b, st);
}

}  // extern "C"
