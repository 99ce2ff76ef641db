// Hand-written BPTT of the teacher-forced SAT decoder step (SURVEY.md appendix E; what autograd
// derives from model.py:510-548 when PL calls loss.backward()).
//
// Only the dh/dc/dz chain is sequential; it costs three launches per step:
//   lstm_bwd_step (elementwise)  ->  GEMM dgz = dG * Wihz  ->  fused attention backward  ->
//   GEMM dh = [dq | dbeta_pre | dG] * [W_h ; W_beta ; W_hh]   (one GEMM, K = A+D+4H)
// Everything else is hoisted to whole-sequence GEMMs over T*B rows (dpre, dHZ, dXe, d_ann), and
// the parameter gradients are plain reductions over (t,b) of the buffers written here.
#include "sat_attention_pipe.cuh"
#include "sat_gemm.cuh"
#include "sat_kernels.cuh"

namespace {

template <typename TS, bool kExact>
int train_backward_impl(const SatDims& d, const SatWeights& w, SatTrainBuffers& b, cudaStream_t st) {
  const int B = d.B, Bi = d.Bi, L = d.L, D = d.D, A = d.A, E = d.E, H = d.H, V = d.V, T = d.T;
  const int NH3 = A + D + 4 * H;
  const bool tc = d.use_tc != 0;
  const TS* ann = (const TS*)b.ann;
  const int M = T * B;

  // dpre = g * (dlogits * Wo) * (1 - Xo^2)            [M,E]
  {
    SatNoPdlScope first_launch;       // first launch of the driver: everything the caller queued before is complete and visible
    SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(b.dlogits, V, V), (const TS*)w.WoT, V, M, E,
                             EpiDpre<TS>{(const TS*)b.Xo, (TS*)b.dpre, E, b.gscale, d.plain_output, b.dropout_p, b.dropout_seed}, st)));
  }
  // dHZ = dpre * [W_ho | W_zo]                         [M,H+D]
  SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(b.dpre, E, E), (const TS*)w.WhozoT, E, M, H + D,
                           EpiStore<float>{b.dHZ, H + D, nullptr, nullptr, 0}, st)));

  // split-K factors of the skinny per-step GEMMs (tensor-core core only; partials are summed by their consumers)
  const int NH3_ = A + D + 4 * H;
  const int nl = d.layers > 1 ? d.layers : 1;
  const int64_t LS = (int64_t)(T + 1) * B * H, GS = (int64_t)T * B * 4 * H;     // layer strides of Hs/Cs and Gates/dGl
  const int64_t BH = (int64_t)B * H;
  const bool tc_dgz = gemm_tn_uses_tc<TS, TS>(tc, gemm_a1((const TS*)b.DY + A + D, NH3_, 4 * H), (const TS*)w.WihzT, 4 * H, B, D);
  const int sk_dgz = tc_dgz ? tc::pick_splitk(B, D, 4 * H) : 1;
  // one layer: dh = [dq | dbeta_pre | dG] * [W_h ; W_beta ; W_hh] in one GEMM.  Stacked layers: q / beta read the TOP layer's
  // state and the recurrent projection layer 0's, so the GEMM splits in two (dhq: K = A+D, dh: K = 4H).
  const int k_dh = nl == 1 ? NH3_ : 4 * H;
  const TS* w_dh = (const TS*)w.WhcatT + (nl == 1 ? 0 : A + D);
  const bool tc_dh = gemm_tn_uses_tc<TS, TS>(tc, gemm_a1((const TS*)b.DY + (nl == 1 ? 0 : A + D), NH3_, k_dh), w_dh, NH3_, B, H);
  const int sk_dh = tc_dh ? tc::pick_splitk(B, H, k_dh) : 1;
  int sk_hq = 1, sk_x = 1;
  if (nl > 1) {
    SAT_REQUIRE(b.dGl && b.dxl && b.dhq, "sat_train_backward: decoder_layers > 1 needs the dGl / dxl / dhq buffers");
    for (int l = 1; l < nl; ++l) SAT_REQUIRE(w.WlT[l - 1], "sat_train_backward: transposed weights of LSTM layer %d missing", l);
    if (gemm_tn_uses_tc<TS, TS>(tc, gemm_a1(b.DY, NH3_, A + D), (const TS*)w.WhcatT, NH3_, B, H)) sk_hq = tc::pick_splitk(B, H, A + D);
    if (gemm_tn_uses_tc<TS, TS>(tc, gemm_a1(b.dGl, 4 * H, 4 * H), (const TS*)w.WlT[0], 4 * H, B, 2 * H)) sk_x = tc::pick_splitk(B, 2 * H, 4 * H);
    SAT_CUDA(cudaMemsetAsync(b.dhq, 0, sizeof(float) * (size_t)sk_hq * BH, st));
    SAT_CUDA(cudaMemsetAsync(b.dxl, 0, sizeof(float) * (size_t)(nl - 1) * 16 * BH * 2, st));
  }
  SAT_CUDA(cudaMemsetAsync(b.dh, 0, sizeof(float) * (size_t)sk_dh * BH, st));
  SAT_CUDA(cudaMemsetAsync(b.dc, 0, sizeof(float) * (size_t)nl * BH, st));
  auto dxl_of = [&](int l) { return b.dxl + (int64_t)(l - 1) * 16 * BH * 2; };   // [16][B][2H] partials of layer l >= 1
  const bool dann_tc = tc && b.dP16 != nullptr && !std::is_same<TS, float>::value;
  const float scale = (float)(1.0 / sqrt((double)L));
  // pipelined attention backward: saves de_t per step and dP is rebuilt once after the loop (dP_deferred_kernel);
  // the plain kernel accumulates dP step by step and needs it zeroed
  const int dpd_cols = dP_deferred_cols(T, A);
  const bool att_pipe = attention_bwd_pipe_ok<TS>(D, A) && b.de != nullptr && A % 4 == 0 && dpd_cols > 0;
  if (!att_pipe) {
    SAT_CUDA(cudaMemsetAsync(b.dP, 0, sizeof(float) * (size_t)B * L * A, st));
    if (dann_tc) SAT_CUDA(cudaMemsetAsync(b.dP16, 0, sizeof(TS) * (size_t)B * L * A, st));
  }
  const size_t att_smem = att_pipe ? attention_bwd_pipe_smem(L, D, A) : attention_bwd_smem(L, D, A);
  // instantiation by attention_dim: 128-column slices per lane (pipelined: 2 / 4 / 8; step-by-step kernel: 4 / 8)
  const int ka = attp_ka(A);
  auto att_k = att_pipe ? (ka == 2 ? attention_step_bwd_pipe_kernel<TS, kExact, ATTP_BWD_CW, 2>
                                   : (ka == 4 ? attention_step_bwd_pipe_kernel<TS, kExact, ATTP_BWD_CW, 4>
                                              : attention_step_bwd_pipe_kernel<TS, kExact, ATTP_BWD_CW, 8>))
                        : (A <= 512 ? attention_step_bwd_kernel<TS, kExact, 4> : attention_step_bwd_kernel<TS, kExact, 8>);
  const int att_threads = att_pipe ? ATTP_BWD_CW * 32 + 32 : ATT_THREADS;
  if (att_smem > 48 * 1024) SAT_CUDA(cudaFuncSetAttribute(att_k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)att_smem));

  struct L2Scope {
    L2Scope(const void* p, size_t n) {
      const size_t lim = sat_l2_persist_limit();
      if (lim > 0 && n > 0) { sat_l2_window().ptr = p; sat_l2_window().bytes = n < lim ? n : lim; sat_l2_window().hit_ratio = n <= lim ? 1.0f : (float)lim / (float)n; }
    }
    ~L2Scope() { sat_l2_window().ptr = nullptr; sat_l2_window().bytes = 0; }
  } l2scope(b.ann, sizeof(TS) * (size_t)Bi * L * D);
  for (int t = T - 1; t >= 0; --t) {
    TS* DY_t = (TS*)b.DY + (int64_t)t * B * NH3;
    const float* dHZ_t = b.dHZ + (int64_t)t * B * (H + D);
    for (int l = nl - 1; l >= 1; --l) {
      // layer l: grad wrt its new state = its own recurrent use at t+1 (dxl[l][:, H:], written at step t+1) + the layer
      // above's input use at this step (dxl[l+1][:, :H]) or, for the top layer, q / beta at t+1 (dhq) and the output layer
      DhSrc src{{dxl_of(l) + H, l < nl - 1 ? dxl_of(l + 1) : b.dhq, b.dc}, {sk_x, l < nl - 1 ? sk_x : sk_hq, 0},
                {2 * BH, l < nl - 1 ? 2 * BH : BH, 0}, {2 * H, l < nl - 1 ? 2 * H : H, 0}};
      TS* dG_l = (TS*)b.dGl + (l - 1) * GS + (int64_t)t * B * 4 * H;
      SAT_CUDA(sat_launch_pdl(lstm_bwd_step_kernel<TS, kExact>, dim3((B * H + 255) / 256), dim3(256), 0, st,
          (const TS*)b.Gates + l * GS + (int64_t)t * B * 4 * H, (const float*)(b.Cs + l * LS + (int64_t)t * BH),
          (const float*)(b.Cs + l * LS + (int64_t)(t + 1) * BH), src, l == nl - 1 ? dHZ_t : (const float*)nullptr, (int64_t)(H + D),
          b.dc + l * BH, dG_l, (int64_t)(4 * H), (const int32_t*)b.lens, t, B, H));
      SAT_COUNT_LAUNCH();
      // [d input | d own previous state] = dG_l * [W_ih_l | W_hh_l]
      SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(dG_l, 4 * H, 4 * H), (const TS*)w.WlT[l - 1], 4 * H, B, 2 * H,
                               EpiStore<float>{dxl_of(l), 2 * H, nullptr, nullptr, 0, 2 * BH}, st, sk_x)));
    }
    {
      DhSrc src{{b.dh, nl > 1 ? dxl_of(1) : b.dc, b.dc}, {sk_dh, nl > 1 ? sk_x : 0, 0}, {BH, 2 * BH, 0}, {H, 2 * H, 0}};
      SAT_CUDA(sat_launch_pdl(lstm_bwd_step_kernel<TS, kExact>, dim3((B * H + 255) / 256), dim3(256), 0, st,
          (const TS*)b.Gates + (int64_t)t * B * 4 * H, (const float*)(b.Cs + (int64_t)t * BH), (const float*)(b.Cs + (int64_t)(t + 1) * BH), src,
          nl == 1 ? dHZ_t : (const float*)nullptr, (int64_t)(H + D), b.dc, DY_t + A + D, (int64_t)NH3, (const int32_t*)b.lens, t, B, H));
    }
    SAT_COUNT_LAUNCH();
    // dgz = dG * Wihz     (A operand: DY_t[:, A+D:], K = 4H)
    SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(DY_t + A + D, NH3, 4 * H), (const TS*)w.WihzT, 4 * H, B, D,
                             EpiStore<float>{b.dgz, D, nullptr, nullptr, 0, (int64_t)B * D}, st, sk_dgz)));
    SAT_PROF(2, st);
    SAT_CUDA(sat_launch_pdl(att_k, dim3(B), dim3(att_threads), att_smem, st, ann, (const TS*)b.P, w.wf, b.Q + (int64_t)t * B * A, b.alphas + (int64_t)t * L,
                                            (int64_t)T * L, b.S, (const TS*)b.Z + (int64_t)t * B * D,
                                            (const TS*)b.Beta + (int64_t)t * B * D, b.dgz, sk_dgz, (int64_t)B * D, dHZ_t + H, H + D, b.lens,
                                            t, d.ncap,
                                            B, L, D, A, scale, b.att_gamma, b.gscale,
                                            b.dalpha_ext ? b.dalpha_ext + (int64_t)t * L : nullptr, b.dP, dann_tc ? (TS*)b.dP16 : (TS*)nullptr, (TS*)b.dZ + (int64_t)t * B * D,
                                            DY_t, NH3, b.dwf_part + (int64_t)t * B * A,
                                            b.de ? b.de + (int64_t)t * B * L : (float*)nullptr));
    SAT_PROF(2, st);
    SAT_COUNT_LAUNCH();
    // dh = [dq | dbeta_pre | dG] * [W_h ; W_beta ; W_hh]   (rows inactive at t keep their dh)
    // (rows not active at t have an all-zero DY row, and their dh is still zero in backward order, so a plain store is exact)
    SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(DY_t + (nl == 1 ? 0 : A + D), NH3, k_dh), w_dh, NH3, B, H,
                             EpiStore<float>{b.dh, H, nullptr, nullptr, 0, BH}, st, sk_dh)));
    if (nl > 1)
      SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1(DY_t, NH3, A + D), (const TS*)w.WhcatT, NH3, B, H,
                               EpiStore<float>{b.dhq, H, nullptr, nullptr, 0, BH}, st, sk_hq)));
  }

  if (att_pipe) {
    const size_t sm = sizeof(float) * (size_t)T * (dpd_cols + DPD_ROWS);
    auto kp = dpd_cols == A ? dP_deferred_kernel<TS, kExact, false> : dP_deferred_kernel<TS, kExact, true>;
    if (sm > 48 * 1024) SAT_CUDA(cudaFuncSetAttribute(kp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    kp<<<dim3((L + DPD_ROWS - 1) / DPD_ROWS, B, (A + dpd_cols - 1) / dpd_cols), 256, sm, st>>>(
        (const TS*)b.P, w.wf, b.Q, b.de, b.lens, d.ncap, B, L, A, T, b.dP, dann_tc ? (TS*)b.dP16 : (TS*)nullptr, dpd_cols);
    SAT_COUNT_LAUNCH();
    SAT_LAUNCH_OK();
  }
  // dXe = dG * Wihe + dpre                               [M,E]
  SAT_TRY((gemm_tn<TS, TS>(tc, gemm_a1((const TS*)b.DY + A + D, NH3, 4 * H), (const TS*)w.WiheT, 4 * H, M, E,
                           EpiStore<float, TS>{b.dXe, E, nullptr, d.plain_output ? (const TS*)nullptr : (const TS*)b.dpre, E}, st)));

  if (b.emb_dropout_p > 0.0f) {   // embedding_dropout backward: dXe is the grad wrt the dropped embeddings
    dropout_bwd_kernel<<<(unsigned)(((int64_t)M * E + 255) / 256), 256, 0, st>>>(b.dXe, (int64_t)M * E, b.emb_dropout_p, b.dropout_seed, 2u);
    SAT_COUNT_LAUNCH();
  }
  // initial state: inverse of the [B,2H] -> [2,B,H] reinterpretation, then the two Linear layers
  const bool init_tc = tc && !std::is_same<TS, float>::value && b.d_init_out16 != nullptr && b.df116 != nullptr;
  const int IO = 2 * nl * H;
  InitBwdSrc isrc{};
  for (int l = 0; l < nl; ++l)
    for (int q = 0; q < 2; ++q) { isrc.p[l][q] = b.dc; isrc.ns[l][q] = 0; isrc.stride[l][q] = 0; isrc.ld[l][q] = 0; }
  // grad wrt h0 of layer l: what its step-0 consumers left behind (recurrent projection; for the top layer also q / beta)
  isrc.p[0][0] = b.dh; isrc.ns[0][0] = sk_dh; isrc.stride[0][0] = BH; isrc.ld[0][0] = H;
  for (int l = 1; l < nl; ++l) { isrc.p[l][0] = dxl_of(l) + H; isrc.ns[l][0] = sk_x; isrc.stride[l][0] = 2 * BH; isrc.ld[l][0] = 2 * H; }
  if (nl > 1) { isrc.p[nl - 1][1] = b.dhq; isrc.ns[nl - 1][1] = sk_hq; isrc.stride[nl - 1][1] = BH; isrc.ld[nl - 1][1] = H; }
  init_state_bwd_kernel<<<(Bi * IO + 255) / 256, 256, 0, st>>>(isrc, b.dc, H, BH, b.d_init_out, init_tc ? (bf16*)b.d_init_out16 : (bf16*)nullptr,
                                                               IO, B, d.H0 ? d.H0 : H, d.ncap, nl);
  SAT_COUNT_LAUNCH();
  SAT_LAUNCH_OK();
  if (init_tc) {
    SAT_TRY((gemm_tn<TS, TS>(true, gemm_a1(b.d_init_out16, IO, IO), (const TS*)w.WinitT, IO, Bi, E,
                             EpiStoreDual<TS>{b.df1, (TS*)b.df116, E}, st)));
    SAT_TRY((gemm_tn<TS, TS>(true, gemm_a1(b.df116, E, E), (const TS*)w.WfactT, E, Bi, D,
                             EpiStore<float>{b.dmean, D, nullptr, nullptr, 0}, st)));
  } else {
    SAT_TRY((gemm_tn<float, TS>(false, gemm_a1(b.d_init_out, IO, IO), (const TS*)w.WinitT, IO, Bi, E,
                                EpiStore<float>{b.df1, E, nullptr, nullptr, 0}, st)));
    SAT_TRY((gemm_tn<float, TS>(false, gemm_a1(b.df1, E, E), (const TS*)w.WfactT, E, Bi, D,
                                EpiStore<float>{b.dmean, D, nullptr, nullptr, 0}, st)));
  }
  if (b.dropout_p > 0.0f) {       // InitLSTM dropout on the mean (model.py:78)
    dropout_bwd_kernel<<<(unsigned)(((int64_t)Bi * D + 255) / 256), 256, 0, st>>>(b.dmean, (int64_t)Bi * D, b.dropout_p, b.dropout_seed, 1u);
    SAT_COUNT_LAUNCH();
  }
  // d_ann[b,l,:] = dP[b,l,:] * Wa + sum_t alpha[b,t,l] dZ[t,b,:] + dmean[img]/(L*ncap)
  // (for ncap > 1 the buffer holds per-caption rows [B,L,D]; the host sums the ncap rows of an image)
  EpiDAnn<TS> epi_dann{(TS*)b.d_ann, b.alphas, (const TS*)b.dZ, b.dmean, B, T, L, D, d.ncap, 1.0f / ((float)L * (float)d.ncap)};
  if (dann_tc) {
    // tensor-core path: the attention part + mean term is written to d_ann itself (operand dtype), then dP16 * Wa is
    // added in place by the GEMM epilogue (every element is read and written by the same thread)
    const size_t sm = sizeof(float) * ((size_t)T * DANN_DC + (size_t)T * L);
    auto kd = dann_alpha_kernel<TS, TS>;
    if (sm > 48 * 1024) SAT_CUDA(cudaFuncSetAttribute(kd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    kd<<<dim3(B, (D + DANN_DC - 1) / DANN_DC), 256, sm, st>>>(b.alphas, (const TS*)b.dZ, b.dmean, (TS*)b.d_ann, B, T, L, D, d.ncap,
                                                              1.0f / ((float)L * (float)d.ncap));
    SAT_COUNT_LAUNCH();
    SAT_LAUNCH_OK();
    SAT_TRY((gemm_tn<TS, TS>(true, gemm_a1(b.dP16, A, A), (const TS*)w.WaT, A, B * L, D,
                             EpiStore<TS, TS>{(TS*)b.d_ann, D, nullptr, (const TS*)b.d_ann, D, 0}, st)));
  } else {
    SAT_TRY((gemm_tn<float, TS>(false, gemm_a1(b.dP, A, A), (const TS*)w.WaT, A, B * L, D, epi_dann, st)));
  }
  return 0;
}

}  // namespace

extern "C" int sat_train_backward(const SatDims* d, const SatWeights* w, SatTrainBuffers* b, void* stream) {
  SAT_REQUIRE(d && w && b, "sat_train_backward: NULL struct");
  SAT_REQUIRE(d->A <= 128 * ATTB_MAXKA, "sat_train_backward: attention_dim %d exceeds the training limit of %d", d->A, 128 * ATTB_MAXKA);
  SAT_REQUIRE(b->dlogits && b->gscale && b->dpre && b->dHZ && b->DY && b->dgz && b->dh && b->dc && b->dZ && b->dP &&
                  b->dwf_part && b->dXe && b->d_init_out && b->df1 && b->dmean && b->d_ann,
              "sat_train_backward: NULL backward buffer");
  SAT_REQUIRE(w->WoT && w->WhozoT && w->WihzT && w->WiheT && w->WhcatT && w->WaT && w->WinitT && w->WfactT,
              "sat_train_backward: transposed weights missing");
  cudaStream_t st = (cudaStream_t)stream;
  if (d->dtype == SAT_F32)
    return d->exact ? train_backward_impl<float, true>(*d, *w, *b, st) : train_backward_impl<float, false>(*d, *w, *b, st);
  return d->exact ? train_backward_impl<bf16, true>(*d, *w, *b, st) : train_backward_impl<bf16, false>(*d, *w, *b, st);
}
