// Vocabulary projection fused with what consumes it (DeepOutput's last Linear, model.py:130, + LabelSmoothing, util.py:105-112,
// + accuracy, model.py:596-597; or + log-softmax / masks / arg-max of greedy decoding, model.py:330-343): row-owner epilogues
// of the tcgen05 GEMM core (sat_gemm_tc.cuh).  The [T*B, V] logits never reach HBM:
//   pass 1 (VOCAB_STATS)   per (row, 128-column tile): max, sum exp(x - max), sum x, arg-max, and the target logit
//   ce_finalize_kernel     per row: log-sum-exp, token loss, arg-max
//   ss_feedback_kernel     scheduled sampling: pass 1 over one step's B rows inside the time loop, then the arg-max of each row
//                          becomes the next step's input word (the same rule as ce_finalize_kernel's arg-max)
//   pass 2 (VOCAB_DLOGITS) recomputes the tile and writes dlogits = (softmax - target distribution) / N_tok in the operand
//                          dtype -- the only [T*B, V] array of the training step (it feeds dpre = dlogits * Wo and dWo)
//   VOCAB_GREEDY           per (row, tile): soft-max statistics of x / temperature and the best non-masked word;
//                          greedy_finalize_kernel turns them into the row's candidate (score, word)
//   VOCAB_TOPK             per (row, tile): soft-max statistics of x / temperature and the tile's best kcap non-masked words
//                          (beam search, the "topk" sampler); cand_finalize_kernel<false> merges the tiles of a row
//   VOCAB_SAMPLE           per (row, tile): the same statistics, (max, sum exp) of s * x over the unmasked words and the best kcap
//                          words by s * x + Gumbel noise (multinomial sampler, s = 20 / step); cand_finalize_kernel<true>
// After tcgen05.ld a thread holds one accumulator row, so all of these reductions are thread-local; the two column halves
// of a tile (two warps per TMEM lane quarter) are combined through the drained operand ring.
#pragma once
#include <stdlib.h>

#include "sat_gemm_tc.cuh"

namespace tc {

constexpr float LOG2E_F = 1.4426950408889634f;
__device__ __forceinline__ float ex2_fast(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

enum { VOCAB_STATS = 0, VOCAB_DLOGITS = 1, VOCAB_GREEDY = 2, VOCAB_TOPK = 3, VOCAB_SAMPLE = 4 };
constexpr int CAND_NONE = 0x7fffffff;      // word of an empty candidate slot (a tile with fewer than kcap candidate words)

struct VocabArgs {
  const float* bias;        // [N] over the storage vocabulary, or nullptr
  int V0;                   // true vocabulary size: columns >= V0 are padding and never count
  int NT;                   // 128-column tiles per row (row pitch of `stats`)
  float4* stats;            // [M][NT]
  // cross entropy (STATS / DLOGITS): row m = t*B + b, target y = caps[b*caplen + t + 1], active iff t < lens[b]
  const int32_t* caps;
  const int32_t* lens;
  int B, caplen;
  int row0;                 // time-major row of the launch's first row (0: whole sequence; (t-1)*B: one step of scheduled sampling)
  float* row_xt;            // [M] logit of the target word (written by the one thread that owns its column)
  const float* row_lse;     // [M]                                     (DLOGITS)
  const float* inv_ntok_p;  //                                         (DLOGITS)
  float smoothing;
  bf16* dlogits;            // [M, ldd]                                (DLOGITS)
  int64_t ldd;
  // greedy decode (GREEDY, TOPK, SAMPLE): row r is live iff alive[r] != 0
  const int32_t* alive;
  float inv_temp;
  int tokPAD, tokSTART, tokEND, tokUNK, step0;
  // candidate lists (TOPK, SAMPLE): [M][NT][kcap], per tile in (key descending, word ascending) order
  int kcap;
  float* cand_x;            // x = logit / T of the candidate (-inf: empty slot)
  int32_t* cand_col;        // its word (CAND_NONE: empty slot)
  float* cand_key;          // s * x + Gumbel(seed, step, m * N + word)  (SAMPLE)
  float2* stats2;           // [M][NT] max and sum exp of s * x over the unmasked words  (SAMPLE)
  float sharp;              // s = 20 / step  (SAMPLE)
  uint64_t seed;
  int step;
};

template <int MODE>
struct EpiVocab {
  static constexpr bool kRowOwner = true;
  VocabArgs a;

  // bias tile of this CTA -> aux[0..128); -inf beyond the true vocabulary (padding and the N tail), so that padded
  // columns drop out of every maximum / sum without further tests
  __device__ __forceinline__ void prologue(float* aux, int n0, int N, int warp, int lane) const {
    const int i = (warp - 2) * 32 + lane;
    if (i < 128) {
      const int n = n0 + i;
      aux[i] = n < a.V0 ? (a.bias ? a.bias[n] : 0.0f) : -INFINITY;
    }
    (void)N;
  }

  // NW epilogue warps (8: one-tile-per-CTA kernel, 16: persistent kernel): warp w reads TMEM lane quarter w & 3 (rows) and the
  // column part (w - 2) >> 2 of the tile, 128 / (NW / 4) columns.
  template <int BN, int NW>
  __device__ __forceinline__ void run(uint8_t* scratch, const float* aux, uint32_t tmem, bool has_acc, int warp, int lane, int m0,
                                      int n0, int M, int N, int tile_n) const {
    static_assert(BN == 128, "the vocabulary epilogues work on 128-column tiles");
    static_assert(NW == 8 || NW == 16, "two or four column parts");
    if constexpr (MODE == VOCAB_TOPK || MODE == VOCAB_SAMPLE) {
      run_cand<BN, NW>(scratch, aux, tmem, has_acc, warp, lane, m0, n0, M, N, tile_n);
      return;
    }
    constexpr int PARTS = NW / 4, PCOLS = BN / PARTS, NCH = PCOLS / 16;
    const int q = warp & 3, part = (warp - 2) >> 2;
    const int r = q * 32 + lane, m = m0 + r;
    const int cbase = part * PCOLS;                                // first tile column of this thread
    asm volatile("bar.sync 1, %0;" ::"n"(NW * 32) : "memory");     // bias tile staged by prologue()
    bool active = m < M;
    int y = -1;
    if (MODE == VOCAB_GREEDY) {
      active = active && a.alive[m] != 0;
    } else {
      const int mg = a.row0 + m, t = mg / a.B, b = mg - t * a.B;
      active = active && t < a.lens[b];
      if (active) y = sat_word_or_pad(a.caps[(int64_t)b * a.caplen + t + 1], a.V0);
    }
    const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)cbase;
    const bool tile_full = n0 + BN <= a.V0;                        // no padded / out-of-range column in this tile (CTA-uniform)
    if (MODE == VOCAB_DLOGITS) {
      // ---- pass 2: dlogits tile, staged as bf16 [128][128 + 8] and written out with whole rows per half warp ----
      constexpr int PITCH = (BN + 8) * 2;                          // bytes; 272: quarter-warp 16-byte stores hit distinct banks
      const float nlse = active ? -a.row_lse[m] * LOG2E_F : -INFINITY;     // finished rows: exp2(-inf) = 0, no overflow
      const float inv_ntok = active ? *a.inv_ntok_p : 0.0f;        // finished rows: all-zero gradient
      const float sv = a.smoothing / (float)a.V0, conf = 1.0f - a.smoothing;
#pragma unroll 1
      for (int ch = 0; ch < NCH; ++ch) {
        float v[16];
        if (has_acc) tmem_ld16(taddr + ch * 16, v);
        else {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = 0.0f;
        }
        const int c0 = cbase + ch * 16;
        const int jy = y - (n0 + c0);                              // target column inside this chunk, or out of [0,16)
        uint32_t pk[8];
#pragma unroll
        for (int j = 0; j < 16; j += 2) {
          float p2[2];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const float x = v[j + u] + aux[c0 + j + u];
            float p = ex2_fast(fmaf(x, LOG2E_F, nlse)) - sv;       // softmax - s/V   (x = -inf: -s/V, zeroed below)
            if (j + u == jy) p -= conf;
            p2[u] = (tile_full || x > -INFINITY) ? p * inv_ntok : 0.0f;
          }
          const __nv_bfloat162 h = __floats2bfloat162_rn(p2[0], p2[1]);
          pk[j >> 1] = *reinterpret_cast<const uint32_t*>(&h);
        }
        uint4* dst = reinterpret_cast<uint4*>(scratch + (size_t)r * PITCH + (size_t)c0 * 2);
        dst[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        dst[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
      }
      asm volatile("bar.sync 1, %0;" ::"n"(NW * 32) : "memory");
      const int ew = warp - 2;
#pragma unroll 1
      for (int it = 0; it < BM / (NW * 2); ++it) {
        const int rr = it * (NW * 2) + ew * 2 + (lane >> 4);
        const int cc = (lane & 15) * 8;
        const int mm = m0 + rr, n = n0 + cc;
        if (mm < M && n < N)
          *reinterpret_cast<uint4*>(a.dlogits + (int64_t)mm * a.ldd + n) = *reinterpret_cast<const uint4*>(scratch + (size_t)rr * PITCH + (size_t)cc * 2);
      }
      return;
    }

    // ---- STATS / GREEDY: running soft-max statistics of this thread's columns (short dependency chains: pairwise trees) ----
    float mx = -INFINITY, se = 0.0f, sx = 0.0f, xt = 0.0f, bestv = -INFINITY;
    int arg = 0x7fffffff, has_xt = 0;
    const float xs = MODE == VOCAB_GREEDY ? a.inv_temp : 1.0f;
#pragma unroll 1
    for (int ch = 0; ch < NCH; ++ch) {
      float v[16];
      if (has_acc) tmem_ld16(taddr + ch * 16, v);
      else {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = 0.0f;
      }
      const int c0 = cbase + ch * 16, col0 = n0 + c0;
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = (v[j] + aux[c0 + j]) * xs;
      // chunk arg-max as a tree of (value, index) pairs; a tie keeps the lower index (torch.argmax / topk order)
      float cv[16];
      int ci[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        cv[j] = v[j];
        ci[j] = j;
        if (MODE == VOCAB_GREEDY) {
          // candidate set: <START>, <PAD> never; <END>, <UNK> not at step 0 (model.py:333,340)
          const int col = col0 + j;
          if (col == a.tokSTART || col == a.tokPAD || (a.step0 && (col == a.tokEND || col == a.tokUNK))) cv[j] = -INFINITY;
        }
      }
#pragma unroll
      for (int w = 1; w < 16; w <<= 1) {
#pragma unroll
        for (int j = 0; j + w < 16; j += 2 * w) {
          const bool keep = cv[j] >= cv[j + w];
          cv[j] = keep ? cv[j] : cv[j + w];
          ci[j] = keep ? ci[j] : ci[j + w];
        }
      }
      if (cv[0] > bestv) { bestv = cv[0]; arg = col0 + ci[0]; }    // strictly greater: earlier chunks win ties
      float cm;                                                    // chunk max over EVERY column (soft-max statistics ignore the masks)
      if (MODE == VOCAB_GREEDY) {
        float t8[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) t8[j] = fmaxf(v[2 * j], v[2 * j + 1]);
        cm = fmaxf(fmaxf(fmaxf(t8[0], t8[1]), fmaxf(t8[2], t8[3])), fmaxf(fmaxf(t8[4], t8[5]), fmaxf(t8[6], t8[7])));
      } else {
        cm = cv[0];
        if ((unsigned)(y - col0) < 16u) {
          const int jy = y - col0;
#pragma unroll
          for (int j = 0; j < 16; ++j)
            if (j == jy) xt = v[j];
          has_xt = 1;
        }
      }
      if (cm > -INFINITY) {
        if (cm > mx) {
          se *= ex2_fast((mx - cm) * LOG2E_F);                     // mx = -inf: se is still 0
          mx = cm;
        }
        const float nm = -mx * LOG2E_F;
        float s4[4] = {0.f, 0.f, 0.f, 0.f}, t4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          s4[j & 3] += ex2_fast(fmaf(v[j], LOG2E_F, nm));
          if (MODE != VOCAB_GREEDY) t4[j & 3] += (tile_full || v[j] > -INFINITY) ? v[j] : 0.0f;
        }
        se += (s4[0] + s4[1]) + (s4[2] + s4[3]);
        sx += (t4[0] + t4[1]) + (t4[2] + t4[3]);
      }
    }
    // combine the column parts of the tile (same row, warps w, w + 4, ..) through shared memory, lower columns first
    float* xch = reinterpret_cast<float*>(scratch);
    if (part > 0) {
      float* o = xch + ((part - 1) * BM + r) * 8;
      o[0] = mx; o[1] = se; o[2] = sx; o[3] = bestv; o[4] = __int_as_float(arg); o[5] = xt; o[6] = __int_as_float(has_xt);
    }
    asm volatile("bar.sync 1, %0;" ::"n"(NW * 32) : "memory");
    if (part == 0 && active) {
#pragma unroll
      for (int p2 = 1; p2 < PARTS; ++p2) {
        const float* o = xch + ((p2 - 1) * BM + r) * 8;
        const float mx1 = o[0], se1 = o[1], bv1 = o[3];
        const float mm = fmaxf(mx, mx1);
        float s = 0.0f;
        if (mx > -INFINITY) s += se * ex2_fast((mx - mm) * LOG2E_F);
        if (mx1 > -INFINITY) s += se1 * ex2_fast((mx1 - mm) * LOG2E_F);
        mx = mm;
        se = s;
        sx += o[2];
        if (bv1 > bestv) { bestv = bv1; arg = __float_as_int(o[4]); }   // ties keep the lower columns
        if (__float_as_int(o[6]) != 0) { xt = o[5]; has_xt = 1; }
      }
      if (MODE == VOCAB_GREEDY) {
        a.stats[(int64_t)m * a.NT + tile_n] = make_float4(mx, se, bestv, __int_as_float(arg));
      } else {
        a.stats[(int64_t)m * a.NT + tile_n] = make_float4(mx, se, sx, __int_as_float(arg));
        if (has_xt) a.row_xt[m] = xt;
      }
    }
    (void)N;
  }

  // TOPK / SAMPLE.  A thread keeps the selection keys of its PCOLS columns in registers (masked words and padding: -inf).  The
  // tile's candidates are then extracted one per round: every thread proposes its best key after the last pick (only the
  // thread that supplied the last pick has to rescan), the proposals of a row's column parts meet in shared memory, and the
  // thread that owns the winner writes it.  Exact, in (key descending, word ascending) order, no atomics; one barrier a round.
  // SAMPLE re-reads the winner's x from tensor memory (same expression, same bits) rather than keeping a second register array.
  template <int BN, int NW>
  __device__ __forceinline__ void run_cand(uint8_t* scratch, const float* aux, uint32_t tmem, bool has_acc, int warp, int lane, int m0,
                                           int n0, int M, int N, int tile_n) const {
    constexpr bool SAMP = MODE == VOCAB_SAMPLE;
    constexpr int PARTS = NW / 4, PCOLS = BN / PARTS, NCH = PCOLS / 16;
    const int q = warp & 3, part = (warp - 2) >> 2;
    const int r = q * 32 + lane, m = m0 + r;
    const int cbase = part * PCOLS;
    asm volatile("bar.sync 1, %0;" ::"n"(NW * 32) : "memory");     // bias tile staged by prologue()
    const bool active = m < M && a.alive[m] != 0;
    const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)cbase;
    float key[PCOLS];
    float mx = -INFINITY, se = 0.0f, mx2 = -INFINITY, se2 = 0.0f;
#pragma unroll
    for (int ch = 0; ch < NCH; ++ch) {
      float v[16];
      if (has_acc) tmem_ld16(taddr + ch * 16, v);
      else {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = 0.0f;
      }
      const int c0 = cbase + ch * 16, col0 = n0 + c0;
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = (v[j] + aux[c0 + j]) * a.inv_temp;
      // candidate set: <START>, <PAD> never; <END>, <UNK> not at step 0 (model.py:333,340); padding is -inf already.
      // TOPK: key = x.  SAMPLE: key = y = s * x for now (the Gumbel noise is added below, once the chunks are done)
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const int col = col0 + j;
        const bool masked = col == a.tokSTART || col == a.tokPAD || (a.step0 && (col == a.tokEND || col == a.tokUNK));
        key[ch * 16 + j] = masked ? -INFINITY : (SAMP ? a.sharp * v[j] : v[j]);
      }
      // running soft-max statistics over EVERY real column (as VOCAB_GREEDY), and (SAMPLE) of y over the unmasked ones
      float t8[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) t8[j] = fmaxf(v[2 * j], v[2 * j + 1]);
      const float cm = fmaxf(fmaxf(fmaxf(t8[0], t8[1]), fmaxf(t8[2], t8[3])), fmaxf(fmaxf(t8[4], t8[5]), fmaxf(t8[6], t8[7])));
      if (cm > -INFINITY) {
        if (cm > mx) {
          se *= ex2_fast((mx - cm) * LOG2E_F);
          mx = cm;
        }
        const float nm = -mx * LOG2E_F;
        float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int j = 0; j < 16; ++j) s4[j & 3] += ex2_fast(fmaf(v[j], LOG2E_F, nm));
        se += (s4[0] + s4[1]) + (s4[2] + s4[3]);
      }
      if (SAMP) {
        const float* y = key + ch * 16;
#pragma unroll
        for (int j = 0; j < 8; ++j) t8[j] = fmaxf(y[2 * j], y[2 * j + 1]);
        const float cm2 = fmaxf(fmaxf(fmaxf(t8[0], t8[1]), fmaxf(t8[2], t8[3])), fmaxf(fmaxf(t8[4], t8[5]), fmaxf(t8[6], t8[7])));
        if (cm2 > -INFINITY) {
          if (cm2 > mx2) {
            se2 *= ex2_fast((mx2 - cm2) * LOG2E_F);
            mx2 = cm2;
          }
          const float nm = -mx2 * LOG2E_F;
          float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int j = 0; j < 16; ++j) s4[j & 3] += ex2_fast(fmaf(y[j], LOG2E_F, nm));
          se2 += (s4[0] + s4[1]) + (s4[2] + s4[3]);
        }
      }
    }
    if (SAMP) {
      uint64_t idx0 = (uint64_t)m * (uint64_t)N + (uint64_t)(n0 + cbase);
#pragma unroll
      for (int j = 0; j < PCOLS; ++j) {
        key[j] = (active && key[j] > -INFINITY) ? key[j] + sat_gumbel(a.seed, (uint32_t)a.step, idx0 + (uint64_t)j) : -INFINITY;
        // four draws at a time: without this dependence the compiler overlaps all PCOLS hash chains and runs out of registers
        if ((j & 3) == 3) asm volatile("" : "+l"(idx0) : "f"(key[j]));
      }
    }
    // scratch: [PARTS-1][BM] float4 statistics of the upper column parts, then [2][PARTS][BM] float2 proposals (double-buffered:
    // round i + 2 overwrites round i's slot only after every thread has passed round i + 1's barrier)
    float4* xch = reinterpret_cast<float4*>(scratch);
    float2* prop = reinterpret_cast<float2*>(scratch + (size_t)(PARTS - 1) * BM * sizeof(float4));
    if (part > 0) xch[(part - 1) * BM + r] = make_float4(mx, se, mx2, se2);
    float pv = INFINITY, bv = -INFINITY;                           // pv, pi: the tile's last pick; bv, bi: this thread's proposal
    int pi = -1, bi = CAND_NONE;
    bool rescan = true;
    const int64_t out0 = ((int64_t)m * a.NT + tile_n) * a.kcap;
#pragma unroll 1
    for (int i = 0; i < a.kcap; ++i) {
      if (rescan) {
        bv = -INFINITY; bi = CAND_NONE;
        if (active) {
#pragma unroll
          for (int j = 0; j < PCOLS; ++j) {                        // columns ascend, strict '>': ties keep the lower word
            const float kv = key[j];
            const int c = n0 + cbase + j;
            if ((kv < pv || (kv == pv && c > pi)) && kv > bv) {
              bv = kv; bi = c;
            }
          }
        }
        rescan = false;
      }
      prop[((i & 1) * PARTS + part) * BM + r] = make_float2(bv, __int_as_float(bi));
      asm volatile("bar.sync 1, %0;" ::"n"(NW * 32) : "memory");
      if (i == 0 && part == 0 && active) {
#pragma unroll
        for (int p2 = 1; p2 < PARTS; ++p2) {
          const float4 o = xch[(p2 - 1) * BM + r];
          float mm = fmaxf(mx, o.x), s = 0.0f;
          if (mx > -INFINITY) s += se * ex2_fast((mx - mm) * LOG2E_F);
          if (o.x > -INFINITY) s += o.y * ex2_fast((o.x - mm) * LOG2E_F);
          mx = mm; se = s;
          mm = fmaxf(mx2, o.z); s = 0.0f;
          if (mx2 > -INFINITY) s += se2 * ex2_fast((mx2 - mm) * LOG2E_F);
          if (o.z > -INFINITY) s += o.w * ex2_fast((o.z - mm) * LOG2E_F);
          mx2 = mm; se2 = s;
        }
        a.stats[(int64_t)m * a.NT + tile_n] = make_float4(mx, se, 0.0f, 0.0f);
        if (SAMP) a.stats2[(int64_t)m * a.NT + tile_n] = make_float2(mx2, se2);
      }
      float wv = -INFINITY;                                        // the round's winner: parts ascend with the columns
      int wi = CAND_NONE;
#pragma unroll
      for (int p2 = 0; p2 < PARTS; ++p2) {
        const float2 o = prop[((i & 1) * PARTS + p2) * BM + r];
        if (o.x > wv) { wv = o.x; wi = __float_as_int(o.y); }
      }
      const bool win = active && wi != CAND_NONE && wi == bi;
      float bx = bv;
      if (SAMP) {
#pragma unroll
        for (int ch = 0; ch < NCH; ++ch) {
          if (__any_sync(0xffffffffu, win && ((bi - n0 - cbase) >> 4) == ch)) {      // warp-uniform: tcgen05.ld is collective
            float v[16];
            if (has_acc) tmem_ld16(taddr + ch * 16, v);
            else {
#pragma unroll
              for (int j = 0; j < 16; ++j) v[j] = 0.0f;
            }
            const int c0 = cbase + ch * 16;
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (n0 + c0 + j == bi) bx = (v[j] + aux[c0 + j]) * a.inv_temp;
          }
        }
      }
      if (win || (active && wi == CAND_NONE && part == 0)) {
        const bool none = wi == CAND_NONE;
        a.cand_x[out0 + i] = none ? -INFINITY : bx;
        a.cand_col[out0 + i] = wi;
        if (SAMP) a.cand_key[out0 + i] = none ? -INFINITY : bv;
        rescan = !none;
      }
      pv = wv; pi = wi;
    }
  }
};

// Arg-max of a row over its VOCAB_STATS tiles, the first maximal word (torch.argmax): a tile's max is the value of its arg-max
// and tiles ascend with the columns.  Warp-collective; every lane returns the row's (max, arg-max).  The one rule for both the
// reported arg-max (ce_finalize_kernel) and the word scheduled sampling feeds back (ss_feedback_kernel).
__device__ __forceinline__ int tiles_argmax(const float4* __restrict__ st, int NT, int lane, float& mx_out) {
  float mx = -INFINITY;
  int arg = 0x7fffffff;
  for (int i = lane; i < NT; i += 32) {
    const float4 s4 = st[i];
    if (s4.x > mx) { mx = s4.x; arg = __float_as_int(s4.w); }
  }
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, mx, o);
    const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
    if (om > mx || (om == mx && oa < arg)) { mx = om; arg = oa; }
  }
  mx_out = mx;
  return arg;
}

// Row-wise finish of the fused cross entropy: log-sum-exp over the tile statistics, token loss (util.py:105-112) and arg-max
// (model.py:596).  One warp per row, fixed combination order.
static __global__ void __launch_bounds__(256)
ce_finalize_kernel(const float4* __restrict__ stats, int NT, const float* __restrict__ row_xt, const int32_t* __restrict__ lens, int B,
                   int M, int V0, float smoothing, float* __restrict__ row_lse, float* __restrict__ row_loss,
                   int32_t* __restrict__ row_argmax) {
  SAT_PDL_TRIGGER();
  SAT_PDL_WAIT();
  const int lane = threadIdx.x & 31, m = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (m >= M) return;
  const int t = m / B, b = m - t * B;
  if (t >= lens[b]) {
    if (lane == 0) { row_loss[m] = 0.0f; row_argmax[m] = -1; row_lse[m] = 0.0f; }
    return;
  }
  const float4* st = stats + (int64_t)m * NT;
  float mx;
  const int arg = tiles_argmax(st, NT, lane, mx);
  float se = 0.0f, sx = 0.0f;
  for (int i = lane; i < NT; i += 32) {
    const float4 s4 = st[i];
    se += s4.y * __expf(s4.x - mx);
    sx += s4.z;
  }
  se = warp_sum(se);
  sx = warp_sum(sx);
  if (lane == 0) {
    const float lse = mx + __logf(se);
    const float nll = lse - row_xt[m];
    const float smooth = lse - sx / (float)V0;
    row_lse[m] = lse;
    row_loss[m] = (1.0f - smoothing) * nll + smoothing * smooth;
    row_argmax[m] = arg;
  }
}

// Scheduled sampling on the fused path (model.py:518-523): the word fed at step t is the arg-max of step t-1's logits, read from
// the VOCAB_STATS tiles of those B rows (stats = [B][NT] of step t-1).  A caption finished at step t-1 (t-1 >= lens[b])
// keeps its teacher-forced word (it only has to be a valid id: nothing reads that row's outputs).  A row without a finite maximum
// (non-finite logits) is fed <PAD>, as row_argmax_kernel does; the bad-id flag out[6] belongs to the captions and is left alone.
static __global__ void __launch_bounds__(256)
ss_feedback_kernel(const float4* __restrict__ stats, int NT, const int32_t* __restrict__ lens, int B, int t, int V0,
                   int32_t* __restrict__ tok_t) {
  SAT_PDL_TRIGGER();
  SAT_PDL_WAIT();
  const int lane = threadIdx.x & 31, b = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (b >= B || t - 1 >= lens[b]) return;
  float mx;
  const int arg = tiles_argmax(stats + (int64_t)b * NT, NT, lane, mx);
  if (lane == 0) tok_t[b] = sat_word_or_pad(arg, V0);
}

// Greedy decode: candidate (score, word) of every live row from the tile statistics -- the k = 1 output of
// row_topk_kernel (log-softmax(x / T), masks, + parent score; model.py:330-351) without materialising the logits.
static __global__ void __launch_bounds__(256)
greedy_finalize_kernel(const float4* __restrict__ stats, int NT, const int32_t* __restrict__ alive, const float* __restrict__ top_scores,
                       int R, int step0, float* __restrict__ cand_val, int32_t* __restrict__ cand_idx) {
  SAT_PDL_TRIGGER();
  SAT_PDL_WAIT();
  const int lane = threadIdx.x & 31, r = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= R || alive[r] == 0) return;
  const float4* st = stats + (int64_t)r * NT;
  float mx = -INFINITY, bv = -INFINITY;
  int arg = 0x7fffffff;
  for (int i = lane; i < NT; i += 32) {
    const float4 s4 = st[i];
    mx = fmaxf(mx, s4.x);
    if (s4.z > bv) { bv = s4.z; arg = __float_as_int(s4.w); }
  }
  mx = warp_max(mx);
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
    if (ov > bv || (ov == bv && oa < arg)) { bv = ov; arg = oa; }
  }
  float se = 0.0f;
  for (int i = lane; i < NT; i += 32) {
    const float4 s4 = st[i];
    se += s4.y * __expf(s4.x - mx);
  }
  se = warp_sum(se);
  if (lane == 0) {
    const float lp = (bv - mx) - __logf(se);
    cand_val[r] = step0 ? lp : lp + top_scores[r];
    cand_idx[r] = arg;
  }
}

// Beam search, the "topk" sampler (SAMP = false) and the multinomial sampler at steps > 0 (SAMP = true): the row's candidates
// from the per-tile lists, in exactly the layout and meaning of row_topk_thresh_kernel / row_sample_kernel (sat_decode_kernels.cuh)
// without materialising the logits.  One warp per row, fixed order: lane l owns tiles l, l + 32, ..; every round each lane offers
// its best entry after the last pick (the first such entry of each of its sorted tile lists), the warp takes the best offer.
template <bool SAMP>
static __global__ void __launch_bounds__(256)
cand_finalize_kernel(const float4* __restrict__ stats, const float2* __restrict__ stats2, const float* __restrict__ tx,
                     const float* __restrict__ tkey, const int32_t* __restrict__ tcol, int NT, int kcap, const float* __restrict__ top_scores,
                     const int32_t* __restrict__ kcur, int k, int kk_req, int R, int step0, float* __restrict__ cand_key,
                     float* __restrict__ cand_val, int32_t* __restrict__ cand_idx) {
  SAT_PDL_TRIGGER();
  SAT_PDL_WAIT();
  const int lane = threadIdx.x & 31, r = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= R) return;
  const int n = r / k, j = r - n * k, kc = kcur[n];
  if (j >= kc) return;
  if (step0 && j != 0) return;                        // step 0 looks at beam 0 only (model.py:343)
  // log-sum-exp of x over the row, and (SAMP) of s * x over the unmasked words
  const float4* st = stats + (int64_t)r * NT;
  float mx = -INFINITY, mx2 = -INFINITY;
  for (int i = lane; i < NT; i += 32) {
    mx = fmaxf(mx, st[i].x);
    if (SAMP) mx2 = fmaxf(mx2, stats2[(int64_t)r * NT + i].x);
  }
  mx = warp_max(mx);
  mx2 = warp_max(mx2);
  float se = 0.0f, se2 = 0.0f;
  for (int i = lane; i < NT; i += 32) {
    const float4 s4 = st[i];
    se += s4.y * expf(s4.x - mx);
    if (SAMP) {
      const float2 s2 = stats2[(int64_t)r * NT + i];
      if (s2.x > -INFINITY) se2 += s2.y * expf(s2.x - mx2);
    }
  }
  se = warp_sum(se);
  se2 = warp_sum(se2);
  const float lse = logf(se), lse2 = mx2 + logf(se2);
  const float base = step0 ? 0.0f : top_scores[r];
  const int kk = SAMP ? kc : (step0 ? k : (kk_req > 0 ? kk_req : kc));
  const float* tk = SAMP ? tkey : tx;                 // selection key
  const int64_t row0 = (int64_t)r * NT * kcap;
  float pv = INFINITY, bv = -INFINITY, bx = -INFINITY;
  int pi = -1, bi = CAND_NONE;
  bool rescan = true;
  for (int i = 0; i < kk; ++i) {
    if (rescan) {
      bv = -INFINITY; bi = CAND_NONE;
      for (int t = lane; t < NT; t += 32) {
        const int64_t o = row0 + (int64_t)t * kcap;
        for (int e = 0; e < kcap; ++e) {
          const int c = tcol[o + e];
          if (c == CAND_NONE) break;
          const float kv = tk[o + e];
          if (kv < pv || (kv == pv && c > pi)) {      // first entry of this list after the last pick
            if (kv > bv || (kv == bv && c < bi)) {
              bv = kv; bi = c;
              if (SAMP) bx = tx[o + e];
            }
            break;
          }
        }
      }
      rescan = false;
    }
    float wv = bv;
    int wi = bi;
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, wv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, wi, o);
      if (ov > wv || (ov == wv && oi < wi)) { wv = ov; wi = oi; }
    }
    const bool ok = wi != CAND_NONE;
    if (ok && wi == bi) {                             // the lane that owns the pick writes it
      rescan = true;
      if (SAMP) {
        cand_key[(int64_t)r * kcap + i] = bv - lse2;
        cand_val[(int64_t)r * kcap + i] = ((bx - mx) - lse) + base;
      } else {
        const float lp = (bv - mx) - lse;
        cand_val[(int64_t)r * kcap + i] = step0 ? lp : lp + base;
      }
      cand_idx[(int64_t)r * kcap + i] = wi;
    } else if (!ok && lane == 0) {                    // fewer candidate words than kk (as the row kernels)
      if (SAMP) cand_key[(int64_t)r * kcap + i] = -INFINITY;
      cand_val[(int64_t)r * kcap + i] = -INFINITY;
      cand_idx[(int64_t)r * kcap + i] = SAMP ? 0 : CAND_NONE;
    }
    pv = wv; pi = wi;
  }
}

template <int MODE>
static int launch_vocab(const GemmOperandA& A, const bf16* W, int64_t ldw, int M, int N, const VocabArgs& va, cudaStream_t stream) {
  EpiVocab<MODE> epi{va};
  // persistent kernel (one CTA per SM, double-buffered tensor memory) at every size, so that a row's statistics do not depend
  // on the batch it is computed in (the two kernels split a tile's columns differently); SAT_VOCAB_PERSIST=0 forces the
  // one-tile-per-CTA kernel (A/B timing)
  static const int pers_mode = getenv("SAT_VOCAB_PERSIST") ? atoi(getenv("SAT_VOCAB_PERSIST")) : 1;
  if (pers_mode != 0 && persistent_ok(A)) return launch_persistent<EpiVocab<MODE>>(A, W, ldw, M, N, epi, stream);
  return launch_bn<128, EpiVocab<MODE>>(A, W, ldw, M, N, epi, stream);
}

}  // namespace tc
