// Integer / indexing kernels of greedy (beamk = 1) and beam decoding (model.py:237-472), batched over
// images with all beam state resident on the device:
//   row_topk_kernel     : log-softmax(logit / T) + masks + parent score, per-row top-k candidates
//   beam_update_kernel  : per image k^2 -> k merge, <END> handling, rescoring, order-preserving
//                         compaction of live beams, history append, flush at max length
//   gather_state_kernel : h, c reorder by source row (model.py:397)
#pragma once
#include "sat_common.cuh"

constexpr int SAT_ALIVE = 1 << 30;
enum { SAT_RESCORE_NONE = 0, SAT_RESCORE_LN = 1, SAT_RESCORE_WR = 2, SAT_RESCORE_BAR = 3 };

// Per-image InitLSTM reinterpretation for a beam of k identical rows (model.py:265-269, SURVEY.md §A.2-1):
//   h0[j] = o[(j % 2) * H : ...],  c0[j] = o[((k + j) % 2) * H : ...]   where o = init_out[img] ([2H]).
template <typename T>
__global__ void init_state_decode_kernel(const float* __restrict__ init_out, int64_t ld_io, T* __restrict__ h0, float* __restrict__ c0,
                                         int n_img, int k, int H, int ld, int nl) {
  // The k rows of an image are identical, so the [k, 2*nl*H] init output read row-major as [2*nl, k, H] (model.py:79-80,
  // 265-269) gives state st, beam j, unit jj the element o[(st*k*H + j*H + jj) mod (2*nl*H)] of the image's init vector o.
  // H = the module's true decoder_dim; ld = storage pitch of the state rows (columns H..ld are padding and get zeros);
  // layer l of h / c lives at h0 + l * n_img*k*ld.
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t per = (int64_t)n_img * k * ld;
  if (idx >= nl * per) return;
  const int l = (int)(idx / per);
  const int64_t rem = idx - l * per;
  const int jj = (int)(rem % ld);
  const int64_t row = rem / ld;
  const int j = (int)(row % k);
  const int64_t n = row / k;
  const float* o = init_out + n * ld_io;
  const int64_t W2 = 2 * (int64_t)nl * H;
  const int64_t fh = ((int64_t)l * k + j) * H + jj, fc = ((int64_t)(nl + l) * k + j) * H + jj;
  h0[idx] = from_f<T>(jj < H ? o[fh % W2] : 0.0f);
  c0[idx] = jj < H ? o[fc % W2] : 0.0f;
}

// scores = log_softmax(logit / temp) (model.py:330); <START>,<PAD> -> -inf (model.py:333); step 0 also
// <END>,<UNK> (model.py:340); + parent score (model.py:351).  Emits the row's best `kk` candidates in
// descending order (ties: lower vocabulary index first).
// log-softmax and "+ parent score" are monotone per row, so the candidates are selected on the scaled logits
// x = logit / temp (one pass from global memory fused with the running max / argmax, one pass over shared memory
// for the sum of exponentials) and only the winners are converted: score = (x - max) - log(sum exp(x - max)) + parent.
__global__ void __launch_bounds__(256)
row_topk_kernel(const float* __restrict__ logits, const float* __restrict__ top_scores, const int32_t* __restrict__ kcur,
                int k, int kcap, int kk_req, int V, int step, float temp, int tokPAD, int tokSTART, int tokEND, int tokUNK,
                float* __restrict__ cand_val, int32_t* __restrict__ cand_idx) {
  SAT_PDL_TRIGGER();
  SAT_PDL_WAIT();
  extern __shared__ __align__(16) float smem[];
  float* x = smem;            // [V]  scaled logits, masked entries set to -inf after the softmax statistics
  float* scratch = x + V;     // [33]
  __shared__ float s_val[8];
  __shared__ int s_idx[8];
  const int r = blockIdx.x, n = r / k, j = r - n * k, tid = threadIdx.x;
  const int kc = kcur[n];
  if (j >= kc) return;
  if (step == 0 && j != 0) return;                    // step 0 looks at beam 0 only (model.py:343)
  const float* row = logits + (int64_t)r * V;
  const bool s0 = step == 0;
  // pass 1 (global -> shared): x = logit / temp, row max over ALL entries (softmax statistics ignore the masks)
  float mx = -INFINITY;
  for (int v = tid * 4; v < V; v += 256 * 4) {
    float4 q = *reinterpret_cast<const float4*>(row + v);
    q.x = q.x / temp; q.y = q.y / temp; q.z = q.z / temp; q.w = q.w / temp;
    *reinterpret_cast<float4*>(x + v) = q;
    mx = fmaxf(fmaxf(mx, fmaxf(q.x, q.y)), fmaxf(q.z, q.w));
  }
  mx = block_max(mx, scratch);
  // pass 2 (shared): sum of exponentials; masked tokens are then removed from the candidate set
  float se = 0.0f;
  for (int v = tid; v < V; v += 256) {
    const float xv = x[v];
    se += expf(xv - mx);
    if (v == tokSTART || v == tokPAD || (s0 && (v == tokEND || v == tokUNK))) x[v] = -INFINITY;
  }
  se = block_sum(se, scratch);
  const float lse = logf(se);
  const float base = s0 ? 0.0f : top_scores[r];
  const int kk = s0 ? k : (kk_req > 0 ? kk_req : kc);      // kk_req: the "topk" sampler asks for sample_topk candidates per row (pitch kcap)
  float pv = INFINITY;
  int pi = -1;
  for (int i = 0; i < kk; ++i) {
    float bv = -INFINITY;
    int bi = 0x7fffffff;
    for (int v = tid; v < V; v += 256) {
      const float xv = x[v];
      const bool after = (xv < pv) || (xv == pv && v > pi);      // strictly after the previous pick in (val desc, idx asc)
      if (after && (xv > bv || (xv == bv && v < bi))) { bv = xv; bi = v; }
    }
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    __syncthreads();
    if ((tid & 31) == 0) { s_val[tid >> 5] = bv; s_idx[tid >> 5] = bi; }
    __syncthreads();
    bv = s_val[0]; bi = s_idx[0];
    for (int w = 1; w < 8; ++w)
      if (s_val[w] > bv || (s_val[w] == bv && s_idx[w] < bi)) { bv = s_val[w]; bi = s_idx[w]; }
    if (tid == 0) {
      const float lp = (bv - mx) - lse;                            // -inf stays -inf
      cand_val[(int64_t)r * kcap + i] = s0 ? lp : lp + base;
      cand_idx[(int64_t)r * kcap + i] = bi;
    }
    pv = bv; pi = bi;
  }
}

// Same selection without one block-wide scan per candidate.  While summing the exponentials every thread keeps the
// maximum of its strided slice; the kk-th largest of those 256 maxima is a lower bound T of the kk-th largest entry of
// the row, so one more pass collects the (few) entries >= T and warp 0 orders them.  Rows with more than TOPK_CAP
// entries >= T (massive ties) take the scan of row_topk_kernel.  The statistics (max, sum of exponentials) are
// accumulated in exactly the order of row_topk_kernel, so both kernels emit bit-identical candidates.  kk <= 32.
constexpr int TOPK_CAP = 256;
__device__ __forceinline__ bool topk_before(float av, int ai, float bv, int bi) { return av > bv || (av == bv && ai < bi); }

__global__ void __launch_bounds__(256)
row_topk_thresh_kernel(const float* __restrict__ logits, const float* __restrict__ top_scores, const int32_t* __restrict__ kcur,
                       int k, int kcap, int kk_req, int V, int step, float temp, int tokPAD, int tokSTART, int tokEND, int tokUNK,
                       float* __restrict__ cand_val, int32_t* __restrict__ cand_idx) {
  SAT_PDL_TRIGGER();
  SAT_PDL_WAIT();
  extern __shared__ __align__(16) float smem[];
  float* x = smem;            // [V]  scaled logits, masked entries set to -inf after the softmax statistics
  float* scratch = x + V;     // [33]
  __shared__ float c_val[TOPK_CAP];     // thread maxima, then the candidates
  __shared__ int c_idx[TOPK_CAP];
  __shared__ float s_T;
  __shared__ int s_cnt;
  const int r = blockIdx.x, n = r / k, j = r - n * k, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int kc = kcur[n];
  if (j >= kc) return;
  if (step == 0 && j != 0) return;                    // step 0 looks at beam 0 only (model.py:343)
  const float* row = logits + (int64_t)r * V;
  const bool s0 = step == 0;
  float mx = -INFINITY;
  for (int v = tid * 4; v < V; v += 256 * 4) {
    float4 q = *reinterpret_cast<const float4*>(row + v);
    q.x = q.x / temp; q.y = q.y / temp; q.z = q.z / temp; q.w = q.w / temp;
    *reinterpret_cast<float4*>(x + v) = q;
    mx = fmaxf(fmaxf(mx, fmaxf(q.x, q.y)), fmaxf(q.z, q.w));
  }
  mx = block_max(mx, scratch);
  float se = 0.0f, tm = -INFINITY;
  for (int v = tid; v < V; v += 256) {
    float xv = x[v];
    se += expf(xv - mx);
    if (v == tokSTART || v == tokPAD || (s0 && (v == tokEND || v == tokUNK))) { xv = -INFINITY; x[v] = xv; }
    tm = fmaxf(tm, xv);
  }
  c_val[tid] = tm;
  if (tid == 0) s_cnt = 0;
  se = block_sum(se, scratch);          // (its barriers also publish c_val / s_cnt)
  const float lse = logf(se);
  const float base = s0 ? 0.0f : top_scores[r];
  const int kk = s0 ? k : (kk_req > 0 ? kk_req : kc);      // kk_req: the "topk" sampler asks for sample_topk candidates per row (pitch kcap)
  if (warp == 0) {                      // T = kk-th largest thread maximum (with multiplicity)
    float m8[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) m8[u] = c_val[lane + 32 * u];
    float T = -INFINITY;
    for (int i = 0; i < kk; ++i) {
      float lb = m8[0];
#pragma unroll
      for (int u = 1; u < 8; ++u) lb = fmaxf(lb, m8[u]);
      const float wb = warp_max(lb);
      T = wb;
      const unsigned who = __ballot_sync(0xffffffffu, lb == wb);
      if (lane == __ffs(who) - 1) {     // remove one instance
        bool done = false;
#pragma unroll
        for (int u = 0; u < 8; ++u)
          if (!done && m8[u] == wb) { m8[u] = -INFINITY; done = true; }
      }
    }
    if (lane == 0) s_T = T;
  }
  __syncthreads();
  const float T = s_T;
  for (int v = tid; v < V; v += 256) {
    const float xv = x[v];
    if (xv >= T) {
      const int pos = atomicAdd(&s_cnt, 1);
      if (pos < TOPK_CAP) { c_val[pos] = xv; c_idx[pos] = v; }
    }
  }
  __syncthreads();
  const int nc = s_cnt;
  if (nc <= TOPK_CAP) {
    if (warp != 0) return;
    float cv[8];
    int ci[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int c = lane + 32 * u;
      cv[u] = c < nc ? c_val[c] : -INFINITY;
      ci[u] = c < nc ? c_idx[c] : 0x7fffffff;
    }
    for (int i = 0; i < kk; ++i) {
      float lb = cv[0];
      int li = ci[0];
#pragma unroll
      for (int u = 1; u < 8; ++u)
        if (topk_before(cv[u], ci[u], lb, li)) { lb = cv[u]; li = ci[u]; }
      float bv = lb;
      int bi = li;
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (topk_before(ov, oi, bv, bi)) { bv = ov; bi = oi; }
      }
      if (li == bi && bi != 0x7fffffff) {
#pragma unroll
        for (int u = 0; u < 8; ++u)
          if (ci[u] == bi) { cv[u] = -INFINITY; ci[u] = 0x7fffffff; }
      }
      if (lane == 0) {
        const float lp = (bv - mx) - lse;                            // -inf stays -inf
        cand_val[(int64_t)r * kcap + i] = s0 ? lp : lp + base;
        cand_idx[(int64_t)r * kcap + i] = bi;
      }
    }
    return;
  }
  // massive ties: block-wide scan per candidate (as row_topk_kernel)
  float pv = INFINITY;
  int pi = -1;
  for (int i = 0; i < kk; ++i) {
    float bv = -INFINITY;
    int bi = 0x7fffffff;
    for (int v = tid; v < V; v += 256) {
      const float xv = x[v];
      const bool after = (xv < pv) || (xv == pv && v > pi);
      if (after && topk_before(xv, v, bv, bi)) { bv = xv; bi = v; }
    }
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (topk_before(ov, oi, bv, bi)) { bv = ov; bi = oi; }
    }
    __syncthreads();
    if (lane == 0) { c_val[warp] = bv; c_idx[warp] = bi; }
    __syncthreads();
    bv = c_val[0]; bi = c_idx[0];
    for (int w = 1; w < 8; ++w)
      if (topk_before(c_val[w], c_idx[w], bv, bi)) { bv = c_val[w]; bi = c_idx[w]; }
    if (tid == 0) {
      const float lp = (bv - mx) - lse;
      cand_val[(int64_t)r * kcap + i] = s0 ? lp : lp + base;
      cand_idx[(int64_t)r * kcap + i] = bi;
    }
    pv = bv; pi = bi;
  }
}

// ---- sampling decoders (model.py:360-379) --------------------------------------------------------------------------------
// torch.multinomial(p, n) without replacement draws a Plackett-Luce ordering of the entries; taking the n largest of
// log p_i + G_i with independent standard Gumbel G_i draws from exactly that distribution (Gumbel-top-k), and it runs on
// the same per-row candidate / per-image merge structure as beam search.  The noise is a pure function of (seed, step, row,
// word), so a decode is reproducible under its seed; it is not the reference's torch RNG stream (not parity-checkable).
enum { SAT_SAMPLE_BEAM = 0, SAT_SAMPLE_MULTINOMIAL = 1, SAT_SAMPLE_TOPK = 2 };


// sample_method = "multinomial" (model.py:360-364), steps > 0: the reference draws kc flat indices from
// softmax(20 * seq_scores / step, dim=1).reshape(-1).  Per row: key_v = y_v - logsumexp(y) + Gumbel, y = 20 * log_softmax(x)_v / step
// (the parent score is constant inside a row and cancels in the row's softmax); the row's kc largest keys are emitted in
// descending order together with the candidates' scores (log-prob + parent score); beam_update_kernel merges the rows by key.
__global__ void __launch_bounds__(256)
row_sample_kernel(const float* __restrict__ logits, const float* __restrict__ top_scores, const int32_t* __restrict__ kcur, int k,
                  int kcap, int V, int step, float temp, int tokPAD, int tokSTART, uint64_t seed, float* __restrict__ cand_key,
                  float* __restrict__ cand_val, int32_t* __restrict__ cand_idx) {
  SAT_PDL_TRIGGER();
  SAT_PDL_WAIT();
  extern __shared__ __align__(16) float smem[];
  float* x = smem;            // [V] scaled logits (masked entries -inf)
  float* key = x + V;         // [V] sampling keys
  float* scratch = key + V;   // [33]
  __shared__ float s_val[8];
  __shared__ int s_idx[8];
  const int r = blockIdx.x, n = r / k, j = r - n * k, tid = threadIdx.x;
  const int kc = kcur[n];
  if (j >= kc) return;
  const float* row = logits + (int64_t)r * V;
  float mx = -INFINITY;
  for (int v = tid * 4; v < V; v += 256 * 4) {
    float4 q = *reinterpret_cast<const float4*>(row + v);
    q.x = q.x / temp; q.y = q.y / temp; q.z = q.z / temp; q.w = q.w / temp;
    *reinterpret_cast<float4*>(x + v) = q;
    mx = fmaxf(fmaxf(mx, fmaxf(q.x, q.y)), fmaxf(q.z, q.w));
  }
  mx = block_max(mx, scratch);
  float se = 0.0f;
  for (int v = tid; v < V; v += 256) {
    se += expf(x[v] - mx);
    if (v == tokSTART || v == tokPAD) x[v] = -INFINITY;            // model.py:333
  }
  se = block_sum(se, scratch);
  const float lse = logf(se);
  const float sharp = 20.0f / (float)step;                          // model.py:363
  float my = -INFINITY;
  for (int v = tid; v < V; v += 256) {
    const float y = sharp * ((x[v] - mx) - lse);                    // -inf for masked / padded words
    key[v] = y;
    my = fmaxf(my, y);
  }
  my = block_max(my, scratch);
  float se2 = 0.0f;
  for (int v = tid; v < V; v += 256) se2 += expf(key[v] - my);
  se2 = block_sum(se2, scratch);
  const float lse2 = my + logf(se2);
  for (int v = tid; v < V; v += 256) {
    const float y = key[v];
    key[v] = y > -INFINITY ? (y - lse2) + sat_gumbel(seed, (uint32_t)step, (uint64_t)r * (uint64_t)V + v) : -INFINITY;
  }
  __syncthreads();
  const float base = top_scores[r];
  float pv = INFINITY;
  int pi = -1;
  for (int i = 0; i < kc; ++i) {
    float bv = -INFINITY;
    int bi = 0x7fffffff;
    for (int v = tid; v < V; v += 256) {
      const float kv = key[v];
      const bool after = (kv < pv) || (kv == pv && v > pi);
      if (after && (kv > bv || (kv == bv && v < bi))) { bv = kv; bi = v; }
    }
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    __syncthreads();
    if ((tid & 31) == 0) { s_val[tid >> 5] = bv; s_idx[tid >> 5] = bi; }
    __syncthreads();
    bv = s_val[0]; bi = s_idx[0];
    for (int w = 1; w < 8; ++w)
      if (s_val[w] > bv || (s_val[w] == bv && s_idx[w] < bi)) { bv = s_val[w]; bi = s_idx[w]; }
    if (tid == 0) {
      const bool ok = bi != 0x7fffffff && bv > -INFINITY;
      cand_key[(int64_t)r * kcap + i] = ok ? bv : -INFINITY;
      cand_val[(int64_t)r * kcap + i] = ok ? ((x[bi] - mx) - lse) + base : -INFINITY;
      cand_idx[(int64_t)r * kcap + i] = ok ? bi : 0;
    }
    pv = bv; pi = bi;
  }
}

// decoder_noise (model.py:322-324): h += randn * noise / (step + 1) right before the LSTM cell -- only the recurrent
// projection W_hh h sees it (attention and the beta gate were computed from the clean state).  Box-Muller on the stateless hash.
template <typename T>
__global__ void __launch_bounds__(256) noisy_state_kernel(const T* __restrict__ h, T* __restrict__ h_noisy, int64_t n, float sigma,
                                                          uint64_t seed, int step) {
  SAT_PDL_TRIGGER();
  SAT_PDL_WAIT();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float u1 = sat_uniform01(seed, 0x40000000u + (uint32_t)step, 2 * (uint64_t)i);
  const float u2 = sat_uniform01(seed, 0x40000000u + (uint32_t)step, 2 * (uint64_t)i + 1);
  const float g = sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
  h_noisy[i] = from_f<T>(to_f(h[i]) + sigma * g);
}

struct BeamParams {
  int k, V, S;                 // beam width, vocab, max_gen_length
  int tokEND;
  int rescore;                 // SAT_RESCORE_*
  float reward;
  int hist_ld;                 // S + 1 entries per slot
  int kcap;                    // candidates stored per row (row pitch of cand_*): max(k, sample_topk)
  int sample;                  // SAT_SAMPLE_*
  int sample_topk;             // candidates per row of the "topk" sampler
  uint64_t seed;
};

// One warp per image.  Lane 0 performs the (tiny) merge; all lanes copy histories.
__global__ void __launch_bounds__(32)
beam_update_kernel(BeamParams p, int step, const float* __restrict__ cand_val, const float* __restrict__ cand_key,
                   const int32_t* __restrict__ cand_idx,
                   int32_t* __restrict__ kcur, float* __restrict__ top_scores, int32_t* __restrict__ cur_tok,
                   int32_t* __restrict__ src_row, int32_t* __restrict__ alive, const int32_t* __restrict__ tok_in,
                   const int32_t* __restrict__ asrc_in, int32_t* __restrict__ tok_out, int32_t* __restrict__ asrc_out,
                   int32_t* __restrict__ fin_tokens, int32_t* __restrict__ fin_asrc, int32_t* __restrict__ fin_len,
                   float* __restrict__ fin_score, float* __restrict__ fin_ppl, int32_t* __restrict__ fin_count,
                   int32_t* __restrict__ live_images, volatile int32_t* done_host, int call_id) {
  SAT_PDL_TRIGGER();
  SAT_PDL_WAIT();
  constexpr int KMAX = 32;
  __shared__ float nval[KMAX];
  __shared__ int nword[KMAX], nsrc[KMAX], dst[KMAX];
  __shared__ int s_kc_new, s_nnew;
  __shared__ float s_mean_all, s_mean_live;
  const int n = blockIdx.x, lane = threadIdx.x, k = p.k;
  const int kc = kcur[n];
  if (kc == 0) return;
  const int64_t r0 = (int64_t)n * k;
  if (lane == 0) {
    int nnew;
    const int cp = p.kcap;                                 // candidates per row in cand_* (row pitch)
    if (step == 0) {
      nnew = k;
      for (int i = 0; i < k; ++i) { nval[i] = cand_val[r0 * cp + i]; nword[i] = cand_idx[r0 * cp + i]; nsrc[i] = i; }
    } else if (p.sample == SAT_SAMPLE_TOPK) {
      // "topk" sampler (model.py:365-379): every live beam offers its sample_topk best words; kc of these kc * sample_topk
      // candidates are drawn without replacement with probability softmax(score / step): Gumbel-top-k over the candidates
      nnew = kc;
      const int tk = p.sample_topk;
      unsigned long long taken[KMAX * KMAX / 64 + 1];
      for (int w = 0; w < KMAX * KMAX / 64 + 1; ++w) taken[w] = 0ull;
      for (int i = 0; i < kc; ++i) {
        int bj = -1, bc = 0;
        float bkey = -INFINITY;
        for (int j = 0; j < kc; ++j) {
          for (int c = 0; c < tk; ++c) {
            const int f = j * tk + c;
            if ((taken[f >> 6] >> (f & 63)) & 1ull) continue;
            const float v = cand_val[(r0 + j) * cp + c];
            if (!(v > -INFINITY)) continue;
            const float key = v / (float)step + sat_gumbel(p.seed, 0x20000000u + (uint32_t)step, (uint64_t)(r0 + j) * (uint64_t)cp + c);
            if (bj < 0 || key > bkey) { bj = j; bc = c; bkey = key; }
          }
        }
        if (bj < 0) { bj = 0; bc = 0; }
        const int f = bj * tk + bc;
        taken[f >> 6] |= 1ull << (f & 63);
        nval[i] = cand_val[(r0 + bj) * cp + bc]; nword[i] = cand_idx[(r0 + bj) * cp + bc]; nsrc[i] = bj;
      }
    } else {
      // beam search: top-kc of the flattened [kc*V] scores (model.py:359); "multinomial": the kc largest sampling keys.  Every
      // row's candidates are sorted by that criterion, so this is a kc-way merge.
      const float* ckey = (p.sample == SAT_SAMPLE_MULTINOMIAL && cand_key != nullptr) ? cand_key : cand_val;
      nnew = kc;
      int ptr[KMAX];
      for (int j = 0; j < kc; ++j) ptr[j] = 0;
      for (int i = 0; i < kc; ++i) {
        int bj = -1;
        float bv = 0.f;
        for (int j = 0; j < kc; ++j) {
          if (ptr[j] >= kc) continue;
          const float v = ckey[(r0 + j) * cp + ptr[j]];
          if (bj < 0 || v > bv) { bj = j; bv = v; }       // j ascending => lower flat index wins ties
        }
        nval[i] = cand_val[(r0 + bj) * cp + ptr[bj]]; nword[i] = cand_idx[(r0 + bj) * cp + ptr[bj]]; nsrc[i] = bj;
        ++ptr[bj];
      }
    }
    int live = 0;
    for (int i = 0; i < nnew; ++i) dst[i] = (nword[i] == p.tokEND) ? -1 : live++;
    // BAR rescoring uses mean(top_scores) as the variable stands when rescore() is called (model.py:414):
    // the whole new beam for hypotheses that just ended, the survivors only for the max-length flush.
    float mean_all = 0.0f, mean_live = 0.0f;
    for (int i = 0; i < nnew; ++i) {
      mean_all += nval[i];
      if (dst[i] >= 0) mean_live += nval[i];
    }
    s_mean_all = mean_all / (float)nnew;
    s_mean_live = live > 0 ? mean_live / (float)live : 0.0f;
    s_kc_new = live;
    s_nnew = nnew;
  }
  __syncwarp();
  const int nnew = s_nnew;
  const bool flush = step >= p.S;                       // model.py:441
  const float fstep = (float)step;
  for (int i = 0; i < nnew; ++i) {
    const int64_t rs = r0 + nsrc[i];
    const bool done = dst[i] < 0;
    if (done || flush) {
      // finished hypothesis: words / alphas of steps 0..step-1 along the ancestry ([1:-1], model.py:421,442)
      int slot = 0;
      if (lane == 0) slot = fin_count[n];
      slot = __shfl_sync(0xffffffffu, slot, 0);
      // completed ones of this step are appended first (in beam order), flushed survivors after them
      if (!done) {
        int ndone = 0;
        for (int q = 0; q < nnew; ++q) ndone += dst[q] < 0;
        slot += ndone + dst[i];
      } else {
        int before = 0;
        for (int q = 0; q < i; ++q) before += dst[q] < 0;
        slot += before;
      }
      const int64_t fo = ((int64_t)n * k + slot) * p.hist_ld;
      for (int s = lane; s < step; s += 32) {
        fin_tokens[fo + s] = tok_in[rs * p.hist_ld + s];
        fin_asrc[fo + s] = asrc_in[rs * p.hist_ld + s];
      }
      if (lane == 0) {
        const float v = nval[i];
        float sc = v;
        if (p.rescore == SAT_RESCORE_LN) sc = v / fstep;
        else if (p.rescore == SAT_RESCORE_WR) sc = v + p.reward * fstep;
        else if (p.rescore == SAT_RESCORE_BAR) sc = v + p.reward * (-(done ? s_mean_all : s_mean_live));
        fin_len[(int64_t)n * k + slot] = step;
        fin_score[(int64_t)n * k + slot] = sc;
        fin_ppl[(int64_t)n * k + slot] = expf(-v / fstep);
      }
    }
    if (!done && !flush) {
      const int64_t rd = r0 + dst[i];
      for (int s = lane; s < step; s += 32) {
        tok_out[rd * p.hist_ld + s] = tok_in[rs * p.hist_ld + s];
        asrc_out[rd * p.hist_ld + s] = asrc_in[rs * p.hist_ld + s];
      }
      if (lane == 0) {
        tok_out[rd * p.hist_ld + step] = nword[i];
        asrc_out[rd * p.hist_ld + step] = (int)rs;
        top_scores[rd] = nval[i];
        cur_tok[rd] = nword[i];
        src_row[rd] = (int)rs;
      }
    }
  }
  __syncwarp();
  if (lane == 0) {
    fin_count[n] += flush ? nnew : (nnew - s_kc_new);
    kcur[n] = flush ? 0 : s_kc_new;
    // this image just used up its beams (it had kc > 0 on entry): the last image to do so tells the host's launch loop
    if ((flush || s_kc_new == 0) && live_images != nullptr && atomicSub(live_images, 1) == 1 && done_host != nullptr) {
      *done_host = call_id;
      __threadfence_system();
    }
  }
  const int kc_after = flush ? 0 : s_kc_new;
  for (int j = lane; j < k; j += 32) alive[r0 + j] = j < kc_after ? SAT_ALIVE : 0;
}

// h, c <- hn, cn gathered by source row (model.py:397); dead rows are left alone.
template <typename T>
__global__ void gather_state_kernel(const T* __restrict__ hn, const float* __restrict__ cn, const int32_t* __restrict__ src_row,
                                    const int32_t* __restrict__ alive, T* __restrict__ h, float* __restrict__ c, int R, int H, int nl) {
  SAT_PDL_TRIGGER();
  SAT_PDL_WAIT();
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;      // over [layers, R, H]: R = rows of ONE layer
  const int64_t RH = (int64_t)R * H;
  const int64_t l = idx / RH, rem = idx - l * RH;
  if (l >= nl) return;
  const int64_t r = rem / H;
  if (alive[r] == 0) return;
  const int j = (int)(rem - r * H);
  const int64_t s = src_row[r];
  h[idx] = hn[l * RH + s * H + j];
  c[idx] = cn[l * RH + s * H + j];
}

static __global__ void decode_init_kernel(int32_t* cur_tok, int32_t* alive, float* top_scores, int32_t* kcur, int32_t* fin_count,
                                          int32_t* fin_len, int R, int n_img, int k, int tokSTART, int32_t* live_images) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0 && live_images != nullptr) *live_images = n_img;
  if (i < R) {
    cur_tok[i] = tokSTART;
    alive[i] = SAT_ALIVE;
    top_scores[i] = 0.0f;
    fin_len[i] = 0;
  }
  if (i < n_img) {
    kcur[i] = k;
    fin_count[i] = 0;
  }
}
