// Non-GEMM kernels of the SAT decoder hot path (sm_100a): fused attention step (forward/backward),
// row-wise cross-entropy, state initialisation, gathers and the small deterministic reductions.
#pragma once
#include "sat_common.cuh"

constexpr int ATT_THREADS = 256;

// =============================================================================================
// K1  fused attention step, forward.   One CTA per caption row b (rows with t >= lens[b] write zeros).
//   e_l   = (sum_a wf[a] * tanh(P[img,l,a] + q[a])) * L^-0.5        model.py:104
//   alpha = softmax_l(e)                                             model.py:106
//   z     = sum_l alpha_l * ann[img,l,:]                             model.py:108
//   beta  = sigmoid(beta_pre) ; gz = beta * z                        model.py:538-541
// q and beta_pre (bias included) come from the h-projection GEMM (hp[b, 0:A], hp[b, A:A+D]).
// Algorithmic traffic per active row: L*(A+D)*sizeof(T) read once + (A+2D) small vectors + L floats out.
// =============================================================================================
template <typename T, bool kExact>
__global__ void __launch_bounds__(ATT_THREADS)
attention_step_fwd_kernel(const T* __restrict__ ann, const T* __restrict__ P, const float* __restrict__ wf,
                          const float* __restrict__ hp, int64_t ldhp, const int32_t* __restrict__ lens, int t,
                          int ncap, int L, int D, int A, float scale, float* __restrict__ alpha, int64_t ld_alpha,
                          float* __restrict__ qsave, T* __restrict__ z, T* __restrict__ gz, T* __restrict__ beta,
                          int64_t ld_z) {
  extern __shared__ __align__(16) float smem[];
  constexpr int VN = Vec16<T>::N;
  const int NV = D / VN;
  const int RG = NV >= ATT_THREADS ? 1 : ATT_THREADS / NV;
  float* e = smem;                 // [L]
  float* qs = e + ((L + 3) & ~3);  // [A]
  float* ws = qs + A;              // [A]
  float* red = ws + A;             // [RG*D]
  float* scratch = red + RG * D;   // [33]

  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool active = lens == nullptr || t < lens[b];
  float* alpha_b = alpha + (int64_t)b * ld_alpha;
  if (!active) {
    for (int l = tid; l < L; l += ATT_THREADS) alpha_b[l] = 0.0f;
    for (int d = tid; d < D; d += ATT_THREADS) {
      z[(int64_t)b * ld_z + d] = from_f<T>(0.f);
      gz[(int64_t)b * ld_z + d] = from_f<T>(0.f);
      if (beta) beta[(int64_t)b * ld_z + d] = from_f<T>(0.f);
    }
    if (qsave) for (int a = tid; a < A; a += ATT_THREADS) qsave[(int64_t)b * A + a] = 0.0f;
    return;
  }
  const int img = b / ncap;
  const float* hp_b = hp + (int64_t)b * ldhp;
  for (int a = tid; a < A; a += ATT_THREADS) {
    const float q = hp_b[a];
    qs[a] = q;
    ws[a] = wf[a];
    if (qsave) qsave[(int64_t)b * A + a] = q;
  }
  __syncthreads();

  // ---- phase 1: scores (one warp per location, lanes over attention_dim; 4 rows in flight per warp) ---
  const T* Pb = P + (int64_t)img * L * A;
  constexpr int NWARP = ATT_THREADS / 32;
  for (int l0 = warp; l0 < L; l0 += 4 * NWARP) {
    float s[4] = {0.f, 0.f, 0.f, 0.f};
    for (int a = lane * 4; a < A; a += 128) {
      float4 p[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int l = l0 + u * NWARP;
        p[u] = l < L ? ld4(Pb + (int64_t)l * A + a) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        s[u] = fmaf(ws[a + 0], sat_tanh<kExact>(p[u].x + qs[a + 0]), s[u]);
        s[u] = fmaf(ws[a + 1], sat_tanh<kExact>(p[u].y + qs[a + 1]), s[u]);
        s[u] = fmaf(ws[a + 2], sat_tanh<kExact>(p[u].z + qs[a + 2]), s[u]);
        s[u] = fmaf(ws[a + 3], sat_tanh<kExact>(p[u].w + qs[a + 3]), s[u]);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int l = l0 + u * NWARP;
      const float r = warp_sum(s[u]);
      if (lane == 0 && l < L) e[l] = r * scale;
    }
  }
  __syncthreads();

  // ---- phase 2: softmax over L --------------------------------------------------------------
  float mx = -INFINITY;
  for (int l = tid; l < L; l += ATT_THREADS) mx = fmaxf(mx, e[l]);
  mx = block_max(mx, scratch);
  float sum = 0.0f;
  for (int l = tid; l < L; l += ATT_THREADS) {
    const float p = sat_exp<kExact>(e[l] - mx);
    e[l] = p;
    sum += p;
  }
  sum = block_sum(sum, scratch);
  for (int l = tid; l < L; l += ATT_THREADS) {
    const float al = e[l] / sum;
    e[l] = al;
    alpha_b[l] = al;
  }
  __syncthreads();

  // ---- phase 3: context z = sum_l alpha_l * a_l (16-byte loads, RG row groups) ----------------
  const T* ab = ann + (int64_t)img * L * D;
  if (RG == 1) {
    for (int cv = tid; cv < NV; cv += ATT_THREADS) {
      float acc[VN];
#pragma unroll
      for (int i = 0; i < VN; ++i) acc[i] = 0.0f;
      int l = 0;
      for (; l + 4 <= L; l += 4) {
        float v[4][VN];
#pragma unroll
        for (int u = 0; u < 4; ++u) Vec16<T>::load(ab + (int64_t)(l + u) * D + cv * VN, v[u]);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float al = e[l + u];
#pragma unroll
          for (int i = 0; i < VN; ++i) acc[i] = fmaf(al, v[u][i], acc[i]);
        }
      }
      for (; l < L; ++l) {
        float v[VN];
        Vec16<T>::load(ab + (int64_t)l * D + cv * VN, v);
        const float al = e[l];
#pragma unroll
        for (int i = 0; i < VN; ++i) acc[i] = fmaf(al, v[i], acc[i]);
      }
#pragma unroll
      for (int i = 0; i < VN; ++i) red[cv * VN + i] = acc[i];
    }
  } else {
    const int rg = tid / NV, cv = tid - rg * NV;
    if (rg < RG) {
      float acc[VN];
#pragma unroll
      for (int i = 0; i < VN; ++i) acc[i] = 0.0f;
      int l = rg;
      for (; l + 3 * RG < L; l += 4 * RG) {
        float v[4][VN];
#pragma unroll
        for (int u = 0; u < 4; ++u) Vec16<T>::load(ab + (int64_t)(l + u * RG) * D + cv * VN, v[u]);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float al = e[l + u * RG];
#pragma unroll
          for (int i = 0; i < VN; ++i) acc[i] = fmaf(al, v[u][i], acc[i]);
        }
      }
      for (; l < L; l += RG) {
        float v[VN];
        Vec16<T>::load(ab + (int64_t)l * D + cv * VN, v);
        const float al = e[l];
#pragma unroll
        for (int i = 0; i < VN; ++i) acc[i] = fmaf(al, v[i], acc[i]);
      }
#pragma unroll
      for (int i = 0; i < VN; ++i) red[rg * D + cv * VN + i] = acc[i];
    }
  }
  __syncthreads();
  for (int d = tid; d < D; d += ATT_THREADS) {
    float zs = 0.0f;
    for (int r = 0; r < RG; ++r) zs += red[r * D + d];
    const float bt = sat_sigmoid<kExact>(hp_b[A + d]);
    z[(int64_t)b * ld_z + d] = from_f<T>(zs);
    gz[(int64_t)b * ld_z + d] = from_f<T>(bt * zs);
    if (beta) beta[(int64_t)b * ld_z + d] = from_f<T>(bt);
  }
}

static inline size_t attention_fwd_smem(int L, int D, int A, int vn) {
  const int NV = D / vn;
  const int RG = NV >= ATT_THREADS ? 1 : ATT_THREADS / NV;
  return sizeof(float) * (size_t)(((L + 3) & ~3) + 2 * A + RG * D + 40);
}

// =============================================================================================
// mean over locations: meanv[i,d] = (1/L) sum_l ann[i,l,d]                        model.py:78
// =============================================================================================
template <typename T>
__global__ void __launch_bounds__(256) mean_L_kernel(const T* __restrict__ ann, T* __restrict__ meanv, int L, int D, float drop_p,
                                                      uint64_t seed) {
  // CTA = (32 column vectors) x (8 row groups); partial sums of the row groups are combined through shared memory
  constexpr int VN = Vec16<T>::N;
  __shared__ float part[8][32][VN + 1];
  const int NV = D / VN;
  const int cl = threadIdx.x & 31, rg = threadIdx.x >> 5;
  const int cv = blockIdx.x * 32 + cl;
  const int i = blockIdx.y;
  float acc[VN];
#pragma unroll
  for (int k = 0; k < VN; ++k) acc[k] = 0.0f;
  if (cv < NV) {
    const T* a = ann + (int64_t)i * L * D + cv * VN;
    for (int l = rg; l < L; l += 8) {
      float v[VN];
      Vec16<T>::load(a + (int64_t)l * D, v);
#pragma unroll
      for (int k = 0; k < VN; ++k) acc[k] += v[k];
    }
  }
#pragma unroll
  for (int k = 0; k < VN; ++k) part[rg][cl][k] = acc[k];
  __syncthreads();
  if (rg == 0 && cv < NV) {
    const float inv = 1.0f / (float)L;
#pragma unroll
    for (int k = 0; k < VN; ++k) {
      float sum = 0.0f;
#pragma unroll
      for (int r = 0; r < 8; ++r) sum += part[r][cl][k];
      acc[k] = sum * inv * sat_dropout_scale(drop_p, seed, 1u, (uint64_t)i * D + cv * VN + k);    // model.py:78
    }
    Vec16<T>::store(meanv + (int64_t)i * D + cv * VN, acc);
  }
}

// =============================================================================================
// InitLSTM state reinterpretation (model.py:79-80): the [B,2H] init output (row b = image b/ncap)
// is read row-major as [2,B,H]:  h0[b,j] = flat[b*H+j],  c0[b,j] = flat[(B+b)*H+j].
// =============================================================================================
template <typename T>
__global__ void init_state_kernel(const float* __restrict__ init_out, int64_t ld_io, T* __restrict__ h0, float* __restrict__ c0,
                                  int64_t ld_h, int64_t ld_c, int64_t lstride_h, int64_t lstride_c, int B, int H, int ncap, int nl) {
  // H is the module's TRUE decoder_dim (the reinterpretation mixes rows and columns, so it must not see the padding);
  // ld_io / ld_h / ld_c are the storage pitches, lstride_* the distance between the layers' state arrays.  The [B, 2*nl*H]
  // init output is read row-major as [2*nl, B, H]: states 0..nl-1 are h of the layers, nl..2nl-1 their c (model.py:79-80).
  // Padded state columns are zeroed by the caller.
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t BH = (int64_t)B * H;
  if (idx >= 2 * nl * BH) return;
  const int64_t r = idx / (2 * nl * H);     // row of the (virtual) repeated [B, 2*nl*H] matrix
  const int col = (int)(idx - r * 2 * nl * H);
  const float v = init_out[(r / ncap) * ld_io + col];
  const int st = (int)(idx / BH);
  const int64_t g = idx - (int64_t)st * BH;
  const int64_t b = g / H;
  const int j = (int)(g - b * H);
  if (st < nl) h0[st * lstride_h + b * ld_h + j] = from_f<T>(v);
  else c0[(st - nl) * lstride_c + b * ld_c + j] = v;
}

// inverse of the above for the backward pass: d_init_out[i, col] = sum over the ncap caption rows of image i of the state
// gradient that element fed.  dh0 of layer l: ns_dh[l] split-K partials at dh0[l] (see the backward driver); dc0: [nl,B,ld_st].
struct InitBwdSrc {
  const float* p[SAT_MAX_LAYERS][2];   // up to two partial sets per layer (recurrent GEMM, q/beta GEMM)
  int ns[SAT_MAX_LAYERS][2];
  int64_t stride[SAT_MAX_LAYERS][2];   // distance between partials
  int64_t ld[SAT_MAX_LAYERS][2];       // row pitch
};
static __global__ void init_state_bwd_kernel(const __grid_constant__ InitBwdSrc src, const float* __restrict__ dc0, int64_t ld_st,
                                             int64_t lstride_c, float* __restrict__ d_init_out, bf16* __restrict__ d_init_out16,
                                             int64_t ld_io, int B, int H, int ncap, int nl) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // over [Bi, ld_io]
  const int Bi = B / ncap;
  if (idx >= (int64_t)Bi * ld_io) return;
  const int64_t i = idx / ld_io;
  const int col = (int)(idx - i * ld_io);
  const int64_t BH = (int64_t)B * H;
  float s = 0.0f;
  if (col < 2 * nl * H) {
    for (int c = 0; c < ncap; ++c) {
      const int64_t r = i * ncap + c;
      const int64_t f = r * 2 * nl * H + col;     // flat index into the [2*nl,B,H] view
      const int st = (int)(f / BH);
      const int64_t g = f - (int64_t)st * BH;
      const int64_t b = g / H, j = g - b * H;
      if (st < nl) {
        for (int q = 0; q < 2; ++q)
          for (int sp = 0; sp < src.ns[st][q]; ++sp) s += src.p[st][q][(int64_t)sp * src.stride[st][q] + b * src.ld[st][q] + j];
      } else {
        s += dc0[(st - nl) * lstride_c + b * ld_st + j];
      }
    }
  }
  d_init_out[idx] = s;
  if (d_init_out16) d_init_out16[idx] = __float2bfloat16_rn(s);
}

// =============================================================================================
// previous-word ids, time-major: tok[t,b] = caps[b,t]   (teacher forcing, model.py:520)
// =============================================================================================
static __global__ void tok_init_kernel(const int32_t* __restrict__ caps, int32_t* __restrict__ tok, int B, int T_, int caplen, int V0,
                                       float* __restrict__ err_flag) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= T_ * B) return;
  const int t = m / B, b = m - t * B;
  const int w = caps[(int64_t)b * caplen + t];
  if ((unsigned)w >= (unsigned)V0) *err_flag = 1.0f;     // nn.Embedding would raise; here the word is fed as <PAD>, flagged (out[6])
  tok[m] = sat_word_or_pad(w, V0);
}

// the dataset hands out int64 word ids / lengths (torch.LongTensor, util.py:43-44); the kernels index with int32
static __global__ void cast_captions_kernel(const int64_t* __restrict__ caps64, const int64_t* __restrict__ lens64, int32_t* __restrict__ caps32,
                                            int32_t* __restrict__ lens32, int64_t n_caps, int64_t n_lens) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_caps) caps32[i] = (int32_t)caps64[i];
  else if (i < n_caps + n_lens) lens32[i - n_caps] = (int32_t)lens64[i - n_caps];
}

// =============================================================================================
// embedding gather over `rows` time-major rows:  Xe[m,:] = Emb[tok[m],:]                 model.py:526
// =============================================================================================
template <typename T>
__global__ void embed_gather_kernel(const T* __restrict__ Emb, const int32_t* __restrict__ tok, T* __restrict__ Xe, int E,
                                    int64_t m_base, float drop_p, uint64_t seed) {
  const int m = blockIdx.x;            // row of this launch; m_base + m is the global time-major row (dropout index)
  const int w = tok[m];
  constexpr int VN = Vec16<T>::N;
  for (int c = threadIdx.x; c < E / VN; c += blockDim.x) {
    if (drop_p <= 0.0f) {
      const uint4 v = *reinterpret_cast<const uint4*>(Emb + (int64_t)w * E + c * VN);
      *reinterpret_cast<uint4*>(Xe + (int64_t)m * E + c * VN) = v;
    } else {                          // embedding_dropout (model.py:526)
      float v[VN];
      Vec16<T>::load(Emb + (int64_t)w * E + c * VN, v);
#pragma unroll
      for (int k = 0; k < VN; ++k) v[k] *= sat_dropout_scale(drop_p, seed, 2u, (uint64_t)(m_base + m) * E + c * VN + k);
      Vec16<T>::store(Xe + (int64_t)m * E + c * VN, v);
    }
  }
}

// x[i] *= dropout multiplier of (stream, i): backward of the InitLSTM-mean and embedding dropouts
static __global__ void dropout_bwd_kernel(float* __restrict__ x, int64_t n, float drop_p, uint64_t seed, uint32_t stream) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] *= sat_dropout_scale(drop_p, seed, stream, (uint64_t)i);
}

// =============================================================================================
// scheduled sampling feedback: tok[b] = argmax_v logits[b,:] (first maximal index, like torch.argmax, model.py:523)
// =============================================================================================
template <typename TL>
__global__ void __launch_bounds__(256) row_argmax_kernel(const TL* __restrict__ logits, int32_t* __restrict__ tok, int V) {
  __shared__ float s_val[8];
  __shared__ int s_arg[8];
  const int b = blockIdx.x, tid = threadIdx.x;
  const TL* row = logits + (int64_t)b * V;
  float mx = -INFINITY;
  int arg = 0x7fffffff;
  for (int v = tid; v < V; v += 256) {
    const float xv = to_f(row[v]);
    if (xv > mx) { mx = xv; arg = v; }
  }
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, mx, o);
    const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
    if (om > mx || (om == mx && oa < arg)) { mx = om; arg = oa; }
  }
  if ((tid & 31) == 0) { s_val[tid >> 5] = mx; s_arg[tid >> 5] = arg; }
  __syncthreads();
  if (tid == 0) {
    mx = s_val[0]; arg = s_arg[0];
    for (int w = 1; w < 8; ++w)
      if (s_val[w] > mx || (s_val[w] == mx && s_arg[w] < arg)) { mx = s_val[w]; arg = s_arg[w]; }
    tok[b] = arg == 0x7fffffff ? 0 : arg;
  }
}

// =============================================================================================
// row-wise cross entropy with label smoothing + argmax + dlogits (util.py:105-112, model.py:596)
//   rows are time-major m = t*B + b;  inactive rows (t >= lens[b]) give zeros (model.py:504,548).
//   loss_row = (1-s)*(lse - x_y) + s*(lse - mean_v x)
//   dlogits  = (softmax - (1-s)*onehot(y) - s/V) * inv_ntok
// =============================================================================================
template <typename TL, typename TD, bool kExact>
__global__ void __launch_bounds__(256)
ce_rows_kernel(TL* __restrict__ logits, TD* __restrict__ dlogits, const int32_t* __restrict__ caps,
               const int32_t* __restrict__ lens, const float* __restrict__ inv_ntok_p, float* __restrict__ row_loss,
               int32_t* __restrict__ row_argmax, int B, int V0, int V, int caplen, float smoothing, int zero_inactive_logits) {
  // V0 = true vocabulary, V = storage row pitch (multiple of 8).  Padded entries hold -inf logits (bias padding): they drop
  // out of the max / sum of exponentials by themselves, are skipped in the sum of logits, and get a zero gradient.
  extern __shared__ __align__(16) float smem[];
  float* x = smem;              // [V]
  float* scratch = x + V;       // [33]
  __shared__ int s_arg[8];
  __shared__ float s_val[8];
  const int m = blockIdx.x, t = m / B, b = m - t * B, tid = threadIdx.x;
  TL* row = logits + (int64_t)m * V;
  const bool active = t < lens[b];
  if (!active) {
    if (zero_inactive_logits) for (int v = tid; v < V; v += 256) row[v] = from_f<TL>(0.f);
    if (dlogits) for (int v = tid; v < V; v += 256) dlogits[(int64_t)m * V + v] = from_f<TD>(0.f);
    if (tid == 0) { row_loss[m] = 0.0f; row_argmax[m] = -1; }
    return;
  }
  const int y = sat_word_or_pad(caps[(int64_t)b * caplen + t + 1], V0);
  float mx = -INFINITY, sx = 0.0f;
  int arg = 0x7fffffff;
  for (int v = tid * 4; v < V; v += 256 * 4) {      // 4 logits per access (rows are 16 B (bf16) / 32 B (fp32) aligned)
    const float4 q = ld4(row + v);
    *reinterpret_cast<float4*>(x + v) = q;
    sx += ((v < V0 ? q.x : 0.f) + (v + 1 < V0 ? q.y : 0.f)) + ((v + 2 < V0 ? q.z : 0.f) + (v + 3 < V0 ? q.w : 0.f));
    if (q.x > mx) { mx = q.x; arg = v; }
    if (q.y > mx) { mx = q.y; arg = v + 1; }
    if (q.z > mx) { mx = q.z; arg = v + 2; }
    if (q.w > mx) { mx = q.w; arg = v + 3; }
  }
  // block argmax with lowest-index tie break (torch.argmax returns the first maximal index)
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, mx, o);
    const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
    if (om > mx || (om == mx && oa < arg)) { mx = om; arg = oa; }
  }
  if ((tid & 31) == 0) { s_val[tid >> 5] = mx; s_arg[tid >> 5] = arg; }
  __syncthreads();
  mx = s_val[0]; arg = s_arg[0];
  for (int w = 1; w < 8; ++w)
    if (s_val[w] > mx || (s_val[w] == mx && s_arg[w] < arg)) { mx = s_val[w]; arg = s_arg[w]; }
  float se = 0.0f;
  for (int v = tid * 4; v < V; v += 256 * 4) {
    const float4 q = *reinterpret_cast<const float4*>(x + v);
    se += (sat_exp<kExact>(q.x - mx) + sat_exp<kExact>(q.y - mx)) + (sat_exp<kExact>(q.z - mx) + sat_exp<kExact>(q.w - mx));
  }
  se = block_sum(se, scratch);
  sx = block_sum(sx, scratch);
  const float lse = mx + (kExact ? logf(se) : __logf(se));
  if (tid == 0) {
    const float nll = lse - x[y];
    const float smooth = lse - sx / (float)V0;
    row_loss[m] = (1.0f - smoothing) * nll + smoothing * smooth;
    row_argmax[m] = arg;
  }
  if (dlogits) {
    const float inv_ntok = *inv_ntok_p;
    const float sv = smoothing / (float)V0;
    TD* drow = dlogits + (int64_t)m * V;
    for (int v = tid * 4; v < V; v += 256 * 4) {
      const float4 q = *reinterpret_cast<const float4*>(x + v);
      float p0 = sat_exp<kExact>(q.x - lse) - sv, p1 = sat_exp<kExact>(q.y - lse) - sv;
      float p2 = sat_exp<kExact>(q.z - lse) - sv, p3 = sat_exp<kExact>(q.w - lse) - sv;
      if (y == v) p0 -= (1.0f - smoothing);
      if (y == v + 1) p1 -= (1.0f - smoothing);
      if (y == v + 2) p2 -= (1.0f - smoothing);
      if (y == v + 3) p3 -= (1.0f - smoothing);
      if (v >= V0) p0 = 0.f;
      if (v + 1 >= V0) p1 = 0.f;
      if (v + 2 >= V0) p2 = 0.f;
      if (v + 3 >= V0) p3 = 0.f;
      st4(drow + v, make_float4(p0 * inv_ntok, p1 * inv_ntok, p2 * inv_ntok, p3 * inv_ntok));
    }
  }
}

// ntok = sum_b lens[b] ; out[4] = 1/ntok        (single CTA)
static __global__ void ntok_kernel(const int32_t* __restrict__ lens, int B, float* __restrict__ out) {
  __shared__ int sh[32];
  int s = 0;
  for (int b = threadIdx.x; b < B; b += blockDim.x) s += lens[b];
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    int tot = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += sh[w];
    out[4] = 1.0f / (float)tot;
    out[5] = (float)tot;
  }
}

// S[b,l] = sum_t alphas[b,t,l]                                                  model.py:594
// also writes the CTA's partial of sum (1-S)^2 so that the final reduction touches gridDim.x values instead of B*L
static __global__ void __launch_bounds__(256)
alpha_sum_kernel(const float* __restrict__ alphas, float* __restrict__ S, float* __restrict__ reg_part, int B, int T_, int L) {
  __shared__ float scratch[33];
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float r = 0.0f;
  if (idx < (int64_t)B * L) {
    const int64_t b = idx / L;
    const int l = (int)(idx - b * L);
    float s = 0.0f;
    for (int t = 0; t < T_; ++t) s += alphas[(b * T_ + t) * L + l];
    S[idx] = s;
    r = (1.0f - s) * (1.0f - s);
  }
  r = block_sum(r, scratch);
  if (threadIdx.x == 0) reg_part[blockIdx.x] = r;
}

// loss = mean_tok(row_loss) + gamma * mean_{b,l} (1-S)^2 ; accuracy.  Single CTA, fixed summation order.
static __global__ void __launch_bounds__(1024)
loss_finalize_kernel(const float* __restrict__ row_loss, const int32_t* __restrict__ row_argmax,
                     const int32_t* __restrict__ tok_next, const int32_t* __restrict__ lens, const float* __restrict__ reg_part,
                     int nparts, int B, int T_, int L, int caplen, float gamma, float* __restrict__ out) {
  __shared__ float scratch[33];
  float ce = 0.0f, hit = 0.0f, reg = 0.0f;
  for (int m = threadIdx.x; m < B * T_; m += blockDim.x) {
    const int t = m / B, b = m - t * B;
    if (t < lens[b]) {
      ce += row_loss[m];
      hit += (row_argmax[m] == tok_next[(int64_t)b * caplen + t + 1]) ? 1.0f : 0.0f;
    }
  }
  for (int i = threadIdx.x; i < nparts; i += blockDim.x) reg += reg_part[i];
  ce = block_sum(ce, scratch);
  hit = block_sum(hit, scratch);
  reg = block_sum(reg, scratch);
  if (threadIdx.x == 0) {
    const float inv = out[4];
    const float cem = ce * inv, regm = reg / ((float)B * (float)L);
    out[0] = cem + gamma * regm;
    out[1] = cem;
    out[2] = regm;
    out[3] = hit * inv;
  }
}

// =============================================================================================
// LSTM cell backward for one step (elementwise over [B,H]); see SURVEY.md appendix E.
//   dh (in) = grad wrt h_{t+1} from later steps; dHo = grad from the deep-output path at step t.
//   Writes dG (gate-interleaved, pre-activation grads) into DY[t,:,A+D:], updates dc in place and
//   leaves dh untouched (the h-chain GEMM that follows overwrites it for active rows).
// =============================================================================================
struct DhSrc {                 // gradient contributions to this layer's new hidden state, summed in fixed order
  const float* p[3];           // partial sets: [ns][B rows at pitch ld][H]
  int ns[3];
  int64_t stride[3], ld[3];
};
template <typename TS, bool kExact>
__global__ void lstm_bwd_step_kernel(const TS* __restrict__ gates, const float* __restrict__ c_prev,
                                     const float* __restrict__ c_next, const __grid_constant__ DhSrc dh,
                                     const float* __restrict__ dHo, int64_t ld_dho, float* __restrict__ dc,
                                     TS* __restrict__ dG, int64_t ld_dg, const int32_t* __restrict__ lens, int t, int B,
                                     int H) {
  SAT_PDL_TRIGGER();
  SAT_PDL_WAIT();
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * H) return;
  const int b = idx / H, j = idx - b * H;
  TS* dg = dG + (int64_t)b * ld_dg + 4 * j;
  // every operand is fetched before the first dependent instruction (one exposed latency; all addresses are valid for
  // finished rows too)
  const int len_b = lens[b];
  const float4 g4 = ld4(gates + (int64_t)b * 4 * H + 4 * j);
  const float cp = c_prev[idx], cn = c_next[idx];
  const float dho = dHo ? dHo[(int64_t)b * ld_dho + j] : 0.0f, dc_in = dc[idx];
  float dhs = 0.0f;
#pragma unroll
  for (int q = 0; q < 3; ++q) {
    const float* base = dh.p[q] + (int64_t)b * dh.ld[q] + j;
    for (int sp0 = 0; sp0 < dh.ns[q]; sp0 += 8) {      // split-K partials, 8 loads in flight
      float p[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) p[u] = (sp0 + u) < dh.ns[q] ? base[(int64_t)(sp0 + u) * dh.stride[q]] : 0.0f;
#pragma unroll
      for (int u = 0; u < 8; ++u) dhs += p[u];
    }
  }
  if (t >= len_b) {
    st4(dg, make_float4(0.f, 0.f, 0.f, 0.f));
    return;
  }
  const float gi = g4.x, gf = g4.y, gg = g4.z, go = g4.w;
  const float tc = sat_tanh<kExact>(cn);
  const float dht = dhs + dho;
  const float dct = dc_in + dht * go * (1.0f - tc * tc);
  st4(dg, make_float4(dct * gg * gi * (1.0f - gi), dct * cp * gf * (1.0f - gf), dct * gi * (1.0f - gg * gg),
                      dht * tc * go * (1.0f - go)));
  dc[idx] = dct * gf;
}

// =============================================================================================
// K1b  fused attention step, backward.  One CTA per caption row b.
//   dz      = dZout + dgz * beta                      dbeta_pre = dgz * z * beta (1-beta)
//   dalpha_l= a_l . dz  +  g * gamma * (-2)(1 - S_l)/(B L)
//   de_l    = alpha_l (dalpha_l - sum_l' alpha_l' dalpha_l')
//   dpu_la  = scale * de_l * wf_a * (1 - u_la^2),  u = tanh(P + q)  (recomputed)
//   dP[b,l,a] += dpu ;  dq_a = sum_l dpu_la ;  dwf_a = scale * sum_l de_l u_la
// Algorithmic traffic per active row: L*(A+D)*sizeof(T) read + 2*L*A*4 (dP read-modify-write).
// =============================================================================================
// A lane keeps dq / dwf of the attention columns lane*4 + 128k, k < KA, in registers: the instantiation for KA serves
// attention_dim <= 128 * KA (KA = 4: A <= 512, KA = 8: A <= 1024, the training limit).
constexpr int ATTB_MAXKA = 8;   // attention_dim <= 1024

template <typename T, bool kExact, int KA = 4>
__global__ void __launch_bounds__(ATT_THREADS)
attention_step_bwd_kernel(const T* __restrict__ ann, const T* __restrict__ P, const float* __restrict__ wf,
                          const float* __restrict__ q_t, const float* __restrict__ alpha, int64_t ld_alpha,
                          const float* __restrict__ S, const T* __restrict__ z_t, const T* __restrict__ beta_t,
                          const float* __restrict__ dgz, int ns_dgz, int64_t dgz_stride,
                          const float* __restrict__ dZout, int64_t ld_dzout,
                          const int32_t* __restrict__ lens, int t, int ncap, int B, int L, int D, int A, float scale,
                          float gamma, const float* __restrict__ gscale, const float* __restrict__ dalpha_ext,
                          float* __restrict__ dP, T* __restrict__ dP16, T* __restrict__ dZ_t,
                          T* __restrict__ DY_t, int64_t ld_dy, float* __restrict__ dwf_t, float* /*de_t: pipelined kernel only*/) {
  extern __shared__ __align__(16) float smem[];
  constexpr int VN = Vec16<T>::N;
  constexpr int NW = ATT_THREADS / 32;
  SAT_PDL_TRIGGER();      // launched through sat_launch_pdl by the backward driver
  SAT_PDL_WAIT();
  float* dz_s = smem;                         // [D]
  float* dal = dz_s + D;                      // [L] (padded to 4)
  float* qs = dal + ((L + 3) & ~3);           // [A]
  float* ws = qs + A;                         // [A]
  float* red = ws + A;                        // [NW][2A]
  float* scratch = red + NW * 2 * A;          // [33]

  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  T* dy_b = DY_t + (int64_t)b * ld_dy;
  if (t >= lens[b]) {
    for (int i = tid; i < A + D; i += ATT_THREADS) dy_b[i] = from_f<T>(0.f);
    for (int d = tid; d < D; d += ATT_THREADS) dZ_t[(int64_t)b * D + d] = from_f<T>(0.f);
    for (int a = tid; a < A; a += ATT_THREADS) dwf_t[(int64_t)b * A + a] = 0.0f;
    return;
  }
  const int img = b / ncap;
  const float g = gscale ? *gscale : 1.0f;
  // phase A
  for (int d = tid; d < D; d += ATT_THREADS) {
    float dg = 0.0f;
    for (int sp = 0; sp < ns_dgz; ++sp) dg += dgz[(int64_t)sp * dgz_stride + (int64_t)b * D + d];
    const float bt = to_f(beta_t[(int64_t)b * D + d]);
    const float zz = to_f(z_t[(int64_t)b * D + d]);
    const float dzv = dZout[(int64_t)b * ld_dzout + d] + dg * bt;
    dz_s[d] = dzv;
    dZ_t[(int64_t)b * D + d] = from_f<T>(dzv);
    dy_b[A + d] = from_f<T>(dg * zz * bt * (1.0f - bt));
  }
  for (int a = tid; a < A; a += ATT_THREADS) {
    qs[a] = q_t[(int64_t)b * A + a];
    ws[a] = wf[a];
  }
  __syncthreads();
  // phase B: dalpha_l = a_l . dz + regulariser
  const T* ab = ann + (int64_t)img * L * D;
  const float* alpha_b = alpha + (int64_t)b * ld_alpha;
  const float regc = g * gamma * (-2.0f) / ((float)B * (float)L);
  const int NV = D / VN;
  for (int l = warp; l < L; l += NW) {
    float s = 0.0f;
    for (int cv = lane; cv < NV; cv += 32) {
      float v[VN];
      Vec16<T>::load(ab + (int64_t)l * D + cv * VN, v);
#pragma unroll
      for (int i = 0; i < VN; ++i) s = fmaf(v[i], dz_s[cv * VN + i], s);
    }
    s = warp_sum(s);
    if (lane == 0) {
      float v = s + regc * (1.0f - S[(int64_t)b * L + l]);
      if (dalpha_ext) v += dalpha_ext[(int64_t)b * ld_alpha + l];
      dal[l] = v;
    }
  }
  __syncthreads();
  // phase C: softmax backward
  float dot = 0.0f;
  for (int l = tid; l < L; l += ATT_THREADS) dot = fmaf(alpha_b[l], dal[l], dot);
  dot = block_sum(dot, scratch);
  for (int l = tid; l < L; l += ATT_THREADS) dal[l] = alpha_b[l] * (dal[l] - dot);   // de_l
  __syncthreads();
  // phase D: through tanh into P, q, wf
  const T* Pb = P + (int64_t)img * L * A;
  float* dPb = dP + (int64_t)b * L * A;
  float dq[KA][4], dw[KA][4];
#pragma unroll
  for (int k = 0; k < KA; ++k)
#pragma unroll
    for (int i = 0; i < 4; ++i) { dq[k][i] = 0.0f; dw[k][i] = 0.0f; }
  for (int l = warp; l < L; l += NW) {
    const float de = dal[l] * scale;
#pragma unroll
    for (int k = 0; k < KA; ++k) {
      const int a = lane * 4 + k * 128;
      if (a < A) {
        const float4 p = ld4(Pb + (int64_t)l * A + a);
        const float pv[4] = {p.x, p.y, p.z, p.w};
        float4 acc = *reinterpret_cast<float4*>(dPb + (int64_t)l * A + a);
        float o[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float u = sat_tanh<kExact>(pv[i] + qs[a + i]);
          const float dpu = de * ws[a + i] * (1.0f - u * u);
          o[i] = dpu;
          dq[k][i] += dpu;
          dw[k][i] = fmaf(de, u, dw[k][i]);
        }
        acc.x += o[0]; acc.y += o[1]; acc.z += o[2]; acc.w += o[3];
        *reinterpret_cast<float4*>(dPb + (int64_t)l * A + a) = acc;
        if (dP16 != nullptr && t == 0) st4(dP16 + ((int64_t)b * L + l) * A + a, acc);   // final value, operand dtype
      }
    }
  }
#pragma unroll
  for (int k = 0; k < KA; ++k) {
    const int a = lane * 4 + k * 128;
    if (a < A) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        red[warp * 2 * A + a + i] = dq[k][i];
        red[warp * 2 * A + A + a + i] = dw[k][i];
      }
    }
  }
  __syncthreads();
  for (int a = tid; a < A; a += ATT_THREADS) {
    float sq = 0.0f, sw = 0.0f;
#pragma unroll
    for (int w2 = 0; w2 < NW; ++w2) { sq += red[w2 * 2 * A + a]; sw += red[w2 * 2 * A + A + a]; }
    dy_b[a] = from_f<T>(sq);
    dwf_t[(int64_t)b * A + a] = sw;
  }
}

static inline size_t attention_bwd_smem(int L, int D, int A) {
  return sizeof(float) * (size_t)(D + ((L + 3) & ~3) + 2 * A + (ATT_THREADS / 32) * 2 * A + 40);
}


// =============================================================================================
// d_ann, attention part:  tmp[b,l,d] = sum_t alpha[b,t,l] * dZ[t,b,d] + dmean[img,d] * mean_scale   (fp32)
// The tensor-core GEMM dP * Wa then adds tmp as a coalesced residual and writes d_ann in the operand dtype
// (SURVEY.md appendix E: d_a += alpha (x) dz, deferred to one pass after the time loop).
// One CTA per (caption, 512-column chunk): dZ[:,b,chunk] and alpha[b,:,:] are staged in shared memory.
// =============================================================================================
constexpr int DANN_DC = 512;
template <typename T, typename TO>
__global__ void __launch_bounds__(256)
dann_alpha_kernel(const float* __restrict__ alphas, const T* __restrict__ dZ, const float* __restrict__ dmean,
                  TO* __restrict__ tmp, int B, int T_, int L, int D, int ncap, float mean_scale) {
  extern __shared__ __align__(16) float smem[];
  float* dzs = smem;                       // [T][DANN_DC]
  float* als = dzs + (size_t)T_ * DANN_DC; // [T][L]
  const int b = blockIdx.x, d0 = blockIdx.y * DANN_DC, tid = threadIdx.x;
  const int dc = min(DANN_DC, D - d0);
  for (int i = tid * 4; i < T_ * DANN_DC; i += 256 * 4) {
    const int t = i / DANN_DC, c = i - t * DANN_DC;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c < dc) v = ld4(dZ + ((int64_t)t * B + b) * D + d0 + c);
    *reinterpret_cast<float4*>(dzs + i) = v;
  }
  for (int i = tid; i < T_ * L; i += 256) als[i] = alphas[(int64_t)b * T_ * L + i];
  __syncthreads();
  const int cq = (tid & 127) * 4, lg = tid >> 7;
  if (cq >= dc) return;
  const float4 dm = ld4(dmean + (int64_t)(b / ncap) * D + d0 + cq);
  const float4 m4 = make_float4(dm.x * mean_scale, dm.y * mean_scale, dm.z * mean_scale, dm.w * mean_scale);
  for (int l0 = lg * 4; l0 < L; l0 += 8) {           // 4 consecutive rows per thread share every dz vector load
    float4 acc[4] = {m4, m4, m4, m4};
    for (int t = 0; t < T_; ++t) {
      const float4 z = *reinterpret_cast<const float4*>(dzs + (size_t)t * DANN_DC + cq);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float a = (l0 + u) < L ? als[t * L + l0 + u] : 0.0f;
        acc[u].x = fmaf(a, z.x, acc[u].x); acc[u].y = fmaf(a, z.y, acc[u].y);
        acc[u].z = fmaf(a, z.z, acc[u].z); acc[u].w = fmaf(a, z.w, acc[u].w);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if ((l0 + u) < L) st4(tmp + ((int64_t)b * L + l0 + u) * D + d0 + cq, acc[u]);
  }
}
