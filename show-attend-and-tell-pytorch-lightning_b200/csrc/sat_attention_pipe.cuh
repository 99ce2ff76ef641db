// K1 v3: fused attention step (forward) as a TMA-fed shared-memory pipeline, one CTA per caption row.
//
//   warp 8 (one elected lane) is the producer: it streams the caption's P tile (L x A) and then its
//   annotation tile (L x D) through a ring of NST 16-KB stages with 1-D TMA bulk copies
//   (cp.async.bulk + mbarrier complete_tx), running up to NST stages (96 KB) ahead of the consumers, so
//   the annotation rows are already in flight while the scores and the softmax are being computed.
//   warps 0-7 are consumers: scores from the P stages, softmax over L, alpha-weighted context from the
//   annotation stages (16-byte shared-memory loads), beta gate, stores.
//   Every byte of P / annotations is read from global memory exactly once per step; 2 CTAs per SM keep
//   ~190 KB of loads in flight per SM, which is what an HBM-bound kernel needs on B200.
//   Tried and dropped (measured slower on B200, see DESIGN.md §6): an 8-CTA cluster/DSMEM split of each caption, a
//   context phase on mma.sync + ldmatrix (also with a pre-swizzled annotation copy), one CTA per image for beam
//   groups, 16 consumer warps, and single-lane mbarrier polling.
#pragma once
#include <stdlib.h>
#include <algorithm>

#include <type_traits>

#include "sat_gemm_tc.cuh"
#include "sat_kernels.cuh"

__device__ __forceinline__ uint32_t sat_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void sat_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(sat_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void sat_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(sat_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void sat_mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(sat_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void sat_mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = sat_smem_u32(bar);
  uint32_t done;
  do {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, 0x989680;\n\t"   // suspend-time hint: sleep, don't spin
        "selp.b32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
  } while (!done);
}
// 1-D TMA bulk copy global -> shared (size a multiple of 16 B, both addresses 16 B aligned)
__device__ __forceinline__ void sat_bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(sat_smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(sat_smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void sat_named_bar(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

constexpr int ATTP_MAXCW = 16;                       // max consumer warps (template parameter CW of the kernels)
constexpr int ATTP_FWD_CW = 8;                       // forward: 8 consumer warps measured fastest (17.8 us vs 25.8 us at B=256 bf16)
constexpr int ATTP_BWD_CW = 8;                       // backward: with the dP accumulation deferred, 8 consumer warps (16-row stages:
                                                     // 2 rows per warp, 86 registers) beat 12 (25.1 vs 27.3 us at C2, 91 vs 97 us at
                                                     // C3 dims) and 16 (30 us, spills); two CTAs per SM either way
constexpr int ATTP_NST = 6;
constexpr int ATTP_STAGE_BYTES = 16384;
constexpr size_t SAT_ATT_GROUP_MIN_BYTES = 0;   // per-image annotation tile from which the grouped kernel is used (measured faster at every size tried)
// Attention columns: a lane owns columns lane*4 + 128*k, k < KA, so a kernel instantiated for KA serves attention_dim
// <= 128*KA.  KA = 2 (A <= 256) keeps q and w_f in registers (ATTP_REG_KA); KA = 4 / 8 (A <= 512 / 1024) read them from
// shared memory, where a register copy would cost 8*KA registers per lane.
constexpr int ATTP_REG_KA = 2;
constexpr int ATTP_MAXKA = 8;                        // attention_dim <= 1024 on the pipelined kernels
constexpr int ATTC_MAXA = 256;                       // the opt-in 2-CTA pair kernel: attention_dim <= 256
static inline int attp_ka(int A) { return A <= 256 ? 2 : (A <= 512 ? 4 : 8); }
constexpr size_t ATTP_SMEM_MAX = 227 * 1024;         // opt-in dynamic shared memory per block (sm_100)

struct AttPipeSmem {
  uint64_t full[ATTP_NST];
  uint64_t empty[ATTP_NST];
  float red_a[ATTP_MAXCW];
  float red_b[ATTP_MAXCW];
};

// KA > 2: scores of the rows l0 .. l0+3 of a P stage against one caption row, q and w_f read from shared memory (16-byte
// loads; A % 4 == 0).  Per lane the sum runs over the column slices in order and then over the 4 columns of a slice, as
// in the register path of the KA = 2 kernels.
template <typename T, bool kExact, int KA>
__device__ __forceinline__ void attp_scores4_smem(const T* Ps, int l0, int rows, int A, int lane, const float* q, const float* w,
                                                  float s4[4]) {
#pragma unroll 2
  for (int k = 0; k < KA; ++k) {
    const int a = lane * 4 + 128 * k;
    if (a < A) {
      float4 p[4];
#pragma unroll
      for (int u = 0; u < 4; ++u)
        p[u] = (l0 + u) < rows ? ld4(Ps + (size_t)(l0 + u) * A + a) : make_float4(0.f, 0.f, 0.f, 0.f);
      const float4 q4 = *reinterpret_cast<const float4*>(q + a);
      const float4 w4 = *reinterpret_cast<const float4*>(w + a);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        s4[u] = fmaf(w4.x, sat_tanh<kExact>(p[u].x + q4.x), s4[u]);
        s4[u] = fmaf(w4.y, sat_tanh<kExact>(p[u].y + q4.y), s4[u]);
        s4[u] = fmaf(w4.z, sat_tanh<kExact>(p[u].z + q4.z), s4[u]);
        s4[u] = fmaf(w4.w, sat_tanh<kExact>(p[u].w + q4.w), s4[u]);
      }
    }
  }
}

// KA > 2: first 4-row group of P stage i that warp `warp` scores.  A stage holds 16 KB / (A * sizeof(T)) rows, only 4 to 16
// at A > 256, so the groups are dealt round-robin over the warps across stages (all warps work while several stages are
// in flight) instead of every stage starting at warp 0.  Each row is still scored by one warp.
template <int CW>
__device__ __forceinline__ int attp_first_row(int warp, int i, int RCP) {
  const int ngr = (RCP + 3) / 4;
  return 4 * (((warp - (int)(((int64_t)i * ngr) % CW)) + CW) % CW);
}

// KA > 2, grouped kernels: the scores of every active caption row of the image for the rows of one P stage
template <typename T, bool kExact, int KA, int CW>
__device__ __forceinline__ void attp_group_stage_scores(const T* Ps, int i, int RCP, int r0, int rows, int A, int lane, int warp,
                                                        int ncap, unsigned act, const float* qs, const float* ws, float* e, int L4,
                                                        float scale) {
  for (int l0 = attp_first_row<CW>(warp, i, RCP); l0 < rows; l0 += CW * 4) {
    for (int g = 0; g < ncap; ++g) {
      if (!(act & (1u << g))) continue;
      float s4[4] = {0.f, 0.f, 0.f, 0.f};
      attp_scores4_smem<T, kExact, KA>(Ps, l0, rows, A, lane, qs + g * A, ws, s4);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int u = 0; u < 4; ++u) s4[u] += __shfl_xor_sync(0xffffffffu, s4[u], o);
      }
      if (lane < 4 && (l0 + lane) < rows) {
        const float sv = lane == 0 ? s4[0] : (lane == 1 ? s4[1] : (lane == 2 ? s4[2] : s4[3]));
        e[g * L4 + r0 + l0 + lane] = sv * scale;
      }
    }
  }
}

template <typename T, bool kExact, int CW, int KA = ATTP_REG_KA>
__global__ void __launch_bounds__(CW * 32 + 32)
attention_step_fwd_pipe_kernel(const T* __restrict__ ann, const T* __restrict__ P, const float* __restrict__ wf,
                               const float* __restrict__ hp, int64_t ldhp, const int32_t* __restrict__ lens, int t, int ncap,
                               int L, int D, int A, float scale, float* __restrict__ alpha, int64_t ld_alpha,
                               float* __restrict__ qsave, T* __restrict__ z, T* __restrict__ gz, T* __restrict__ beta,
                               int64_t ld_z, int lens_dyn) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  constexpr int VN = Vec16<T>::N;
  constexpr int ATTP_CWARPS = CW, ATTP_CONSUMERS = CW * 32, ATTP_THREADS = CW * 32 + 32;
  // Programmatic dependent launch: ann and P are never written inside a launch chain (P's GEMM is always followed by a
  // fully serialised launch), so the ring is primed while the predecessor kernel is still draining; everything that
  // reads the predecessor's output (or writes) sits behind SAT_PDL_WAIT() on the consumer side.  `lens` is constant in
  // the training chain (lens_dyn = 0) but is the beam-liveness array in decode, rewritten every step by
  // beam_update_kernel (lens_dyn = 1): there every thread waits for the predecessors BEFORE reading it.
  SAT_PDL_TRIGGER();
  if (lens_dyn) SAT_PDL_WAIT();
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = blockIdx.x;
  AttPipeSmem* hd = reinterpret_cast<AttPipeSmem*>(smem_raw);
  float* e = reinterpret_cast<float*>(smem_raw + sizeof(AttPipeSmem));   // [L4]
  const int L4 = (L + 3) & ~3;
  float* qs = e + L4;                   // [A]
  float* ws = qs + A;                   // [A]
  const int NV = D / VN;
  const int RG = NV >= ATTP_CONSUMERS ? 1 : ATTP_CONSUMERS / NV;
  float* red = ws + A;                  // [RG * D]
  // stage ring: offset computed with integer arithmetic from the (128-byte aligned) dynamic smem base so that the
  // compiler keeps the shared address space (LDS instead of generic LD)
  const uint32_t stage_off = (uint32_t)((sizeof(AttPipeSmem) + sizeof(float) * (size_t)(L4 + 2 * A + RG * D) + 127) & ~(size_t)127);
  uint8_t* stages = smem_raw + stage_off;

  const bool active = lens == nullptr || t < lens[b];
  float* alpha_b = alpha + (int64_t)b * ld_alpha;
  if (!active) {
    SAT_PDL_WAIT();
    for (int l = tid; l < L; l += ATTP_THREADS) alpha_b[l] = 0.0f;
    for (int d = tid; d < D; d += ATTP_THREADS) {
      z[(int64_t)b * ld_z + d] = from_f<T>(0.f);
      gz[(int64_t)b * ld_z + d] = from_f<T>(0.f);
      if (beta) beta[(int64_t)b * ld_z + d] = from_f<T>(0.f);
    }
    if (qsave) for (int a = tid; a < A; a += ATTP_THREADS) qsave[(int64_t)b * A + a] = 0.0f;
    return;
  }
  const int img = b / ncap;
  const int RCP = ATTP_STAGE_BYTES / (A * (int)sizeof(T));      // P rows per stage
  const int RCA = ATTP_STAGE_BYTES / (D * (int)sizeof(T));      // annotation rows per stage
  const int nP = (L + RCP - 1) / RCP, nA = (L + RCA - 1) / RCA;

  if (tid == 0) {
    for (int i = 0; i < ATTP_NST; ++i) {
      sat_mbar_init(&hd->full[i], 1);
      sat_mbar_init(&hd->empty[i], ATTP_CWARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();

  if (warp == ATTP_CWARPS) {
    // ===== producer =====
    if (lane == 0) {
      const T* Pb = P + (int64_t)img * L * A;
      const T* ab = ann + (int64_t)img * L * D;
      for (int i = 0; i < nP + nA; ++i) {
        const int st = i % ATTP_NST;
        const uint32_t ph = (uint32_t)(i / ATTP_NST) & 1u;
        sat_mbar_wait(&hd->empty[st], ph ^ 1u);
        const void* src;
        uint32_t bytes;
        if (i < nP) {
          const int r0 = i * RCP, rows = min(RCP, L - r0);
          src = Pb + (int64_t)r0 * A;
          bytes = (uint32_t)(rows * A * (int)sizeof(T));
        } else {
          const int r0 = (i - nP) * RCA, rows = min(RCA, L - r0);
          src = ab + (int64_t)r0 * D;
          bytes = (uint32_t)(rows * D * (int)sizeof(T));
        }
        sat_mbar_expect_tx(&hd->full[st], bytes);
        sat_bulk_g2s(stages + (size_t)st * ATTP_STAGE_BYTES, src, bytes, &hd->full[st]);
      }
    }
    return;
  }

  // ===== consumers (256 threads, named barrier 1) =====
  SAT_PDL_WAIT();
  const float* hp_b = hp + (int64_t)b * ldhp;
  for (int a = tid; a < A; a += ATTP_CONSUMERS) {
    const float q = hp_b[a];
    qs[a] = q;
    ws[a] = wf[a];
    if (qsave) qsave[(int64_t)b * A + a] = q;
  }
  sat_named_bar(1, ATTP_CONSUMERS);
  // beta_pre of the columns this thread finalises is fetched now, long before it is needed
  float bpre[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int d = tid + i * ATTP_CONSUMERS;
    bpre[i] = d < D ? hp_b[A + d] : 0.0f;
  }
  // lane-resident slices of q and w_f: lane owns attention columns lane*4 + 128*k .. +3  (A <= 128 * ATTP_REG_KA)
  float qreg[ATTP_REG_KA][4], wreg[ATTP_REG_KA][4];
  if constexpr (KA == ATTP_REG_KA) {
#pragma unroll
    for (int k = 0; k < ATTP_REG_KA; ++k) {
      const int a = lane * 4 + 128 * k;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        qreg[k][i] = a < A ? qs[a + i] : 0.0f;
        wreg[k][i] = a < A ? ws[a + i] : 0.0f;
      }
    }
  }
  int it = 0;   // running chunk index (same sequence as the producer)
  for (int i = 0; i < nP; ++i, ++it) {
    const int st = it % ATTP_NST;
    sat_mbar_wait(&hd->full[st], (uint32_t)(it / ATTP_NST) & 1u);
    const T* Ps = reinterpret_cast<const T*>(stages + (size_t)st * ATTP_STAGE_BYTES);
    const int r0 = i * RCP, rows = min(RCP, L - r0);
    const int lfirst = KA == ATTP_REG_KA ? warp * 4 : attp_first_row<CW>(warp, i, RCP);
    for (int l0 = lfirst; l0 < rows; l0 += ATTP_CWARPS * 4) {     // 4 rows in flight per warp: independent chains
      float s4[4] = {0.f, 0.f, 0.f, 0.f};
      if constexpr (KA != ATTP_REG_KA) {
        attp_scores4_smem<T, kExact, KA>(Ps, l0, rows, A, lane, qs, ws, s4);
      } else {
#pragma unroll
        for (int k = 0; k < ATTP_REG_KA; ++k) {
          const int a = lane * 4 + 128 * k;
          if (a < A) {
            float4 p[4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
              p[u] = (l0 + u) < rows ? ld4(Ps + (size_t)(l0 + u) * A + a) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              s4[u] = fmaf(wreg[k][0], sat_tanh<kExact>(p[u].x + qreg[k][0]), s4[u]);
              s4[u] = fmaf(wreg[k][1], sat_tanh<kExact>(p[u].y + qreg[k][1]), s4[u]);
              s4[u] = fmaf(wreg[k][2], sat_tanh<kExact>(p[u].z + qreg[k][2]), s4[u]);
              s4[u] = fmaf(wreg[k][3], sat_tanh<kExact>(p[u].w + qreg[k][3]), s4[u]);
            }
          }
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int u = 0; u < 4; ++u) s4[u] += __shfl_xor_sync(0xffffffffu, s4[u], o);
      }
      if (lane < 4 && (l0 + lane) < rows) {
        const float sv = lane == 0 ? s4[0] : (lane == 1 ? s4[1] : (lane == 2 ? s4[2] : s4[3]));
        e[r0 + l0 + lane] = sv * scale;
      }
    }
    __syncwarp();
    if (lane == 0) sat_mbar_arrive(&hd->empty[st]);
  }
  sat_named_bar(1, ATTP_CONSUMERS);
  // softmax over L (consumer-only reductions)
  float mx = -INFINITY;
  for (int l = tid; l < L; l += ATTP_CONSUMERS) mx = fmaxf(mx, e[l]);
  mx = warp_max(mx);
  if (lane == 0) hd->red_a[warp] = mx;
  sat_named_bar(1, ATTP_CONSUMERS);
  mx = hd->red_a[0];
#pragma unroll
  for (int w2 = 1; w2 < ATTP_CWARPS; ++w2) mx = fmaxf(mx, hd->red_a[w2]);
  float sum = 0.0f;
  for (int l = tid; l < L; l += ATTP_CONSUMERS) {
    const float p = sat_exp<kExact>(e[l] - mx);
    e[l] = p;
    sum += p;
  }
  sum = warp_sum(sum);
  if (lane == 0) hd->red_b[warp] = sum;
  sat_named_bar(1, ATTP_CONSUMERS);
  sum = 0.0f;
#pragma unroll
  for (int w2 = 0; w2 < ATTP_CWARPS; ++w2) sum += hd->red_b[w2];
  for (int l = tid; l < L; l += ATTP_CONSUMERS) {
    const float al = e[l] / sum;
    e[l] = al;
    alpha_b[l] = al;
  }
  sat_named_bar(1, ATTP_CONSUMERS);

  // context from the annotation stages: thread (rg, cv0) owns column vector cv0 and the rows
  // [rg*RPT, rg*RPT+RPT) of every stage (consecutive rows -> constant-stride, unrolled LDS.128)
  float acc[VN];
#pragma unroll
  for (int i = 0; i < VN; ++i) acc[i] = 0.0f;
  const int rg = RG == 1 ? 0 : tid / NV;
  const int cv0 = RG == 1 ? tid : tid - rg * NV;
  const int RPT = (RCA + RG - 1) / RG;
  const bool worker = rg < RG && cv0 < NV;
  for (int j = 0; j < nA; ++j, ++it) {
    const int st = it % ATTP_NST;
    sat_mbar_wait(&hd->full[st], (uint32_t)(it / ATTP_NST) & 1u);
    const T* As = reinterpret_cast<const T*>(stages + (size_t)st * ATTP_STAGE_BYTES);
    const int r0 = j * RCA, rows = min(RCA, L - r0);
    if (worker) {
      const int lb = rg * RPT, le = min(rows, lb + RPT);
      const T* ap = As + (size_t)lb * D + cv0 * VN;
      const float* ep = e + r0 + lb;
      int l = lb;
      for (; l + 4 <= le; l += 4, ap += 4 * (size_t)D, ep += 4) {
        float v[4][VN];
#pragma unroll
        for (int u = 0; u < 4; ++u) Vec16<T>::load_shared(ap + (size_t)u * D, v[u]);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float al = ep[u];
#pragma unroll
          for (int i2 = 0; i2 < VN; ++i2) acc[i2] = fmaf(al, v[u][i2], acc[i2]);
        }
      }
      for (; l < le; ++l, ap += D, ++ep) {
        float v[VN];
        Vec16<T>::load_shared(ap, v);
        const float al = ep[0];
#pragma unroll
        for (int i2 = 0; i2 < VN; ++i2) acc[i2] = fmaf(al, v[i2], acc[i2]);
      }
    }
    __syncwarp();
    if (lane == 0) sat_mbar_arrive(&hd->empty[st]);
  }
  if (rg < RG && cv0 < NV) {
#pragma unroll
    for (int i = 0; i < VN; ++i) red[rg * D + cv0 * VN + i] = acc[i];
  }
  sat_named_bar(1, ATTP_CONSUMERS);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int d = tid + i * ATTP_CONSUMERS;
    if (d < D) {
      float zs = 0.0f;
      for (int r = 0; r < RG; ++r) zs += red[r * D + d];
      const float bt = sat_sigmoid<kExact>(bpre[i]);
      z[(int64_t)b * ld_z + d] = from_f<T>(zs);
      gz[(int64_t)b * ld_z + d] = from_f<T>(bt * zs);
      if (beta) beta[(int64_t)b * ld_z + d] = from_f<T>(bt);
    }
  }
  for (int d = tid + 8 * ATTP_CONSUMERS; d < D; d += ATTP_CONSUMERS) {     // D > 8 * consumers: plain path
    float zs = 0.0f;
    for (int r = 0; r < RG; ++r) zs += red[r * D + d];
    const float bt = sat_sigmoid<kExact>(hp_b[A + d]);
    z[(int64_t)b * ld_z + d] = from_f<T>(zs);
    gz[(int64_t)b * ld_z + d] = from_f<T>(bt * zs);
    if (beta) beta[(int64_t)b * ld_z + d] = from_f<T>(bt);
  }
}

// =============================================================================================
// K1 grouped: the same pipeline with ONE CTA PER IMAGE serving up to G caption rows (the beams of beam search, or the
// ncap captions of an image): the image's P and annotation tiles are streamed once and every stage is used by all rows,
// instead of once per row through L2.  Per row the arithmetic and its summation order are those of
// attention_step_fwd_pipe_kernel, so both kernels give bit-identical alpha / z / gz.
//   smem: e[G][L4], q[G][A], w[A], ring; the cross-row-group reduction scratch red[G][RG*D] aliases the drained ring.
// =============================================================================================
template <typename T, bool kExact, int CW, int G, int KA = ATTP_REG_KA>
__global__ void __launch_bounds__(CW * 32 + 32, KA == ATTP_REG_KA ? 2 : 1)
attention_step_fwd_group_kernel(const T* __restrict__ ann, const T* __restrict__ P, const float* __restrict__ wf,
                                const float* __restrict__ hp, int64_t ldhp, const int32_t* __restrict__ lens, int t, int ncap,
                                int L, int D, int A, float scale, float* __restrict__ alpha, int64_t ld_alpha,
                                float* __restrict__ qsave, T* __restrict__ z, T* __restrict__ gz, T* __restrict__ beta,
                                int64_t ld_z, int lens_dyn) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  constexpr int VN = Vec16<T>::N;
  constexpr int ATTP_CWARPS = CW, ATTP_CONSUMERS = CW * 32;
  SAT_PDL_TRIGGER();      // ann, P are never written inside a launch chain: the ring is primed before SAT_PDL_WAIT()
  if (lens_dyn) SAT_PDL_WAIT();      // decode: lens (= alive) is rewritten every step by beam_update_kernel
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int img = blockIdx.x;
  const int row0 = img * ncap;          // first caption row of this image; rows row0 .. row0 + ncap - 1  (ncap <= G)
  AttPipeSmem* hd = reinterpret_cast<AttPipeSmem*>(smem_raw);
  const int L4 = (L + 3) & ~3;
  float* e = reinterpret_cast<float*>(smem_raw + sizeof(AttPipeSmem));   // [G][L4]
  float* qs = e + G * L4;               // [G][A]
  float* ws = qs + G * A;               // [A]
  float* part = ws + A;                 // [2][G][CW] softmax partials
  const int NV = D / VN;
  const int RG = NV >= ATTP_CONSUMERS ? 1 : ATTP_CONSUMERS / NV;
  const uint32_t stage_off =
      (uint32_t)((sizeof(AttPipeSmem) + sizeof(float) * (size_t)(G * L4 + G * A + A + 2 * G * CW) + 127) & ~(size_t)127);
  uint8_t* stages = smem_raw + stage_off;
  float* red = reinterpret_cast<float*>(stages);   // [G][RG * D], after the ring is drained

  unsigned act = 0;                     // bit g: row row0+g takes part in this step
  for (int g = 0; g < ncap; ++g)
    if (lens == nullptr || t < lens[row0 + g]) act |= 1u << g;
  const int RCP = ATTP_STAGE_BYTES / (A * (int)sizeof(T));
  const int RCA = ATTP_STAGE_BYTES / (D * (int)sizeof(T));
  const int nP = (L + RCP - 1) / RCP, nA = (L + RCA - 1) / RCA;

  if (act != 0 && tid == 0) {
    for (int i = 0; i < ATTP_NST; ++i) {
      sat_mbar_init(&hd->full[i], 1);
      sat_mbar_init(&hd->empty[i], ATTP_CWARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();

  if (warp == ATTP_CWARPS) {
    if (lane == 0 && act != 0) {        // ===== producer =====
      const T* Pb = P + (int64_t)img * L * A;
      const T* ab = ann + (int64_t)img * L * D;
      for (int i = 0; i < nP + nA; ++i) {
        const int st = i % ATTP_NST;
        const uint32_t ph = (uint32_t)(i / ATTP_NST) & 1u;
        sat_mbar_wait(&hd->empty[st], ph ^ 1u);
        const void* src;
        uint32_t bytes;
        if (i < nP) {
          const int r0 = i * RCP, rows = min(RCP, L - r0);
          src = Pb + (int64_t)r0 * A;
          bytes = (uint32_t)(rows * A * (int)sizeof(T));
        } else {
          const int r0 = (i - nP) * RCA, rows = min(RCA, L - r0);
          src = ab + (int64_t)r0 * D;
          bytes = (uint32_t)(rows * D * (int)sizeof(T));
        }
        sat_mbar_expect_tx(&hd->full[st], bytes);
        sat_bulk_g2s(stages + (size_t)st * ATTP_STAGE_BYTES, src, bytes, &hd->full[st]);
      }
    }
    return;
  }

  // ===== consumers =====
  SAT_PDL_WAIT();
  // rows that sit this step out get zero outputs (as the per-row kernel writes them)
  for (int g = 0; g < ncap; ++g) {
    if (act & (1u << g)) continue;
    const int64_t r = row0 + g;
    for (int l = tid; l < L; l += ATTP_CONSUMERS) alpha[r * ld_alpha + l] = 0.0f;
    for (int d = tid; d < D; d += ATTP_CONSUMERS) {
      z[r * ld_z + d] = from_f<T>(0.f);
      gz[r * ld_z + d] = from_f<T>(0.f);
      if (beta) beta[r * ld_z + d] = from_f<T>(0.f);
    }
    if (qsave) for (int a = tid; a < A; a += ATTP_CONSUMERS) qsave[r * A + a] = 0.0f;
  }
  if (act == 0) return;
  for (int i = tid; i < ncap * A; i += ATTP_CONSUMERS) {
    const int g = i / A, a = i - g * A;
    const float q = hp[(int64_t)(row0 + g) * ldhp + a];
    qs[g * A + a] = q;
    if (qsave && (act & (1u << g))) qsave[(int64_t)(row0 + g) * A + a] = q;
  }
  for (int a = tid; a < A; a += ATTP_CONSUMERS) ws[a] = wf[a];
  sat_named_bar(1, ATTP_CONSUMERS);

  float wreg[ATTP_REG_KA][4];
  if constexpr (KA == ATTP_REG_KA) {
#pragma unroll
    for (int k = 0; k < ATTP_REG_KA; ++k) {
      const int a = lane * 4 + 128 * k;
#pragma unroll
      for (int i = 0; i < 4; ++i) wreg[k][i] = a < A ? ws[a + i] : 0.0f;
    }
  }
  int it = 0;
  for (int i = 0; i < nP; ++i, ++it) {
    const int st = it % ATTP_NST;
    sat_mbar_wait(&hd->full[st], (uint32_t)(it / ATTP_NST) & 1u);
    const T* Ps = reinterpret_cast<const T*>(stages + (size_t)st * ATTP_STAGE_BYTES);
    const int r0 = i * RCP, rows = min(RCP, L - r0);
    if constexpr (KA != ATTP_REG_KA)
      attp_group_stage_scores<T, kExact, KA, CW>(Ps, i, RCP, r0, rows, A, lane, warp, ncap, act, qs, ws, e, L4, scale);
    else
    for (int l0 = warp * 4; l0 < rows; l0 += ATTP_CWARPS * 4) {
      float4 p[ATTP_REG_KA][4];
#pragma unroll
      for (int k = 0; k < ATTP_REG_KA; ++k) {
        const int a = lane * 4 + 128 * k;
#pragma unroll
        for (int u = 0; u < 4; ++u)
          p[k][u] = (a < A && (l0 + u) < rows) ? ld4(Ps + (size_t)(l0 + u) * A + a) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      for (int g = 0; g < ncap; ++g) {
        if (!(act & (1u << g))) continue;
        float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int k = 0; k < ATTP_REG_KA; ++k) {
          const int a = lane * 4 + 128 * k;
          if (a < A) {
            const float4 q4 = *reinterpret_cast<const float4*>(qs + g * A + a);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              s4[u] = fmaf(wreg[k][0], sat_tanh<kExact>(p[k][u].x + q4.x), s4[u]);
              s4[u] = fmaf(wreg[k][1], sat_tanh<kExact>(p[k][u].y + q4.y), s4[u]);
              s4[u] = fmaf(wreg[k][2], sat_tanh<kExact>(p[k][u].z + q4.z), s4[u]);
              s4[u] = fmaf(wreg[k][3], sat_tanh<kExact>(p[k][u].w + q4.w), s4[u]);
            }
          }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
          for (int u = 0; u < 4; ++u) s4[u] += __shfl_xor_sync(0xffffffffu, s4[u], o);
        }
        if (lane < 4 && (l0 + lane) < rows) {
          const float sv = lane == 0 ? s4[0] : (lane == 1 ? s4[1] : (lane == 2 ? s4[2] : s4[3]));
          e[g * L4 + r0 + l0 + lane] = sv * scale;
        }
      }
    }
    __syncwarp();
    if (lane == 0) sat_mbar_arrive(&hd->empty[st]);
  }
  sat_named_bar(1, ATTP_CONSUMERS);
  // softmax over L for every row (same partial / combine order as the per-row kernel)
  float* pmax = part;
  float* psum = part + G * CW;
  for (int g = 0; g < ncap; ++g) {
    float mx = -INFINITY;
    if (act & (1u << g))
      for (int l = tid; l < L; l += ATTP_CONSUMERS) mx = fmaxf(mx, e[g * L4 + l]);
    mx = warp_max(mx);
    if (lane == 0) pmax[g * CW + warp] = mx;
  }
  sat_named_bar(1, ATTP_CONSUMERS);
  for (int g = 0; g < ncap; ++g) {
    if (!(act & (1u << g))) continue;
    float mx = pmax[g * CW];
#pragma unroll
    for (int w2 = 1; w2 < ATTP_CWARPS; ++w2) mx = fmaxf(mx, pmax[g * CW + w2]);
    float sum = 0.0f;
    for (int l = tid; l < L; l += ATTP_CONSUMERS) {
      const float pe = sat_exp<kExact>(e[g * L4 + l] - mx);
      e[g * L4 + l] = pe;
      sum += pe;
    }
    sum = warp_sum(sum);
    if (lane == 0) psum[g * CW + warp] = sum;
  }
  sat_named_bar(1, ATTP_CONSUMERS);
  for (int g = 0; g < G; ++g) {
    float* eg = e + g * L4;
    if (g >= ncap || !(act & (1u << g))) {
      for (int l = tid; l < L; l += ATTP_CONSUMERS) eg[l] = 0.0f;     // contributes nothing to the context loop
      continue;
    }
    float sum = 0.0f;
#pragma unroll
    for (int w2 = 0; w2 < ATTP_CWARPS; ++w2) sum += psum[g * CW + w2];
    float* alpha_r = alpha + (int64_t)(row0 + g) * ld_alpha;
    for (int l = tid; l < L; l += ATTP_CONSUMERS) {
      const float al = eg[l] / sum;
      eg[l] = al;
      alpha_r[l] = al;
    }
  }
  sat_named_bar(1, ATTP_CONSUMERS);

  // context: every annotation vector is loaded once and feeds all rows
  float acc[G][VN];
#pragma unroll
  for (int g = 0; g < G; ++g)
#pragma unroll
    for (int i = 0; i < VN; ++i) acc[g][i] = 0.0f;
  const int rg = RG == 1 ? 0 : tid / NV;
  const int cv0 = RG == 1 ? tid : tid - rg * NV;
  const int RPT = (RCA + RG - 1) / RG;
  const bool worker = rg < RG && cv0 < NV;
  for (int j = 0; j < nA; ++j, ++it) {
    const int st = it % ATTP_NST;
    sat_mbar_wait(&hd->full[st], (uint32_t)(it / ATTP_NST) & 1u);
    const T* As = reinterpret_cast<const T*>(stages + (size_t)st * ATTP_STAGE_BYTES);
    const int r0 = j * RCA, rows = min(RCA, L - r0);
    if (worker) {
      const int lb = rg * RPT, le = min(rows, lb + RPT);
      const T* ap = As + (size_t)lb * D + cv0 * VN;
      const float* ep = e + r0 + lb;
      int l = lb;
      for (; l + 2 <= le; l += 2, ap += 2 * (size_t)D, ep += 2) {
        float v[2][VN];
#pragma unroll
        for (int u = 0; u < 2; ++u) Vec16<T>::load_shared(ap + (size_t)u * D, v[u]);
        float al[G][2];                 // straight-line code: rows g >= ncap carry alpha = 0 (zeroed above)
#pragma unroll
        for (int g = 0; g < G; ++g) {
          al[g][0] = ep[g * L4];
          al[g][1] = ep[g * L4 + 1];
        }
#pragma unroll
        for (int u = 0; u < 2; ++u) {
#pragma unroll
          for (int g = 0; g < G; ++g) {
#pragma unroll
            for (int i2 = 0; i2 < VN; ++i2) acc[g][i2] = fmaf(al[g][u], v[u][i2], acc[g][i2]);
          }
        }
      }
      for (; l < le; ++l, ap += D, ++ep) {
        float v[VN];
        Vec16<T>::load_shared(ap, v);
#pragma unroll
        for (int g = 0; g < G; ++g) {
          const float al = ep[g * L4];
#pragma unroll
          for (int i2 = 0; i2 < VN; ++i2) acc[g][i2] = fmaf(al, v[i2], acc[g][i2]);
        }
      }
    }
    __syncwarp();
    if (lane == 0) sat_mbar_arrive(&hd->empty[st]);
  }
  sat_named_bar(1, ATTP_CONSUMERS);     // the ring is drained: red[] may overwrite it
  if (worker) {
#pragma unroll
    for (int g = 0; g < G; ++g) {
      if (g < ncap) {
#pragma unroll
        for (int i = 0; i < VN; ++i) red[((size_t)g * RG + rg) * D + cv0 * VN + i] = acc[g][i];
      }
    }
  }
  sat_named_bar(1, ATTP_CONSUMERS);
  for (int g = 0; g < ncap; ++g) {
    if (!(act & (1u << g))) continue;
    const int64_t r = row0 + g;
    const float* hp_r = hp + r * ldhp;
    for (int d = tid; d < D; d += ATTP_CONSUMERS) {
      float zs = 0.0f;
      for (int q = 0; q < RG; ++q) zs += red[((size_t)g * RG + q) * D + d];
      const float bt = sat_sigmoid<kExact>(hp_r[A + d]);
      z[r * ld_z + d] = from_f<T>(zs);
      gz[r * ld_z + d] = from_f<T>(bt * zs);
      if (beta) beta[r * ld_z + d] = from_f<T>(bt);
    }
  }
}

template <int G>
static inline size_t attention_fwd_group_smem(int L, int A) {
  return ((sizeof(AttPipeSmem) + sizeof(float) * (size_t)(G * ((L + 3) & ~3) + G * A + A + 2 * G * ATTP_FWD_CW) + 127) & ~(size_t)127) +
         128 + (size_t)ATTP_NST * ATTP_STAGE_BYTES;
}

// =============================================================================================
// K1 grouped, tensor-core context (bf16 operands): as attention_step_fwd_group_kernel, but the context
//   z[g, :] = sum_l alpha[g, l] * ann[l, :]          (g = the <= 8 caption rows of the image)
// is an [8 x L] x [L x D] product, so it runs on mma.sync.m16n8k16 (rows 8..15 of the A tile are zero): the annotation
// tile is streamed as 128-row x 64-column boxes by 2-D TMA with the 128-byte swizzle (conflict-free ldmatrix.trans),
// column block by column block; warp w owns the 8 columns w*8.. of a box and keeps alpha (rounded to bf16) as A
// fragments in registers for the whole kernel.  Scores and softmax are the fp32 code of the grouped kernel.
// Needs bf16, L <= 256, D % 64 == 0, ncap <= 8.  Box rows past the image's L rows are multiplied by alpha = 0.
// =============================================================================================
constexpr int ATTG_BOX_ROWS = 128, ATTG_BOX_COLS = 64, ATTG_MAXKS = 16;     // 16 k-steps of 16 rows: L <= 256

__device__ __forceinline__ uint32_t sat_pack_bf16x2(float lo, float hi) {
  const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&v);
}

template <bool kExact, int CW, int KA = ATTP_REG_KA>
__global__ void __launch_bounds__(CW * 32 + 32, 2)
attention_step_fwd_group_tc_kernel(const __grid_constant__ CUtensorMap tm_ann, const bf16* __restrict__ P,
                                   const float* __restrict__ wf, const float* __restrict__ hp, int64_t ldhp,
                                   const int32_t* __restrict__ lens, int t, int ncap, int L, int D, int A, float scale,
                                   float* __restrict__ alpha, int64_t ld_alpha, float* __restrict__ qsave, bf16* __restrict__ z,
                                   bf16* __restrict__ gz, bf16* __restrict__ beta, int64_t ld_z, int lens_dyn) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  typedef bf16 T;
  constexpr int G = 8;
  constexpr int ATTP_CWARPS = CW, ATTP_CONSUMERS = CW * 32;
  static_assert(CW == 8, "one consumer warp per 8-column slice of a 64-column box");
  SAT_PDL_TRIGGER();      // ann, P are never written inside a launch chain: the ring is primed before SAT_PDL_WAIT()
  if (lens_dyn) SAT_PDL_WAIT();      // decode: lens (= alive) is rewritten every step by beam_update_kernel
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int img = blockIdx.x;
  const int row0 = img * ncap;
  AttPipeSmem* hd = reinterpret_cast<AttPipeSmem*>(smem_raw);
  const int L4 = (L + 3) & ~3;
  float* e = reinterpret_cast<float*>(smem_raw + sizeof(AttPipeSmem));   // [G][L4]
  float* qs = e + G * L4;               // [G][A]
  float* ws = qs + G * A;               // [A]
  float* part = ws + A;                 // [2][G][CW]
  const uint32_t base_u32 = sat_smem_u32(smem_raw);
  const uint32_t hdr = (uint32_t)(sizeof(AttPipeSmem) + sizeof(float) * (size_t)(G * L4 + G * A + A + 2 * G * CW));
  const uint32_t stage_off = ((base_u32 + hdr + 1023u) & ~1023u) - base_u32;       // 1024-byte aligned: 128B swizzle atom
  uint8_t* stages = smem_raw + stage_off;

  unsigned act = 0;
  for (int g = 0; g < ncap; ++g)
    if (lens == nullptr || t < lens[row0 + g]) act |= 1u << g;
  const int RCP = ATTP_STAGE_BYTES / (A * (int)sizeof(T));
  const int nP = (L + RCP - 1) / RCP;
  const int nRB = (L + ATTG_BOX_ROWS - 1) / ATTG_BOX_ROWS, nCB = D / ATTG_BOX_COLS;

  if (act != 0 && tid == 0) {
    for (int i = 0; i < ATTP_NST; ++i) {
      sat_mbar_init(&hd->full[i], 1);
      sat_mbar_init(&hd->empty[i], ATTP_CWARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();

  if (warp == ATTP_CWARPS) {
    if (lane == 0 && act != 0) {        // ===== producer: P chunks (1-D bulk), then annotation boxes (2-D, swizzled) =====
      const T* Pb = P + (int64_t)img * L * A;
      const int nbox = nCB * nRB;
      for (int i = 0; i < nP + nbox; ++i) {
        const int st = i % ATTP_NST;
        const uint32_t ph = (uint32_t)(i / ATTP_NST) & 1u;
        sat_mbar_wait(&hd->empty[st], ph ^ 1u);
        if (i < nP) {
          const int r0 = i * RCP, rows = min(RCP, L - r0);
          const uint32_t bytes = (uint32_t)(rows * A * (int)sizeof(T));
          sat_mbar_expect_tx(&hd->full[st], bytes);
          sat_bulk_g2s(stages + (size_t)st * ATTP_STAGE_BYTES, Pb + (int64_t)r0 * A, bytes, &hd->full[st]);
        } else {
          const int bi = i - nP, cb = bi / nRB, rb = bi - cb * nRB;
          sat_mbar_expect_tx(&hd->full[st], (uint32_t)(ATTG_BOX_ROWS * ATTG_BOX_COLS * sizeof(T)));
          tc::tma_load_2d(&tm_ann, &hd->full[st], stages + (size_t)st * ATTP_STAGE_BYTES, cb * ATTG_BOX_COLS,
                          img * L + rb * ATTG_BOX_ROWS);
        }
      }
    }
    return;
  }

  // ===== consumers =====
  SAT_PDL_WAIT();
  for (int g = 0; g < ncap; ++g) {
    if (act & (1u << g)) continue;
    const int64_t r = row0 + g;
    for (int l = tid; l < L; l += ATTP_CONSUMERS) alpha[r * ld_alpha + l] = 0.0f;
    for (int d = tid; d < D; d += ATTP_CONSUMERS) {
      z[r * ld_z + d] = from_f<T>(0.f);
      gz[r * ld_z + d] = from_f<T>(0.f);
      if (beta) beta[r * ld_z + d] = from_f<T>(0.f);
    }
    if (qsave) for (int a = tid; a < A; a += ATTP_CONSUMERS) qsave[r * A + a] = 0.0f;
  }
  if (act == 0) return;
  for (int i = tid; i < ncap * A; i += ATTP_CONSUMERS) {
    const int g = i / A, a = i - g * A;
    const float q = hp[(int64_t)(row0 + g) * ldhp + a];
    qs[g * A + a] = q;
    if (qsave && (act & (1u << g))) qsave[(int64_t)(row0 + g) * A + a] = q;
  }
  for (int a = tid; a < A; a += ATTP_CONSUMERS) ws[a] = wf[a];
  sat_named_bar(1, ATTP_CONSUMERS);

  float wreg[ATTP_REG_KA][4];
  if constexpr (KA == ATTP_REG_KA) {
#pragma unroll
    for (int k = 0; k < ATTP_REG_KA; ++k) {
      const int a = lane * 4 + 128 * k;
#pragma unroll
      for (int i = 0; i < 4; ++i) wreg[k][i] = a < A ? ws[a + i] : 0.0f;
    }
  }
  int it = 0;
  for (int i = 0; i < nP; ++i, ++it) {
    const int st = it % ATTP_NST;
    sat_mbar_wait(&hd->full[st], (uint32_t)(it / ATTP_NST) & 1u);
    const T* Ps = reinterpret_cast<const T*>(stages + (size_t)st * ATTP_STAGE_BYTES);
    const int r0 = i * RCP, rows = min(RCP, L - r0);
    if constexpr (KA != ATTP_REG_KA)
      attp_group_stage_scores<T, kExact, KA, CW>(Ps, i, RCP, r0, rows, A, lane, warp, ncap, act, qs, ws, e, L4, scale);
    else
    for (int l0 = warp * 4; l0 < rows; l0 += ATTP_CWARPS * 4) {
      float4 p[ATTP_REG_KA][4];
#pragma unroll
      for (int k = 0; k < ATTP_REG_KA; ++k) {
        const int a = lane * 4 + 128 * k;
#pragma unroll
        for (int u = 0; u < 4; ++u)
          p[k][u] = (a < A && (l0 + u) < rows) ? ld4(Ps + (size_t)(l0 + u) * A + a) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      for (int g = 0; g < ncap; ++g) {
        if (!(act & (1u << g))) continue;
        float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int k = 0; k < ATTP_REG_KA; ++k) {
          const int a = lane * 4 + 128 * k;
          if (a < A) {
            const float4 q4 = *reinterpret_cast<const float4*>(qs + g * A + a);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              s4[u] = fmaf(wreg[k][0], sat_tanh<kExact>(p[k][u].x + q4.x), s4[u]);
              s4[u] = fmaf(wreg[k][1], sat_tanh<kExact>(p[k][u].y + q4.y), s4[u]);
              s4[u] = fmaf(wreg[k][2], sat_tanh<kExact>(p[k][u].z + q4.z), s4[u]);
              s4[u] = fmaf(wreg[k][3], sat_tanh<kExact>(p[k][u].w + q4.w), s4[u]);
            }
          }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
          for (int u = 0; u < 4; ++u) s4[u] += __shfl_xor_sync(0xffffffffu, s4[u], o);
        }
        if (lane < 4 && (l0 + lane) < rows) {
          const float sv = lane == 0 ? s4[0] : (lane == 1 ? s4[1] : (lane == 2 ? s4[2] : s4[3]));
          e[g * L4 + r0 + l0 + lane] = sv * scale;
        }
      }
    }
    __syncwarp();
    if (lane == 0) sat_mbar_arrive(&hd->empty[st]);
  }
  sat_named_bar(1, ATTP_CONSUMERS);
  float* pmax = part;
  float* psum = part + G * CW;
  for (int g = 0; g < ncap; ++g) {
    float mx = -INFINITY;
    if (act & (1u << g))
      for (int l = tid; l < L; l += ATTP_CONSUMERS) mx = fmaxf(mx, e[g * L4 + l]);
    mx = warp_max(mx);
    if (lane == 0) pmax[g * CW + warp] = mx;
  }
  sat_named_bar(1, ATTP_CONSUMERS);
  for (int g = 0; g < ncap; ++g) {
    if (!(act & (1u << g))) continue;
    float mx = pmax[g * CW];
#pragma unroll
    for (int w2 = 1; w2 < ATTP_CWARPS; ++w2) mx = fmaxf(mx, pmax[g * CW + w2]);
    float sum = 0.0f;
    for (int l = tid; l < L; l += ATTP_CONSUMERS) {
      const float pe = sat_exp<kExact>(e[g * L4 + l] - mx);
      e[g * L4 + l] = pe;
      sum += pe;
    }
    sum = warp_sum(sum);
    if (lane == 0) psum[g * CW + warp] = sum;
  }
  sat_named_bar(1, ATTP_CONSUMERS);
  for (int g = 0; g < G; ++g) {
    float* eg = e + g * L4;
    if (g >= ncap || !(act & (1u << g))) {
      for (int l = tid; l < L; l += ATTP_CONSUMERS) eg[l] = 0.0f;
      continue;
    }
    float sum = 0.0f;
#pragma unroll
    for (int w2 = 0; w2 < ATTP_CWARPS; ++w2) sum += psum[g * CW + w2];
    float* alpha_r = alpha + (int64_t)(row0 + g) * ld_alpha;
    for (int l = tid; l < L; l += ATTP_CONSUMERS) {
      const float al = eg[l] / sum;
      eg[l] = al;
      alpha_r[l] = al;
    }
  }
  sat_named_bar(1, ATTP_CONSUMERS);

  // A fragments of alpha (row g = lane / 4 of the m16 tile, rows 8..15 zero), one pair of registers per 16-row k-step
  const int g = lane >> 2, kk = (lane & 3) * 2;
  uint32_t afr[ATTG_MAXKS][2];
#pragma unroll
  for (int ks = 0; ks < ATTG_MAXKS; ++ks) {
    const int l = ks * 16 + kk;
    const float* eg = e + g * L4;
    afr[ks][0] = sat_pack_bf16x2(l < L ? eg[l] : 0.0f, l + 1 < L ? eg[l + 1] : 0.0f);
    afr[ks][1] = sat_pack_bf16x2(l + 8 < L ? eg[l + 8] : 0.0f, l + 9 < L ? eg[l + 9] : 0.0f);
  }
  const bool row_on = g < ncap && (act & (1u << g));
  const int64_t r = row0 + g;
  const uint32_t stages_u32 = base_u32 + stage_off;
  const int mrow = (lane >> 3) * 8 + (lane & 7);        // ldmatrix.x4: lane -> row of the 32-row slab it addresses
  for (int cb = 0; cb < nCB; ++cb) {
    const int d = cb * ATTG_BOX_COLS + warp * 8 + kk;   // this thread's two output columns d, d + 1
    float2 hv = make_float2(0.f, 0.f);
    if (row_on) hv = *reinterpret_cast<const float2*>(hp + r * ldhp + A + d);     // consumed after the boxes below
    float c0 = 0.f, c1 = 0.f, c2 = 0.f, c3 = 0.f;
#pragma unroll
    for (int rb = 0; rb < ATTG_MAXKS / 8; ++rb) {
      if (rb < nRB) {
        const int st = it % ATTP_NST;
        sat_mbar_wait(&hd->full[st], (uint32_t)(it / ATTP_NST) & 1u);
        const uint32_t sb = stages_u32 + (uint32_t)st * ATTP_STAGE_BYTES;
#pragma unroll
        for (int k2 = 0; k2 < 4; ++k2) {
          const int rr = k2 * 32 + mrow;
          const uint32_t addr = sb + (uint32_t)rr * 128u + (uint32_t)((warp ^ (rr & 7)) << 4);
          uint32_t b0, b1, b2, b3;
          asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
                       : "=r"(b0), "=r"(b1), "=r"(b2), "=r"(b3)
                       : "r"(addr));
          asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                       : "+f"(c0), "+f"(c1), "+f"(c2), "+f"(c3)
                       : "r"(afr[rb * 8 + 2 * k2][0]), "r"(0u), "r"(afr[rb * 8 + 2 * k2][1]), "r"(0u), "r"(b0), "r"(b1));
          asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                       : "+f"(c0), "+f"(c1), "+f"(c2), "+f"(c3)
                       : "r"(afr[rb * 8 + 2 * k2 + 1][0]), "r"(0u), "r"(afr[rb * 8 + 2 * k2 + 1][1]), "r"(0u), "r"(b2), "r"(b3));
        }
        __syncwarp();
        if (lane == 0) sat_mbar_arrive(&hd->empty[st]);
        ++it;
      }
    }
    if (row_on) {
      const float bt0 = sat_sigmoid<kExact>(hv.x), bt1 = sat_sigmoid<kExact>(hv.y);
      *reinterpret_cast<uint32_t*>(z + r * ld_z + d) = sat_pack_bf16x2(c0, c1);
      *reinterpret_cast<uint32_t*>(gz + r * ld_z + d) = sat_pack_bf16x2(bt0 * c0, bt1 * c1);
      if (beta) *reinterpret_cast<uint32_t*>(beta + r * ld_z + d) = sat_pack_bf16x2(bt0, bt1);
    }
  }
}

// =============================================================================================
// K1 grouped, tensor-core context, ROW-STREAMED (bf16, D a multiple of 256 up to 2048): the 2-D box kernel above fetches
// 128 bytes per annotation row per box, which costs DRAM page locality (3.6 TB/s at D=2048).  Here the tile is streamed
// as whole rows (1-D bulk copies, one per row, issued by 8-16 lanes of the producer warp) into stages whose rows are
// padded by 16 bytes, which makes ldmatrix.trans conflict-free without a swizzle.  The product is transposed:
//   zT[d, g] = sum_l ann[l, d] * alpha[g, l]      mma.sync.m16n8k8: M = 16 columns d, N = 8 caption rows, K = 8 locations
// so no MMA row is wasted; warp w owns columns [w*D/8, (w+1)*D/8) (MT 16-column tiles, 4 accumulator registers each).
// =============================================================================================
template <bool kExact, int CW, int MT, int KA = ATTP_REG_KA>
__global__ void __launch_bounds__(CW * 32 + 32, 2)
attention_step_fwd_group_tcr_kernel(const bf16* __restrict__ ann, const bf16* __restrict__ P, const float* __restrict__ wf,
                                    const float* __restrict__ hp, int64_t ldhp, const int32_t* __restrict__ lens, int t, int ncap,
                                    int L, int D, int A, float scale, float* __restrict__ alpha, int64_t ld_alpha,
                                    float* __restrict__ qsave, bf16* __restrict__ z, bf16* __restrict__ gz, bf16* __restrict__ beta,
                                    int64_t ld_z, int lens_dyn, int rows_per_stage, int nst, int stage_bytes) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  typedef bf16 T;
  constexpr int G = 8;
  constexpr int ATTP_CWARPS = CW, ATTP_CONSUMERS = CW * 32;
  static_assert(CW == 8, "column ranges are split over 8 consumer warps");
  SAT_PDL_TRIGGER();      // ann, P are never written inside a launch chain: the ring is primed before SAT_PDL_WAIT()
  if (lens_dyn) SAT_PDL_WAIT();      // decode: lens (= alive) is rewritten every step by beam_update_kernel
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int img = blockIdx.x;
  const int row0 = img * ncap;
  AttPipeSmem* hd = reinterpret_cast<AttPipeSmem*>(smem_raw);
  const int L4 = (L + 3) & ~3;
  float* e = reinterpret_cast<float*>(smem_raw + sizeof(AttPipeSmem));   // [G][L4]
  float* qs = e + G * L4;               // [G][A]
  float* ws = qs + G * A;               // [A]
  float* part = ws + A;                 // [2][G][CW]
  const uint32_t stage_off = (uint32_t)((sizeof(AttPipeSmem) + sizeof(float) * (size_t)(G * L4 + G * A + A + 2 * G * CW) + 127) & ~(size_t)127);
  uint8_t* stages = smem_raw + stage_off;
  float* red = reinterpret_cast<float*>(stages);   // [G][D] fp32, after the ring is drained
  const int rowb = D * (int)sizeof(T) + 16;        // padded row pitch in a stage

  unsigned act = 0;
  for (int g = 0; g < ncap; ++g)
    if (lens == nullptr || t < lens[row0 + g]) act |= 1u << g;
  const int RCP = stage_bytes / (A * (int)sizeof(T));
  const int nP = (L + RCP - 1) / RCP;
  const int RS = rows_per_stage, nA = (L + RS - 1) / RS;

  if (act != 0 && tid == 0) {
    for (int i = 0; i < nst; ++i) {
      sat_mbar_init(&hd->full[i], 1);
      sat_mbar_init(&hd->empty[i], ATTP_CWARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();

  if (warp == ATTP_CWARPS) {
    if (act != 0) {                     // ===== producer warp: lane 0 arms the barrier, lanes 0..RS-1 copy one row each =====
      const T* Pb = P + (int64_t)img * L * A;
      const T* ab = ann + (int64_t)img * L * D;
      for (int i = 0; i < nP + nA; ++i) {
        const int st = i % nst;
        const uint32_t ph = (uint32_t)(i / nst) & 1u;
        uint8_t* dst = stages + (size_t)st * stage_bytes;
        if (lane == 0) sat_mbar_wait(&hd->empty[st], ph ^ 1u);
        __syncwarp();
        if (i < nP) {
          if (lane == 0) {
            const int r0 = i * RCP, rows = min(RCP, L - r0);
            const uint32_t bytes = (uint32_t)(rows * A * (int)sizeof(T));
            sat_mbar_expect_tx(&hd->full[st], bytes);
            sat_bulk_g2s(dst, Pb + (int64_t)r0 * A, bytes, &hd->full[st]);
          }
        } else {
          // the last stage is filled up to a whole 8-row k-step with copies of the last row (finite data; its alpha is 0)
          const int r0 = (i - nP) * RS, rows = min(RS, (min(RS, L - r0) + 7) & ~7);
          if (lane == 0) sat_mbar_expect_tx(&hd->full[st], (uint32_t)(rows * D * (int)sizeof(T)));
          __syncwarp();
          if (lane < rows)
            sat_bulk_g2s(dst + (size_t)lane * rowb, ab + (int64_t)min(r0 + lane, L - 1) * D, (uint32_t)(D * sizeof(T)), &hd->full[st]);
        }
      }
    }
    return;
  }

  // ===== consumers =====
  SAT_PDL_WAIT();
  for (int g = 0; g < ncap; ++g) {
    if (act & (1u << g)) continue;
    const int64_t r = row0 + g;
    for (int l = tid; l < L; l += ATTP_CONSUMERS) alpha[r * ld_alpha + l] = 0.0f;
    for (int d = tid; d < D; d += ATTP_CONSUMERS) {
      z[r * ld_z + d] = from_f<T>(0.f);
      gz[r * ld_z + d] = from_f<T>(0.f);
      if (beta) beta[r * ld_z + d] = from_f<T>(0.f);
    }
    if (qsave) for (int a = tid; a < A; a += ATTP_CONSUMERS) qsave[r * A + a] = 0.0f;
  }
  if (act == 0) return;
  for (int i = tid; i < ncap * A; i += ATTP_CONSUMERS) {
    const int g = i / A, a = i - g * A;
    const float q = hp[(int64_t)(row0 + g) * ldhp + a];
    qs[g * A + a] = q;
    if (qsave && (act & (1u << g))) qsave[(int64_t)(row0 + g) * A + a] = q;
  }
  for (int a = tid; a < A; a += ATTP_CONSUMERS) ws[a] = wf[a];
  sat_named_bar(1, ATTP_CONSUMERS);

  float wreg[ATTP_REG_KA][4];
  if constexpr (KA == ATTP_REG_KA) {
#pragma unroll
    for (int k = 0; k < ATTP_REG_KA; ++k) {
      const int a = lane * 4 + 128 * k;
#pragma unroll
      for (int i = 0; i < 4; ++i) wreg[k][i] = a < A ? ws[a + i] : 0.0f;
    }
  }
  int it = 0;
  for (int i = 0; i < nP; ++i, ++it) {
    const int st = it % nst;
    sat_mbar_wait(&hd->full[st], (uint32_t)(it / nst) & 1u);
    const T* Ps = reinterpret_cast<const T*>(stages + (size_t)st * stage_bytes);
    const int r0 = i * RCP, rows = min(RCP, L - r0);
    if constexpr (KA != ATTP_REG_KA)
      attp_group_stage_scores<T, kExact, KA, CW>(Ps, i, RCP, r0, rows, A, lane, warp, ncap, act, qs, ws, e, L4, scale);
    else
    for (int l0 = warp * 4; l0 < rows; l0 += ATTP_CWARPS * 4) {
      float4 p[ATTP_REG_KA][4];
#pragma unroll
      for (int k = 0; k < ATTP_REG_KA; ++k) {
        const int a = lane * 4 + 128 * k;
#pragma unroll
        for (int u = 0; u < 4; ++u)
          p[k][u] = (a < A && (l0 + u) < rows) ? ld4(Ps + (size_t)(l0 + u) * A + a) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      for (int g = 0; g < ncap; ++g) {
        if (!(act & (1u << g))) continue;
        float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int k = 0; k < ATTP_REG_KA; ++k) {
          const int a = lane * 4 + 128 * k;
          if (a < A) {
            const float4 q4 = *reinterpret_cast<const float4*>(qs + g * A + a);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              s4[u] = fmaf(wreg[k][0], sat_tanh<kExact>(p[k][u].x + q4.x), s4[u]);
              s4[u] = fmaf(wreg[k][1], sat_tanh<kExact>(p[k][u].y + q4.y), s4[u]);
              s4[u] = fmaf(wreg[k][2], sat_tanh<kExact>(p[k][u].z + q4.z), s4[u]);
              s4[u] = fmaf(wreg[k][3], sat_tanh<kExact>(p[k][u].w + q4.w), s4[u]);
            }
          }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
          for (int u = 0; u < 4; ++u) s4[u] += __shfl_xor_sync(0xffffffffu, s4[u], o);
        }
        if (lane < 4 && (l0 + lane) < rows) {
          const float sv = lane == 0 ? s4[0] : (lane == 1 ? s4[1] : (lane == 2 ? s4[2] : s4[3]));
          e[g * L4 + r0 + l0 + lane] = sv * scale;
        }
      }
    }
    __syncwarp();
    if (lane == 0) sat_mbar_arrive(&hd->empty[st]);
  }
  sat_named_bar(1, ATTP_CONSUMERS);
  float* pmax = part;
  float* psum = part + G * CW;
  for (int g = 0; g < ncap; ++g) {
    float mx = -INFINITY;
    if (act & (1u << g))
      for (int l = tid; l < L; l += ATTP_CONSUMERS) mx = fmaxf(mx, e[g * L4 + l]);
    mx = warp_max(mx);
    if (lane == 0) pmax[g * CW + warp] = mx;
  }
  sat_named_bar(1, ATTP_CONSUMERS);
  for (int g = 0; g < ncap; ++g) {
    if (!(act & (1u << g))) continue;
    float mx = pmax[g * CW];
#pragma unroll
    for (int w2 = 1; w2 < ATTP_CWARPS; ++w2) mx = fmaxf(mx, pmax[g * CW + w2]);
    float sum = 0.0f;
    for (int l = tid; l < L; l += ATTP_CONSUMERS) {
      const float pe = sat_exp<kExact>(e[g * L4 + l] - mx);
      e[g * L4 + l] = pe;
      sum += pe;
    }
    sum = warp_sum(sum);
    if (lane == 0) psum[g * CW + warp] = sum;
  }
  sat_named_bar(1, ATTP_CONSUMERS);
  for (int g = 0; g < G; ++g) {
    float* eg = e + g * L4;
    if (g >= ncap || !(act & (1u << g))) {
      for (int l = tid; l < L4; l += ATTP_CONSUMERS) eg[l] = 0.0f;
      continue;
    }
    float sum = 0.0f;
#pragma unroll
    for (int w2 = 0; w2 < ATTP_CWARPS; ++w2) sum += psum[g * CW + w2];
    float* alpha_r = alpha + (int64_t)(row0 + g) * ld_alpha;
    for (int l = tid; l < L4; l += ATTP_CONSUMERS) {
      const float al = l < L ? eg[l] / sum : 0.0f;
      eg[l] = al;
      if (l < L) alpha_r[l] = al;
    }
  }
  sat_named_bar(1, ATTP_CONSUMERS);

  // context: zT[d, g] accumulators, MT tiles of 16 columns per warp
  float acc[MT][4];
#pragma unroll
  for (int m = 0; m < MT; ++m)
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[m][i] = 0.0f;
  const int gq = lane >> 2, kk = (lane & 3) * 2;                 // B fragment: caption row gq, locations kk, kk + 1 of a k-step
  const float* eg = e + gq * L4;
  const int dw0 = warp * (MT * 16);                              // first column of this warp
  // ldmatrix.x4.trans lane addressing: lanes 8j..8j+7 give the 8 location rows of matrix j = columns dw0 + 32 p + 8 j ..
  const uint32_t lane_off = (uint32_t)((lane & 7) * rowb + (dw0 + (lane >> 3) * 8) * (int)sizeof(T));
  const uint32_t stages_u32 = sat_smem_u32(stages);
  for (int j = 0; j < nA; ++j, ++it) {
    const int st = it % nst;
    sat_mbar_wait(&hd->full[st], (uint32_t)(it / nst) & 1u);
    const uint32_t sb = stages_u32 + (uint32_t)st * (uint32_t)stage_bytes + lane_off;
    const int r0 = j * RS, rows = min(RS, L - r0);
    for (int k0 = 0; k0 < rows; k0 += 8) {                       // rows past L inside a k-step: alpha = 0 below, the stage holds
      const int l = r0 + k0 + kk;                                // stale but finite data there
      const uint32_t bfr = sat_pack_bf16x2(l < L ? eg[l] : 0.0f, l + 1 < L ? eg[l + 1] : 0.0f);
      const uint32_t kb = sb + (uint32_t)(k0 * rowb);
#pragma unroll
      for (int p = 0; p < MT / 2; ++p) {
        uint32_t a0, a1, a2, a3;
        asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
                     : "=r"(a0), "=r"(a1), "=r"(a2), "=r"(a3)
                     : "r"(kb + (uint32_t)(p * 32 * (int)sizeof(T))));
        asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5}, {%6}, {%0, %1, %2, %3};"
                     : "+f"(acc[2 * p][0]), "+f"(acc[2 * p][1]), "+f"(acc[2 * p][2]), "+f"(acc[2 * p][3])
                     : "r"(a0), "r"(a1), "r"(bfr));
        asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5}, {%6}, {%0, %1, %2, %3};"
                     : "+f"(acc[2 * p + 1][0]), "+f"(acc[2 * p + 1][1]), "+f"(acc[2 * p + 1][2]), "+f"(acc[2 * p + 1][3])
                     : "r"(a2), "r"(a3), "r"(bfr));
      }
    }
    __syncwarp();
    if (lane == 0) sat_mbar_arrive(&hd->empty[st]);
  }
  sat_named_bar(1, ATTP_CONSUMERS);     // the ring is drained: red[] may overwrite it
  // C fragment: acc[m][0..1] = column dw0 + 16 m + lane/4, caption rows kk, kk+1;  acc[m][2..3] = column + 8
#pragma unroll
  for (int m = 0; m < MT; ++m) {
    const int d = dw0 + m * 16 + gq;
    red[(size_t)kk * D + d] = acc[m][0];
    red[(size_t)(kk + 1) * D + d] = acc[m][1];
    red[(size_t)kk * D + d + 8] = acc[m][2];
    red[(size_t)(kk + 1) * D + d + 8] = acc[m][3];
  }
  sat_named_bar(1, ATTP_CONSUMERS);
  for (int g = 0; g < ncap; ++g) {
    if (!(act & (1u << g))) continue;
    const int64_t r = row0 + g;
    const float* hp_r = hp + r * ldhp + A;
    for (int d = tid * 2; d < D; d += ATTP_CONSUMERS * 2) {
      const float2 zs = *reinterpret_cast<const float2*>(red + (size_t)g * D + d);
      const float2 hv = *reinterpret_cast<const float2*>(hp_r + d);
      const float bt0 = sat_sigmoid<kExact>(hv.x), bt1 = sat_sigmoid<kExact>(hv.y);
      *reinterpret_cast<uint32_t*>(z + r * ld_z + d) = sat_pack_bf16x2(zs.x, zs.y);
      *reinterpret_cast<uint32_t*>(gz + r * ld_z + d) = sat_pack_bf16x2(bt0 * zs.x, bt1 * zs.y);
      if (beta) *reinterpret_cast<uint32_t*>(beta + r * ld_z + d) = sat_pack_bf16x2(bt0, bt1);
    }
  }
}

// =============================================================================================
// K1 pair: one caption row per 2-CTA CLUSTER (bf16, one row per image, D <= 512).  At BASELINE configs[1] the per-row kernel
// above is a single wave of 256 CTAs whose run time is the critical path of ONE row (prologue -> scores -> softmax -> context
// -> gate): latency-, not bandwidth-bound.  Here two CTAs share a row and halve that path:
//   * scores: CTA r streams the P rows of its half of the locations and computes their scores; every score is written to
//     both CTAs' shared memory (local store + st.shared::cluster to the peer), completion is signalled with a remote
//     mbarrier arrive, so each CTA ends up with all L scores and runs the (cheap) softmax redundantly;
//   * context: CTA r owns the column half [r*D/2, (r+1)*D/2) of z for ALL locations: the annotation tile is streamed as
//     32-row x D/2-column boxes by 2-D TMA; no reduction across the pair is needed, each CTA gates and stores its half.
// 4 CTAs (36 warps) per SM instead of 2 (18): twice the warps hide the same latencies.  Same arithmetic as the per-row
// kernel up to the order of the softmax / context sums.
// =============================================================================================
constexpr int ATTC_CW = 8;          // consumer warps
constexpr int ATTC_NST = 3;         // 3 x 16 KB ring -> ~50 KB per CTA, 4 CTAs per SM
constexpr int ATTC_BOX_ROWS = 32;

struct AttPairSmem {
  uint64_t full[ATTC_NST];
  uint64_t empty[ATTC_NST];
  uint64_t xbar;                    // the peer's scores have landed (remote arrive, one per consumer warp of the peer)
  float red_a[ATTC_CW];
  float red_b[ATTC_CW];
};

__device__ __forceinline__ uint32_t sat_cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t sat_mapa(uint32_t smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void sat_st_cluster_f32(uint32_t addr, float v) {
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ void sat_cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void sat_cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ void sat_mbar_arrive_remote(uint32_t remote_bar) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote_bar) : "memory");
}
__device__ __forceinline__ void sat_mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = sat_smem_u32(bar);
  uint32_t done;
  do {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2, 0x989680;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
  } while (!done);
}

template <bool kExact, int CW>
__global__ void __launch_bounds__(CW * 32 + 32, 4)
attention_step_fwd_pair_kernel(const __grid_constant__ CUtensorMap tm_ann, const bf16* __restrict__ P, const float* __restrict__ wf,
                               const float* __restrict__ hp, int64_t ldhp, const int32_t* __restrict__ lens, int t, int ncap, int L,
                               int D, int A, float scale, float* __restrict__ alpha, int64_t ld_alpha, float* __restrict__ qsave,
                               bf16* __restrict__ z, bf16* __restrict__ gz, bf16* __restrict__ beta, int64_t ld_z, int lens_dyn) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  typedef bf16 T;
  constexpr int CONSUMERS = CW * 32, THREADS = CW * 32 + 32;
  SAT_PDL_TRIGGER();
  if (lens_dyn) SAT_PDL_WAIT();         // decode: lens (= alive) is rewritten every step by beam_update_kernel
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t rank = sat_cluster_ctarank();
  const int b = blockIdx.x >> 1;
  const int Dh = D >> 1, d0 = (int)rank * Dh;
  AttPairSmem* hd = reinterpret_cast<AttPairSmem*>(smem_raw);
  const int L4 = (L + 3) & ~3;
  float* e = reinterpret_cast<float*>(smem_raw + sizeof(AttPairSmem));      // [L4] all scores, then alpha
  const uint32_t stage_off = (uint32_t)((sizeof(AttPairSmem) + sizeof(float) * (size_t)L4 + 127) & ~(size_t)127);
  uint8_t* stages = smem_raw + stage_off;
  float* red = reinterpret_cast<float*>(stages);                             // [CW][Dh], after the ring is drained

  const bool active = lens == nullptr || t < lens[b];                        // the same value in both CTAs of the pair
  if (!active) {                        // no cluster traffic at all for a finished row: both CTAs just write their zeros
    SAT_PDL_WAIT();
    float* alpha_b = alpha + (int64_t)b * ld_alpha;
    if (rank == 0) {
      for (int l = tid; l < L; l += THREADS) alpha_b[l] = 0.0f;
      if (qsave) for (int a = tid; a < A; a += THREADS) qsave[(int64_t)b * A + a] = 0.0f;
    }
    for (int d = tid; d < Dh; d += THREADS) {
      z[(int64_t)b * ld_z + d0 + d] = from_f<T>(0.f);
      gz[(int64_t)b * ld_z + d0 + d] = from_f<T>(0.f);
      if (beta) beta[(int64_t)b * ld_z + d0 + d] = from_f<T>(0.f);
    }
    return;
  }
  const int img = b / ncap;
  const int Ls = min(L, (((L + 1) >> 1) + 3) & ~3);      // locations [0, Ls) belong to CTA 0, [Ls, L) to CTA 1
  const int l0 = rank ? Ls : 0, l1 = rank ? L : Ls, nl = l1 - l0;
  const int RCP = ATTP_STAGE_BYTES / (A * (int)sizeof(T));                   // P rows per stage
  const int nP = (nl + RCP - 1) / RCP, nA = (L + ATTC_BOX_ROWS - 1) / ATTC_BOX_ROWS;
  const uint32_t box_bytes = (uint32_t)(ATTC_BOX_ROWS * Dh * (int)sizeof(T));

  if (tid == 0) {
    for (int i = 0; i < ATTC_NST; ++i) {
      sat_mbar_init(&hd->full[i], 1);
      sat_mbar_init(&hd->empty[i], CW);
    }
    sat_mbar_init(&hd->xbar, CW);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();
  sat_cluster_arrive();                 // both CTAs are running and their barriers exist before any remote access (waited below)

  if (warp == CW) {
    // ===== producer: the CTA's P rows (1-D bulk copies), then the annotation boxes of its column half (2-D TMA) =====
    if (lane == 0) {
      const T* Pb = P + ((int64_t)img * L + l0) * A;
      for (int i = 0; i < nP + nA; ++i) {
        const int st = i % ATTC_NST;
        const uint32_t ph = (uint32_t)(i / ATTC_NST) & 1u;
        sat_mbar_wait(&hd->empty[st], ph ^ 1u);
        uint8_t* dst = stages + (size_t)st * ATTP_STAGE_BYTES;
        if (i < nP) {
          const int r0 = i * RCP, rows = min(RCP, nl - r0);
          const uint32_t bytes = (uint32_t)(rows * A * (int)sizeof(T));
          sat_mbar_expect_tx(&hd->full[st], bytes);
          sat_bulk_g2s(dst, Pb + (int64_t)r0 * A, bytes, &hd->full[st]);
        } else {
          sat_mbar_expect_tx(&hd->full[st], box_bytes);
          tc::tma_load_2d(&tm_ann, &hd->full[st], dst, d0, img * L + (i - nP) * ATTC_BOX_ROWS);
        }
      }
    }
    __syncwarp();
    sat_cluster_wait();                 // pairs with the arrive above (every thread arrives and waits exactly once)
    return;
  }

  // ===== consumers =====
  SAT_PDL_WAIT();
  const float* hp_b = hp + (int64_t)b * ldhp;
  float qreg[ATTP_REG_KA][4], wreg[ATTP_REG_KA][4];
#pragma unroll
  for (int k = 0; k < ATTP_REG_KA; ++k) {
    const int a = lane * 4 + 128 * k;
    float4 q4 = make_float4(0.f, 0.f, 0.f, 0.f), w4 = q4;
    if (a < A) {
      q4 = *reinterpret_cast<const float4*>(hp_b + a);
      w4 = *reinterpret_cast<const float4*>(wf + a);
      if (qsave && rank == 0 && warp == 0) *reinterpret_cast<float4*>(qsave + (int64_t)b * A + a) = q4;
    }
    qreg[k][0] = q4.x; qreg[k][1] = q4.y; qreg[k][2] = q4.z; qreg[k][3] = q4.w;
    wreg[k][0] = w4.x; wreg[k][1] = w4.y; wreg[k][2] = w4.z; wreg[k][3] = w4.w;
  }
  const float bpre = tid < Dh ? hp_b[A + d0 + tid] : 0.0f;                  // beta_pre of the column this thread finalises
  sat_cluster_wait();                                                       // the peer's shared memory and barriers are live
  const uint32_t e_remote = sat_mapa(sat_smem_u32(e), rank ^ 1u);
  int it = 0;
  for (int i = 0; i < nP; ++i, ++it) {
    const int st = it % ATTC_NST;
    sat_mbar_wait(&hd->full[st], (uint32_t)(it / ATTC_NST) & 1u);
    const T* Ps = reinterpret_cast<const T*>(stages + (size_t)st * ATTP_STAGE_BYTES);
    const int r0 = i * RCP, rows = min(RCP, nl - r0);
    for (int lr = warp * 4; lr < rows; lr += CW * 4) {
      float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int k = 0; k < ATTP_REG_KA; ++k) {
        const int a = lane * 4 + 128 * k;
        if (a < A) {
          float4 p[4];
#pragma unroll
          for (int u = 0; u < 4; ++u)
            p[u] = (lr + u) < rows ? ld4(Ps + (size_t)(lr + u) * A + a) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            s4[u] = fmaf(wreg[k][0], sat_tanh<kExact>(p[u].x + qreg[k][0]), s4[u]);
            s4[u] = fmaf(wreg[k][1], sat_tanh<kExact>(p[u].y + qreg[k][1]), s4[u]);
            s4[u] = fmaf(wreg[k][2], sat_tanh<kExact>(p[u].z + qreg[k][2]), s4[u]);
            s4[u] = fmaf(wreg[k][3], sat_tanh<kExact>(p[u].w + qreg[k][3]), s4[u]);
          }
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int u = 0; u < 4; ++u) s4[u] += __shfl_xor_sync(0xffffffffu, s4[u], o);
      }
      if (lane < 4 && (lr + lane) < rows) {
        const float sv = (lane == 0 ? s4[0] : (lane == 1 ? s4[1] : (lane == 2 ? s4[2] : s4[3]))) * scale;
        const int l = l0 + r0 + lr + lane;
        e[l] = sv;
        sat_st_cluster_f32(e_remote + (uint32_t)l * 4u, sv);
      }
    }
    __syncwarp();
    if (lane == 0) sat_mbar_arrive(&hd->empty[st]);
  }
  // this warp's scores are in both CTAs: tell the peer (release at cluster scope orders the remote stores before the arrive)
  __syncwarp();
  if (lane == 0) sat_mbar_arrive_remote(sat_mapa(sat_smem_u32(&hd->xbar), rank ^ 1u));
  sat_named_bar(1, CONSUMERS);                                              // own half complete (local stores)
  sat_mbar_wait_cluster(&hd->xbar, 0);                                      // the peer's half has landed
  // softmax over all L locations (both CTAs compute it; it is ~L exps)
  float mx = -INFINITY;
  for (int l = tid; l < L; l += CONSUMERS) mx = fmaxf(mx, e[l]);
  mx = warp_max(mx);
  if (lane == 0) hd->red_a[warp] = mx;
  sat_named_bar(1, CONSUMERS);
  mx = hd->red_a[0];
#pragma unroll
  for (int w2 = 1; w2 < CW; ++w2) mx = fmaxf(mx, hd->red_a[w2]);
  float sum = 0.0f;
  for (int l = tid; l < L; l += CONSUMERS) {
    const float pe = sat_exp<kExact>(e[l] - mx);
    e[l] = pe;
    sum += pe;
  }
  sum = warp_sum(sum);
  if (lane == 0) hd->red_b[warp] = sum;
  sat_named_bar(1, CONSUMERS);
  sum = 0.0f;
#pragma unroll
  for (int w2 = 0; w2 < CW; ++w2) sum += hd->red_b[w2];
  float* alpha_b = alpha + (int64_t)b * ld_alpha;
  for (int l = tid; l < L; l += CONSUMERS) {
    const float al = e[l] / sum;
    e[l] = al;
    if (l >= l0 && l < l1) alpha_b[l] = al;                                 // each CTA stores the weights of its own locations
  }
  sat_named_bar(1, CONSUMERS);

  // context for the columns [d0, d0 + Dh): a warp takes rows w, w + CW, .. of every 32-row box, a lane one 16-byte vector
  constexpr int VN = 8;
  const int NV = Dh / VN;                                                   // <= 32
  float acc[VN];
#pragma unroll
  for (int i = 0; i < VN; ++i) acc[i] = 0.0f;
  const bool worker = lane < NV;
  for (int j = 0; j < nA; ++j, ++it) {
    const int st = it % ATTC_NST;
    sat_mbar_wait(&hd->full[st], (uint32_t)(it / ATTC_NST) & 1u);
    const T* As = reinterpret_cast<const T*>(stages + (size_t)st * ATTP_STAGE_BYTES);
    const int r0 = j * ATTC_BOX_ROWS, rows = min(ATTC_BOX_ROWS, L - r0);
    if (worker) {
      float v[ATTC_BOX_ROWS / CW][VN];
      float al[ATTC_BOX_ROWS / CW];
#pragma unroll
      for (int u = 0; u < ATTC_BOX_ROWS / CW; ++u) {
        const int rr = warp + u * CW;                                       // rows past the image's last location carry weight 0
        al[u] = rr < rows ? e[r0 + rr] : 0.0f;
        Vec16<T>::load_shared(As + (size_t)rr * Dh + lane * VN, v[u]);
      }
#pragma unroll
      for (int u = 0; u < ATTC_BOX_ROWS / CW; ++u) {
#pragma unroll
        for (int i2 = 0; i2 < VN; ++i2) acc[i2] = fmaf(al[u], v[u][i2], acc[i2]);
      }
    }
    __syncwarp();
    if (lane == 0) sat_mbar_arrive(&hd->empty[st]);
  }
  sat_named_bar(1, CONSUMERS);          // the ring is drained: red[] may overwrite it
  if (worker) {
#pragma unroll
    for (int i = 0; i < VN; ++i) red[warp * Dh + lane * VN + i] = acc[i];
  }
  sat_named_bar(1, CONSUMERS);
  if (tid < Dh) {
    float zs = 0.0f;
#pragma unroll
    for (int w2 = 0; w2 < CW; ++w2) zs += red[w2 * Dh + tid];
    const float bt = sat_sigmoid<kExact>(bpre);
    z[(int64_t)b * ld_z + d0 + tid] = from_f<T>(zs);
    gz[(int64_t)b * ld_z + d0 + tid] = from_f<T>(bt * zs);
    if (beta) beta[(int64_t)b * ld_z + d0 + tid] = from_f<T>(bt);
  }
}

static inline size_t attention_fwd_pair_smem(int L) {
  return ((sizeof(AttPairSmem) + sizeof(float) * (size_t)((L + 3) & ~3) + 127) & ~(size_t)127) + 128 + (size_t)ATTC_NST * ATTP_STAGE_BYTES;
}

// stage geometry of the row-streamed kernel: 8 or 16 padded rows per stage, as many stages as fit ~97 KB (<= ATTP_NST)
struct AttTcrGeom { int rows, nst, stage_bytes; size_t smem; };
static inline AttTcrGeom attention_fwd_group_tcr_geom(int L, int D, int A) {
  AttTcrGeom g;
  const int rowb = D * 2 + 16;
  g.rows = rowb * 16 <= 20 * 1024 ? 16 : 8;
  g.stage_bytes = (g.rows * rowb + 127) & ~127;
  g.nst = (int)std::min<size_t>(ATTP_NST, (size_t)(97 * 1024) / g.stage_bytes);
  g.smem = ((sizeof(AttPipeSmem) + sizeof(float) * (size_t)(8 * ((L + 3) & ~3) + 8 * A + A + 2 * 8 * ATTP_FWD_CW) + 127) & ~(size_t)127) + 128 +
           (size_t)g.nst * g.stage_bytes;
  return g;
}

static inline size_t attention_fwd_group_tc_smem(int L, int A) {
  return sizeof(AttPipeSmem) + sizeof(float) * (size_t)(8 * ((L + 3) & ~3) + 8 * A + A + 2 * 8 * ATTP_FWD_CW) + 1024 +
         (size_t)ATTP_NST * ATTP_STAGE_BYTES;
}

static inline size_t attention_fwd_pipe_smem(int L, int D, int A, int vn) {
  constexpr int ATTP_CONSUMERS = ATTP_FWD_CW * 32;
  const int NV = D / vn;
  const int RG = NV >= ATTP_CONSUMERS ? 1 : ATTP_CONSUMERS / NV;
  return sizeof(AttPipeSmem) + sizeof(float) * (size_t)(((L + 3) & ~3) + 2 * A + (size_t)RG * D) + 128 +
         (size_t)ATTP_NST * ATTP_STAGE_BYTES;
}

// The pipelined kernel needs: one row of P and of the annotations to fit a stage, at most 256 16-byte column vectors per
// annotation row (D <= 2048 bf16 / 1024 fp32) and attention_dim <= 1024 (a multiple of 4 above 256: 16-byte shared-memory
// loads of q and w_f); other shapes use the plain kernel.
template <typename T>
static inline bool attention_pipe_ok(int L, int D, int A) {
  static int mode = -2;                       // SAT_ATT_MODE=0 forces the plain single-pass kernel (A/B timing)
  if (mode == -2) {
    const char* e = getenv("SAT_ATT_MODE");
    mode = e ? atoi(e) : -1;
  }
  if (mode == 0) return false;
  (void)L;
  return D * (int)sizeof(T) <= ATTP_STAGE_BYTES && A <= 128 * ATTP_MAXKA && (A <= 128 * ATTP_REG_KA || A % 4 == 0) &&
         D / Vec16<T>::N <= ATTP_FWD_CW * 32;
}

// launch helper shared by the training and decode drivers
template <typename T, bool kExact>
static int launch_attention_fwd(const T* ann, const T* P, const float* wf, const float* hp, int64_t ldhp, const int32_t* lens,
                                int t, int rows, int ncap, int L, int D, int A, float scale, float* alpha, int64_t ld_alpha,
                                float* qsave, T* z, T* gz, T* beta, int64_t ld_z, cudaStream_t st, int lens_dyn = 0) {
  if (!attention_pipe_ok<T>(L, D, A)) {
    const size_t sm1 = attention_fwd_smem(L, D, A, Vec16<T>::N);
    auto k1 = attention_step_fwd_kernel<T, kExact>;
    if (sm1 > 48 * 1024) SAT_CUDA(cudaFuncSetAttribute(k1, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm1));
    k1<<<rows, ATT_THREADS, sm1, st>>>(ann, P, wf, hp, ldhp, lens, t, ncap, L, D, A, scale, alpha, ld_alpha, qsave, z, gz, beta, ld_z);
    SAT_COUNT_LAUNCH();
    SAT_LAUNCH_OK();
    return 0;
  }
  // one row per image, bf16, small grids: a 2-CTA cluster per row halves the row's critical path (SAT_ATT_PAIR=0/1 forces
  // the choice; by default up to 3 rows per SM, where the per-row kernel is a single latency-bound wave)
  if constexpr (std::is_same<T, bf16>::value && !kExact) {
    // Measured on B200 at BASELINE configs[1] (B = 256): 18.1-18.6 us (ncu) / 20.3 us (in situ) against 18.6 / 20.1 us for the
    // per-row kernel -- halving the row's critical path changes nothing, the launch is bounded by DRAM streaming plus fixed
    // launch / fill / drain costs, not by the path of one row.  Kept as an opt-in variant (SAT_ATT_PAIR=1), off by default.
    static const int pair_mode = getenv("SAT_ATT_PAIR") ? atoi(getenv("SAT_ATT_PAIR")) : 0;
    const int Dh = D / 2;
    const bool pair_fit = ncap == 1 && D % 16 == 0 && Dh <= 256 && Dh * 2 * ATTC_BOX_ROWS <= ATTP_STAGE_BYTES && A <= ATTC_MAXA && A % 4 == 0 &&
                          L >= 8 && ldhp % 4 == 0 && (reinterpret_cast<uintptr_t>(hp) & 15) == 0;
    if (pair_fit && (pair_mode == 1 || (pair_mode != 0 && rows <= 3 * 148))) {
      static thread_local CUtensorMap tmp;
      static thread_local const void* tmp_ptr = nullptr;
      static thread_local int64_t tmp_rows = 0, tmp_d = 0;
      static thread_local int tmp_dev = -1;
      const int64_t n_rows = (int64_t)rows * L;            // ncap == 1: one image per row
      int dev_now = 0;
      SAT_CUDA(cudaGetDevice(&dev_now));
      if (tmp_ptr != (const void*)ann || tmp_rows != n_rows || tmp_d != D || tmp_dev != dev_now) {
        SAT_TRY(tc::make_map_plain(&tmp, ann, n_rows, D, D, Dh, ATTC_BOX_ROWS));
        tmp_ptr = ann; tmp_rows = n_rows; tmp_d = D; tmp_dev = dev_now;
      }
      auto kern = attention_step_fwd_pair_kernel<kExact, ATTC_CW>;
      const size_t smem = attention_fwd_pair_smem(L);
      SAT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      SAT_CUDA(sat_launch_cluster_pdl(kern, dim3(2 * rows), dim3(ATTC_CW * 32 + 32), smem, 2, st, tmp, P, wf, hp, ldhp, lens, t, ncap, L, D, A,
                                      scale, alpha, ld_alpha, qsave, z, gz, beta, ld_z, lens_dyn));
      SAT_COUNT_LAUNCH();
      return 0;
    }
  }
  // several caption rows per image (beams / captions): one CTA per image streams the tiles once for all of them when
  // the per-image tile is large enough for the shared stream to pay (SAT_ATT_GROUP=0/1 forces the choice)
  static const int group_mode = getenv("SAT_ATT_GROUP") ? atoi(getenv("SAT_ATT_GROUP")) : -1;
  const bool group_fit = ncap >= 2 && ncap <= 8 && rows % ncap == 0 && L <= 512 &&
                         (size_t)ncap * (((D / Vec16<T>::N) >= ATTP_FWD_CW * 32 ? 1 : (ATTP_FWD_CW * 32) / (D / Vec16<T>::N)) * (size_t)D) *
                                 sizeof(float) <= (size_t)ATTP_NST * ATTP_STAGE_BYTES;
  const bool group = group_fit && (group_mode == 1 || (group_mode != 0 && (size_t)L * D * sizeof(T) >= SAT_ATT_GROUP_MIN_BYTES));
  // kernel instantiation for the attention_dim: KA column slices of 128 per lane
  const int ka = attp_ka(A);
  auto by_ka = [ka](auto k2, auto k4, auto k8) { return ka == 2 ? k2 : (ka == 4 ? k4 : k8); };
  if constexpr (std::is_same<T, bf16>::value && !kExact) {
    static const int group_tc_mode = getenv("SAT_ATT_GROUP_TC") ? atoi(getenv("SAT_ATT_GROUP_TC")) : 1;
    if (group && group_tc_mode != 0 && D % ATTG_BOX_COLS == 0 && ld_z % 2 == 0 && ldhp % 2 == 0 && A % 2 == 0) {
      // a variant whose shared memory (it grows with A) exceeds the per-block limit falls back to the next one
      static const int tcr_mode = getenv("SAT_ATT_GROUP_TCR") ? atoi(getenv("SAT_ATT_GROUP_TCR")) : 1;
      // measured: row-streamed 89 vs box 100 us at D=2048 (C5), but 49 vs 43 us at D=512 (1 KB rows: too many small copies)
      const AttTcrGeom gm = attention_fwd_group_tcr_geom(L, D, A);
      if ((tcr_mode == 2 || (tcr_mode == 1 && D >= 1024)) && (D == 512 || D == 1024 || D == 2048) && gm.smem <= ATTP_SMEM_MAX) {
        auto launch_r = [&](auto kern) -> int {
          SAT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gm.smem));
          SAT_CUDA(sat_launch_pdl(kern, dim3(rows / ncap), dim3(ATTP_FWD_CW * 32 + 32), gm.smem, st, ann, P, wf, hp, ldhp, lens, t, ncap, L, D,
                                  A, scale, alpha, ld_alpha, qsave, z, gz, beta, ld_z, lens_dyn, gm.rows, gm.nst, gm.stage_bytes));
          SAT_COUNT_LAUNCH();
          return 0;
        };
        if (D == 512)
          return launch_r(by_ka(attention_step_fwd_group_tcr_kernel<kExact, ATTP_FWD_CW, 4, 2>, attention_step_fwd_group_tcr_kernel<kExact, ATTP_FWD_CW, 4, 4>,
                                attention_step_fwd_group_tcr_kernel<kExact, ATTP_FWD_CW, 4, 8>));
        if (D == 1024)
          return launch_r(by_ka(attention_step_fwd_group_tcr_kernel<kExact, ATTP_FWD_CW, 8, 2>, attention_step_fwd_group_tcr_kernel<kExact, ATTP_FWD_CW, 8, 4>,
                                attention_step_fwd_group_tcr_kernel<kExact, ATTP_FWD_CW, 8, 8>));
        return launch_r(by_ka(attention_step_fwd_group_tcr_kernel<kExact, ATTP_FWD_CW, 16, 2>, attention_step_fwd_group_tcr_kernel<kExact, ATTP_FWD_CW, 16, 4>,
                              attention_step_fwd_group_tcr_kernel<kExact, ATTP_FWD_CW, 16, 8>));
      }
      if (L <= 16 * ATTG_MAXKS && attention_fwd_group_tc_smem(L, A) <= ATTP_SMEM_MAX) {
      // annotations as a 2-D tensor [n_img * L, D]; the map is rebuilt only when the buffer or shape changes
      static thread_local CUtensorMap tm;
      static thread_local const void* tm_ptr = nullptr;
      static thread_local int64_t tm_rows = 0, tm_d = 0;
      static thread_local int tm_dev = -1;
      const int64_t n_rows = (int64_t)(rows / ncap) * L;
      int dev_now = 0;
      SAT_CUDA(cudaGetDevice(&dev_now));
      if (tm_ptr != (const void*)ann || tm_rows != n_rows || tm_d != D || tm_dev != dev_now) {
        SAT_TRY(tc::make_map(&tm, ann, n_rows, D, D, ATTG_BOX_ROWS));
        tm_ptr = ann; tm_rows = n_rows; tm_d = D; tm_dev = dev_now;
      }
      auto kern = by_ka(attention_step_fwd_group_tc_kernel<kExact, ATTP_FWD_CW, 2>, attention_step_fwd_group_tc_kernel<kExact, ATTP_FWD_CW, 4>,
                        attention_step_fwd_group_tc_kernel<kExact, ATTP_FWD_CW, 8>);
      const size_t smem = attention_fwd_group_tc_smem(L, A);
      SAT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      SAT_CUDA(sat_launch_pdl(kern, dim3(rows / ncap), dim3(ATTP_FWD_CW * 32 + 32), smem, st, tm, P, wf, hp, ldhp, lens, t, ncap, L, D, A,
                              scale, alpha, ld_alpha, qsave, z, gz, beta, ld_z, lens_dyn));
      SAT_COUNT_LAUNCH();
      return 0;
      }
    }
  }
  const size_t gsmem = ncap <= 3 ? attention_fwd_group_smem<3>(L, A) : (ncap <= 5 ? attention_fwd_group_smem<5>(L, A) : attention_fwd_group_smem<8>(L, A));
  if (group && gsmem <= ATTP_SMEM_MAX) {
    auto launch_g = [&](auto kern, size_t smem) -> int {
      SAT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      SAT_CUDA(sat_launch_pdl(kern, dim3(rows / ncap), dim3(ATTP_FWD_CW * 32 + 32), smem, st, ann, P, wf, hp, ldhp, lens, t, ncap, L, D, A,
                              scale, alpha, ld_alpha, qsave, z, gz, beta, ld_z, lens_dyn));
      SAT_COUNT_LAUNCH();
      return 0;
    };
    if (ncap <= 3)
      return launch_g(by_ka(attention_step_fwd_group_kernel<T, kExact, ATTP_FWD_CW, 3, 2>, attention_step_fwd_group_kernel<T, kExact, ATTP_FWD_CW, 3, 4>,
                            attention_step_fwd_group_kernel<T, kExact, ATTP_FWD_CW, 3, 8>), gsmem);
    if (ncap <= 5)
      return launch_g(by_ka(attention_step_fwd_group_kernel<T, kExact, ATTP_FWD_CW, 5, 2>, attention_step_fwd_group_kernel<T, kExact, ATTP_FWD_CW, 5, 4>,
                            attention_step_fwd_group_kernel<T, kExact, ATTP_FWD_CW, 5, 8>), gsmem);
    return launch_g(by_ka(attention_step_fwd_group_kernel<T, kExact, ATTP_FWD_CW, 8, 2>, attention_step_fwd_group_kernel<T, kExact, ATTP_FWD_CW, 8, 4>,
                          attention_step_fwd_group_kernel<T, kExact, ATTP_FWD_CW, 8, 8>), gsmem);
  }
  const size_t smem = attention_fwd_pipe_smem(L, D, A, Vec16<T>::N);
  auto kern = by_ka(attention_step_fwd_pipe_kernel<T, kExact, ATTP_FWD_CW, 2>, attention_step_fwd_pipe_kernel<T, kExact, ATTP_FWD_CW, 4>,
                    attention_step_fwd_pipe_kernel<T, kExact, ATTP_FWD_CW, 8>);
  // set on every launch (sub-microsecond): a per-translation-unit cache of "largest value set so far" is wrong here, because the
  // kernel is one function for the whole library while this launcher is compiled into several translation units -- another
  // unit's launcher may have lowered the attribute in between (seen as "invalid argument" in a long mixed train / decode run)
  if (smem > 48 * 1024) SAT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  SAT_CUDA(sat_launch_pdl(kern, dim3(rows), dim3(ATTP_FWD_CW * 32 + 32), smem, st, ann, P, wf, hp, ldhp, lens, t, ncap, L, D, A, scale, alpha,
                          ld_alpha, qsave, z, gz, beta, ld_z, lens_dyn));
  SAT_COUNT_LAUNCH();
  return 0;
}

// =============================================================================================
// K1b v2: fused attention step, backward, as the same TMA ring pipeline (one CTA per caption row).
//   The producer lane streams the caption's annotation tile (for dalpha_l = a_l . dz) and then its P tile (for the
//   tanh recompute) through the 6 x 16 KB stage ring; 8 consumer warps do
//     A: dz = dZout + dgz*beta, dbeta_pre                 (dgz = sum of the split-K partials of dG*Wihz)
//     B: dalpha_l = a_l . dz + regulariser (+ external)   from the annotation stages
//     C: softmax backward  de_l = alpha_l (dalpha_l - sum alpha dalpha)
//     D: u = tanh(P + q) recomputed from the P stages; dP += dpu (fp32 read-modify-write, 4 rows in flight per warp),
//        dq = sum_l dpu, dwf partial
//   Same math and summation structure per row as attention_step_bwd_kernel (kept as the fallback).
//   KA > 2 (A > 256): in phase D warp w owns the 128-column slice w % KA for the rows w / KA, w / KA + CW / KA, .. of every
//   stage (KA <= CW), so its dq / dwf accumulators stay 8 registers and every warp works on every stage, however few P rows
//   a stage holds.  q and w_f of the slice are read from shared memory once.
// =============================================================================================
constexpr int ATTB_MAXSEG = 4;   // column segments per annotation row (segmented phase B)
constexpr int ATTB_VPL = 4;      // 16-byte annotation vectors per lane kept in registers (D <= 1024 bf16 / 512 fp32)

template <typename T, bool kExact, int CW, int KA = ATTP_REG_KA>
__global__ void __launch_bounds__(CW * 32 + 32, 2)      // two CTAs per SM: all B=256 captions resident in one wave
attention_step_bwd_pipe_kernel(const T* __restrict__ ann, const T* __restrict__ P, const float* __restrict__ wf,
                               const float* __restrict__ q_t, const float* __restrict__ alpha, int64_t ld_alpha,
                               const float* __restrict__ S, const T* __restrict__ z_t, const T* __restrict__ beta_t,
                               const float* __restrict__ dgz, int ns_dgz, int64_t dgz_stride, const float* __restrict__ dZout,
                               int64_t ld_dzout, const int32_t* __restrict__ lens, int t, int ncap, int B, int L, int D, int A,
                               float scale, float gamma, const float* __restrict__ gscale,
                               const float* __restrict__ dalpha_ext, float* __restrict__ dP, T* __restrict__ dP16,
                               T* __restrict__ dZ_t, T* __restrict__ DY_t, int64_t ld_dy, float* __restrict__ dwf_t, float* __restrict__ de_t) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  constexpr int VN = Vec16<T>::N;
  constexpr int ATTP_CWARPS = CW, ATTP_CONSUMERS = CW * 32, ATTP_THREADS = CW * 32 + 32;
  SAT_PDL_TRIGGER();      // as in the forward kernel: the producer primes the ring before SAT_PDL_WAIT()
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = blockIdx.x;
  AttPipeSmem* hd = reinterpret_cast<AttPipeSmem*>(smem_raw);
  const int L4 = (L + 3) & ~3;
  float* dal = reinterpret_cast<float*>(smem_raw + sizeof(AttPipeSmem));   // [L4] regulariser term, then dalpha, then de
  float* als = dal + L4;                // [L4] alpha of this row
  float* dz_s = als + L4;               // [D]
  float* qs = dz_s + D;                 // [A]
  float* ws = qs + A;                   // [A]
  float* dalp = ws + A;                 // [ATTB_MAXSEG][L4] per-column-segment partials (segmented phase B only)
  const uint32_t stage_off =
      (uint32_t)((sizeof(AttPipeSmem) + sizeof(float) * (size_t)((2 + ATTB_MAXSEG) * L4 + D + 2 * A) + 127) & ~(size_t)127);
  uint8_t* stages = smem_raw + stage_off;
  float* red = reinterpret_cast<float*>(stages);   // [ATTP_CWARPS][2A]: aliases the ring, used only after its last stage is drained

  T* dy_b = DY_t + (int64_t)b * ld_dy;
  if (t >= lens[b]) {
    SAT_PDL_WAIT();
    for (int i = tid; i < A + D; i += ATTP_THREADS) dy_b[i] = from_f<T>(0.f);
    for (int d = tid; d < D; d += ATTP_THREADS) dZ_t[(int64_t)b * D + d] = from_f<T>(0.f);
    for (int a = tid; a < A; a += ATTP_THREADS) dwf_t[(int64_t)b * A + a] = 0.0f;
    return;
  }
  const int img = b / ncap;
  const int RCP = ATTP_STAGE_BYTES / (A * (int)sizeof(T));
  const int RCA = ATTP_STAGE_BYTES / (D * (int)sizeof(T));
  const int nP = (L + RCP - 1) / RCP, nA = (L + RCA - 1) / RCA;
  if (tid == 0) {
    for (int i = 0; i < ATTP_NST; ++i) {
      sat_mbar_init(&hd->full[i], 1);
      sat_mbar_init(&hd->empty[i], ATTP_CWARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();

  if (warp == ATTP_CWARPS) {
    if (lane == 0) {   // ===== producer: annotation chunks first, then P chunks =====
      const T* Pb = P + (int64_t)img * L * A;
      const T* ab = ann + (int64_t)img * L * D;
      for (int i = 0; i < nA + nP; ++i) {
        const int st = i % ATTP_NST;
        const uint32_t ph = (uint32_t)(i / ATTP_NST) & 1u;
        sat_mbar_wait(&hd->empty[st], ph ^ 1u);
        const void* src;
        uint32_t bytes;
        if (i < nA) {
          const int r0 = i * RCA, rows = min(RCA, L - r0);
          src = ab + (int64_t)r0 * D;
          bytes = (uint32_t)(rows * D * (int)sizeof(T));
        } else {
          const int r0 = (i - nA) * RCP, rows = min(RCP, L - r0);
          src = Pb + (int64_t)r0 * A;
          bytes = (uint32_t)(rows * A * (int)sizeof(T));
        }
        sat_mbar_expect_tx(&hd->full[st], bytes);
        sat_bulk_g2s(stages + (size_t)st * ATTP_STAGE_BYTES, src, bytes, &hd->full[st]);
      }
    }
    return;
  }

  // ===== consumers =====
  SAT_PDL_WAIT();
  const float g = gscale ? *gscale : 1.0f;
  const float* alpha_b = alpha + (int64_t)b * ld_alpha;
  // phase A: every global load of this phase is issued up front (4 columns per thread, one latency), and the
  // per-location additive terms of dalpha (regulariser, external grad) are staged in dal[] so that phase B is pure smem
  const float regc = g * gamma * (-2.0f) / ((float)B * (float)L);
  for (int d4 = tid * 4; d4 < D; d4 += ATTP_CONSUMERS * 4) {
    float4 dg = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int sp0 = 0; sp0 < ns_dgz; sp0 += 8) {      // split-K partials: 8 independent loads in flight, then the adds
      float4 p4[8];
#pragma unroll
      for (int u = 0; u < 8; ++u)
        p4[u] = (sp0 + u) < ns_dgz ? *reinterpret_cast<const float4*>(dgz + (int64_t)(sp0 + u) * dgz_stride + (int64_t)b * D + d4)
                                   : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int u = 0; u < 8; ++u) { dg.x += p4[u].x; dg.y += p4[u].y; dg.z += p4[u].z; dg.w += p4[u].w; }
    }
    const float4 bt = ld4(beta_t + (int64_t)b * D + d4);
    const float4 zz = ld4(z_t + (int64_t)b * D + d4);
    const float4 dzo = *reinterpret_cast<const float4*>(dZout + (int64_t)b * ld_dzout + d4);
    const float4 dzv = make_float4(dzo.x + dg.x * bt.x, dzo.y + dg.y * bt.y, dzo.z + dg.z * bt.z, dzo.w + dg.w * bt.w);
    *reinterpret_cast<float4*>(dz_s + d4) = dzv;
    st4(dZ_t + (int64_t)b * D + d4, dzv);
    st4(dy_b + A + d4, make_float4(dg.x * zz.x * bt.x * (1.0f - bt.x), dg.y * zz.y * bt.y * (1.0f - bt.y),
                                   dg.z * zz.z * bt.z * (1.0f - bt.z), dg.w * zz.w * bt.w * (1.0f - bt.w)));
  }
  for (int a = tid; a < A; a += ATTP_CONSUMERS) {
    qs[a] = q_t[(int64_t)b * A + a];
    ws[a] = wf[a];
  }
  for (int l = tid; l < L; l += ATTP_CONSUMERS) {
    als[l] = alpha_b[l];
    float extra = regc * (1.0f - S[(int64_t)b * L + l]);
    if (dalpha_ext) extra += dalpha_ext[(int64_t)b * ld_alpha + l];
    dal[l] = extra;
  }
  sat_named_bar(1, ATTP_CONSUMERS);

  // phase B: dalpha from the annotation stages (one warp per row, lanes over 16-byte vectors of the row)
  const int NV = D / VN;
  // Short stages (rows of a stage < consumer warps) or rows longer than the register slice: split every row into nseg
  // column segments so that (row, segment) items spread evenly over the warps; a warp always owns the same segment.
  int seglen = 0, nseg = 1;
  if (RCA < ATTP_CWARPS || NV > 32 * ATTB_VPL) {
    int best = 1 << 30;
    for (int c = 32; c <= 32 * ATTB_VPL; c += 32) {
      const int ns = (NV + c - 1) / c;
      if (ns > ATTB_MAXSEG || ATTP_CWARPS % ns != 0) continue;
      const int cost = ((RCA * ns + ATTP_CWARPS - 1) / ATTP_CWARPS) * c;
      if (cost <= best) { best = cost; seglen = c; nseg = ns; }
    }
  }
  const bool segpath = seglen > 0;
  const bool regpath = !segpath && NV <= 32 * ATTB_VPL;
  const int seg = segpath ? warp % nseg : 0;
  const int lw = warp / nseg, lstep = ATTP_CWARPS / nseg;     // segmented path: this warp's rows inside a stage
  float dzr[ATTB_VPL][VN];
  if (regpath || segpath) {
#pragma unroll
    for (int k = 0; k < ATTB_VPL; ++k) {
      const int cv = seg * seglen + lane + 32 * k;
      const bool ok = cv < NV && (!segpath || 32 * k < seglen);
#pragma unroll
      for (int i = 0; i < VN; ++i) dzr[k][i] = ok ? dz_s[cv * VN + i] : 0.0f;
    }
  }
  int it = 0;
  for (int j = 0; j < nA; ++j, ++it) {
    const int st = it % ATTP_NST;
    sat_mbar_wait(&hd->full[st], (uint32_t)(it / ATTP_NST) & 1u);
    const T* As = reinterpret_cast<const T*>(stages + (size_t)st * ATTP_STAGE_BYTES);
    const int r0 = j * RCA, rows = min(RCA, L - r0);
    if (segpath) {
      for (int l = lw; l < rows; l += lstep) {
        float s = 0.0f;
#pragma unroll
        for (int k = 0; k < ATTB_VPL; ++k) {
          const int cv = seg * seglen + lane + 32 * k;
          if (32 * k < seglen && cv < NV) {
            float v[VN];
            Vec16<T>::load_shared(As + (size_t)l * D + cv * VN, v);
#pragma unroll
            for (int i = 0; i < VN; ++i) s = fmaf(v[i], dzr[k][i], s);
          }
        }
        s = warp_sum(s);
        if (lane == 0) dalp[seg * L4 + r0 + l] = s;
      }
    } else if (regpath) {
      // two rows of the stage per pass (independent FMA chains and shuffle trees)
      for (int l = warp; l < rows; l += 2 * ATTP_CWARPS) {
        const int l2 = l + ATTP_CWARPS;
        const bool h2 = l2 < rows;
        float s = 0.0f, s2 = 0.0f, sb = 0.0f, s2b = 0.0f;
#pragma unroll
        for (int k = 0; k < ATTB_VPL; ++k) {
          const int cv = lane + 32 * k;
          if (cv < NV) {
            float v[VN], v2[VN];
            Vec16<T>::load_shared(As + (size_t)l * D + cv * VN, v);
            Vec16<T>::load_shared(As + (size_t)(h2 ? l2 : l) * D + cv * VN, v2);
#pragma unroll
            for (int i = 0; i < VN; i += 2) {
              s = fmaf(v[i], dzr[k][i], s);
              sb = fmaf(v[i + 1], dzr[k][i + 1], sb);
              s2 = fmaf(v2[i], dzr[k][i], s2);
              s2b = fmaf(v2[i + 1], dzr[k][i + 1], s2b);
            }
          }
        }
        s = warp_sum(s + sb);
        s2 = warp_sum(s2 + s2b);
        if (lane == 0) {
          dal[r0 + l] += s;
          if (h2) dal[r0 + l2] += s2;
        }
      }
    } else
    for (int l = warp; l < rows; l += ATTP_CWARPS) {
      float s = 0.0f;
      if (false) {
      } else {
        for (int cv = lane; cv < NV; cv += 32) {
          float v[VN];
          Vec16<T>::load_shared(As + (size_t)l * D + cv * VN, v);
#pragma unroll
          for (int i = 0; i < VN; ++i) s = fmaf(v[i], dz_s[cv * VN + i], s);
        }
      }
      s = warp_sum(s);
      if (lane == 0) dal[r0 + l] += s;
    }
    __syncwarp();
    if (lane == 0) sat_mbar_arrive(&hd->empty[st]);
  }
  sat_named_bar(1, ATTP_CONSUMERS);
  if (segpath) {
    for (int l = tid; l < L; l += ATTP_CONSUMERS) {      // same thread -> location mapping as the loops below
      float v = dal[l];
      for (int sg = 0; sg < nseg; ++sg) v += dalp[sg * L4 + l];
      dal[l] = v;
    }
  }
  // phase C: softmax backward
  float dot = 0.0f;
  for (int l = tid; l < L; l += ATTP_CONSUMERS) dot = fmaf(als[l], dal[l], dot);
  dot = warp_sum(dot);
  if (lane == 0) hd->red_a[warp] = dot;
  sat_named_bar(1, ATTP_CONSUMERS);
  dot = 0.0f;
#pragma unroll
  for (int w2 = 0; w2 < ATTP_CWARPS; ++w2) dot += hd->red_a[w2];
  for (int l = tid; l < L; l += ATTP_CONSUMERS) {
    const float de = als[l] * (dal[l] - dot) * scale;   // de_l * scale
    dal[l] = de;
    de_t[(int64_t)b * L + l] = de;      // kept for the deferred dP pass (dP_deferred_kernel)
  }
  sat_named_bar(1, ATTP_CONSUMERS);

  if constexpr (KA != ATTP_REG_KA) {
    static_assert(KA <= CW && CW % KA == 0, "one column slice per warp");
    // phase D, KA > 2: warp w owns columns 128 * (w % KA) + lane * 4 .. +3 for the 4-row groups rsub, rsub + RS, .. of a stage
    constexpr int RS = CW / KA;
    const int ks = warp % KA, rsub = warp / KA;
    const int a = lane * 4 + 128 * ks;
    const bool own = a < A;
    float4 q4 = make_float4(0.f, 0.f, 0.f, 0.f), w4 = q4;
    if (own) {
      q4 = *reinterpret_cast<const float4*>(qs + a);
      w4 = *reinterpret_cast<const float4*>(ws + a);
    }
    const float qv[4] = {q4.x, q4.y, q4.z, q4.w}, wv[4] = {w4.x, w4.y, w4.z, w4.w};
    float dq[4] = {0.f, 0.f, 0.f, 0.f}, dw[4] = {0.f, 0.f, 0.f, 0.f};
    for (int j = 0; j < nP; ++j, ++it) {
      const int st = it % ATTP_NST;
      sat_mbar_wait(&hd->full[st], (uint32_t)(it / ATTP_NST) & 1u);
      const T* Ps = reinterpret_cast<const T*>(stages + (size_t)st * ATTP_STAGE_BYTES);
      const int r0 = j * RCP, rows = min(RCP, L - r0);
      if (own) {
        for (int l0 = rsub * 4; l0 < rows; l0 += RS * 4) {
          float4 p[4];
          float de[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const bool ok = (l0 + u) < rows;
            p[u] = ok ? ld4(Ps + (size_t)(l0 + u) * A + a) : make_float4(0.f, 0.f, 0.f, 0.f);
            de[u] = ok ? dal[r0 + l0 + u] : 0.0f;
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const float pv[4] = {p[u].x, p[u].y, p[u].z, p[u].w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float uu = sat_tanh<kExact>(pv[i] + qv[i]);
              dq[i] = fmaf(de[u] * wv[i], 1.0f - uu * uu, dq[i]);
              dw[i] = fmaf(de[u], uu, dw[i]);
            }
          }
        }
      }
      __syncwarp();
      if (lane == 0) sat_mbar_arrive(&hd->empty[st]);
    }
    sat_named_bar(1, ATTP_CONSUMERS);     // every warp is done reading the ring before red[] overwrites it
    if (own) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        red[rsub * 2 * A + a + i] = dq[i];
        red[rsub * 2 * A + A + a + i] = dw[i];
      }
    }
    sat_named_bar(1, ATTP_CONSUMERS);
    for (int a2 = tid; a2 < A; a2 += ATTP_CONSUMERS) {
      float sq = 0.0f, sw = 0.0f;
#pragma unroll
      for (int r = 0; r < RS; ++r) { sq += red[r * 2 * A + a2]; sw += red[r * 2 * A + A + a2]; }
      dy_b[a2] = from_f<T>(sq);
      dwf_t[(int64_t)b * A + a2] = sw;
    }
    return;
  }
  // phase D: through tanh into P, q, wf (lane owns attention columns lane*4 + 128k)
  float qreg[ATTP_REG_KA][4], wreg[ATTP_REG_KA][4], dq[ATTP_REG_KA][4], dw[ATTP_REG_KA][4];
#pragma unroll
  for (int k = 0; k < ATTP_REG_KA; ++k) {
    const int a = lane * 4 + 128 * k;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      qreg[k][i] = a < A ? qs[a + i] : 0.0f;
      wreg[k][i] = a < A ? ws[a + i] : 0.0f;
      dq[k][i] = 0.0f;
      dw[k][i] = 0.0f;
    }
  }
  // (dP itself is not touched here: it is rebuilt after the time loop from the saved de_t and q_t, which removes a
  //  2 x B*L*A*4-byte read-modify-write per step)
  for (int j = 0; j < nP; ++j, ++it) {
    const int st = it % ATTP_NST;
    sat_mbar_wait(&hd->full[st], (uint32_t)(it / ATTP_NST) & 1u);
    const T* Ps = reinterpret_cast<const T*>(stages + (size_t)st * ATTP_STAGE_BYTES);
    const int r0 = j * RCP, rows = min(RCP, L - r0);
    for (int l0 = warp * 4; l0 < rows; l0 += ATTP_CWARPS * 4) {      // 4 rows in flight per warp
#pragma unroll
      for (int k = 0; k < ATTP_REG_KA; ++k) {
        const int a = lane * 4 + 128 * k;
        if (a < A) {
          float4 p[4];
          float de[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const bool ok = (l0 + u) < rows;
            p[u] = ok ? ld4(Ps + (size_t)(l0 + u) * A + a) : make_float4(0.f, 0.f, 0.f, 0.f);
            de[u] = ok ? dal[r0 + l0 + u] : 0.0f;
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const float pv[4] = {p[u].x, p[u].y, p[u].z, p[u].w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float uu = sat_tanh<kExact>(pv[i] + qreg[k][i]);
              dq[k][i] = fmaf(de[u] * wreg[k][i], 1.0f - uu * uu, dq[k][i]);
              dw[k][i] = fmaf(de[u], uu, dw[k][i]);
            }
          }
        }
      }
    }
    __syncwarp();
    if (lane == 0) sat_mbar_arrive(&hd->empty[st]);
  }
  sat_named_bar(1, ATTP_CONSUMERS);     // every warp is done reading the ring before red[] overwrites it
#pragma unroll
  for (int k = 0; k < ATTP_REG_KA; ++k) {
    const int a = lane * 4 + 128 * k;
    if (a < A) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        red[warp * 2 * A + a + i] = dq[k][i];
        red[warp * 2 * A + A + a + i] = dw[k][i];
      }
    }
  }
  sat_named_bar(1, ATTP_CONSUMERS);
  for (int a = tid; a < A; a += ATTP_CONSUMERS) {
    float sq = 0.0f, sw = 0.0f;
#pragma unroll
    for (int w2 = 0; w2 < ATTP_CWARPS; ++w2) { sq += red[w2 * 2 * A + a]; sw += red[w2 * 2 * A + A + a]; }
    dy_b[a] = from_f<T>(sq);
    dwf_t[(int64_t)b * A + a] = sw;
  }
}

// dP[b,l,a] = sum_t de[t,b,l] * w_f[a] * (1 - tanh^2(P[img,l,a] + q[t,b,a])), t = lens[b]-1 .. 0: the grad wrt the
// per-image projection P, rebuilt once after the time loop (model.py:100-104 under autograd).  One CTA per (row tile,
// caption, column chunk): q[:,b,chunk] and de[:,b,tile] are staged in smem, every warp walks 4 rows at a time, a lane owns
// 4 columns.  The column chunk (AC columns, a multiple of 128, or all of A) bounds the staged q at Tmax * AC floats.
constexpr int DPD_ROWS = 32;
template <typename T, bool kExact, bool kCols>
__global__ void __launch_bounds__(256, kCols ? 1 : 4)     // kCols: the staged q fills most of the shared memory of an SM
dP_deferred_kernel(const T* __restrict__ P, const float* __restrict__ wf, const float* __restrict__ Q,
                   const float* __restrict__ de, const int32_t* __restrict__ lens, int ncap, int B, int L, int A, int Tmax,
                   float* __restrict__ dP, T* __restrict__ dP16, int ac_arg) {
  extern __shared__ __align__(16) float dpd_smem[];
  const int b = blockIdx.y, r0 = blockIdx.x * DPD_ROWS, rows = min(DPD_ROWS, L - r0);
  const int AC = kCols ? ac_arg : A;                                    // !kCols: one chunk, all of A
  const int a0 = kCols ? (int)blockIdx.z * AC : 0, nac = kCols ? min(AC, A - a0) : A;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int Tb = min(lens[b], Tmax);    // shared memory is sized for Tmax steps
  float* qs = dpd_smem;                       // [Tb][AC]
  float* des = qs + (size_t)Tb * AC;          // [Tb][DPD_ROWS]
  for (int i = tid; i < Tb * nac; i += 256) qs[(i / nac) * AC + (i % nac)] = Q[((int64_t)(i / nac) * B + b) * A + a0 + (i % nac)];
  for (int i = tid; i < Tb * DPD_ROWS; i += 256) {
    const int t = i / DPD_ROWS, l = i % DPD_ROWS;
    des[i] = l < rows ? de[((int64_t)t * B + b) * L + r0 + l] : 0.0f;
  }
  __syncthreads();
  const T* Pb = P + ((int64_t)(b / ncap) * L + r0) * A;
  const int l0 = warp * 4;
  if (l0 >= rows) return;
  for (int a = a0 + lane * 4; a < a0 + nac; a += 128) {
    const float4 w4 = *reinterpret_cast<const float4*>(wf + a);
    const float wv[4] = {w4.x, w4.y, w4.z, w4.w};
    float pv[4][4], acc[4][4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float4 p = (l0 + u) < rows ? ld4(Pb + (size_t)(l0 + u) * A + a) : make_float4(0.f, 0.f, 0.f, 0.f);
      pv[u][0] = p.x; pv[u][1] = p.y; pv[u][2] = p.z; pv[u][3] = p.w;
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[u][i] = 0.0f;
    }
    for (int t = Tb - 1; t >= 0; --t) {
      const float4 q4 = *reinterpret_cast<const float4*>(qs + (size_t)t * AC + (a - a0));
      const float qv[4] = {q4.x, q4.y, q4.z, q4.w};
      const float4 d4 = *reinterpret_cast<const float4*>(des + (size_t)t * DPD_ROWS + l0);
      const float dv[4] = {d4.x, d4.y, d4.z, d4.w};
#pragma unroll
      for (int u = 0; u < 4; ++u) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float uu = sat_tanh<kExact>(pv[u][i] + qv[i]);
          acc[u][i] += dv[u] * wv[i] * (1.0f - uu * uu);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if ((l0 + u) < rows) {
        const float4 r = make_float4(acc[u][0], acc[u][1], acc[u][2], acc[u][3]);
        const int64_t o = ((int64_t)b * L + r0 + l0 + u) * A + a;
        *reinterpret_cast<float4*>(dP + o) = r;
        if (dP16) st4(dP16 + o, r);
      }
    }
  }
}

static inline size_t attention_bwd_pipe_smem(int L, int D, int A) {
  const int L4 = (L + 3) & ~3;
  return ((sizeof(AttPipeSmem) + sizeof(float) * (size_t)((2 + ATTB_MAXSEG) * L4 + D + 2 * A) + 127) & ~(size_t)127) + 128 +
         (size_t)ATTP_NST * ATTP_STAGE_BYTES;
}

// dP_deferred_kernel: columns per CTA so that q of Tmax steps fits the shared memory of a block (all of A when it fits, as
// many 128-column slices as fit otherwise); 0 where not even one slice fits (the step-by-step backward kernel runs instead)
static inline int dP_deferred_cols(int T, int A) {
  auto bytes = [T](int ac) { return sizeof(float) * (size_t)T * (ac + DPD_ROWS); };
  if (bytes(A) <= ATTP_SMEM_MAX) return A;
  int ac = 128;
  while (ac + 128 < A && bytes(ac + 128) <= ATTP_SMEM_MAX) ac += 128;
  return bytes(ac) <= ATTP_SMEM_MAX ? ac : 0;
}

template <typename T>
static inline bool attention_bwd_pipe_ok(int D, int A) {
  static int mode = -2;                       // SAT_ATTB_MODE=0 forces the plain kernel (A/B timing)
  if (mode == -2) {
    const char* e = getenv("SAT_ATTB_MODE");
    mode = e ? atoi(e) : -1;
  }
  if (mode == 0) return false;
  return D * (int)sizeof(T) <= ATTP_STAGE_BYTES && A <= 128 * ATTP_MAXKA;
}
