// Common device/host helpers for the SAT decoder kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/sat_b200.h"

typedef __nv_bfloat16 bf16;

// ---- error plumbing (thread-local message behind sat_last_error()) --------------------
void sat_set_error(const char* fmt, ...);

#define SAT_REQUIRE(cond, ...)                                   \
  do {                                                           \
    if (!(cond)) {                                               \
      sat_set_error(__VA_ARGS__);                                \
      return SAT_ERR_INVALID;                                    \
    }                                                            \
  } while (0)

#define SAT_CUDA(call)                                                               \
  do {                                                                               \
    cudaError_t e__ = (call);                                                        \
    if (e__ != cudaSuccess) {                                                        \
      sat_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
      return (int)e__;                                                               \
    }                                                                                \
  } while (0)

#define SAT_LAUNCH_OK() SAT_CUDA(cudaGetLastError())

#define SAT_TRY(call)            \
  do {                           \
    int r__ = (call);            \
    if (r__ != 0) return r__;    \
  } while (0)

// launch counter (gpu_launches claim in bench.py)
extern unsigned long long g_sat_launches;
#define SAT_COUNT_LAUNCH() (++g_sat_launches)

// optional per-kernel event timing (sat_profile_begin / sat_profile_end)
extern int g_sat_prof_kind;
void sat_prof_mark(cudaStream_t st);
#define SAT_PROF(kind, st) do { if (g_sat_prof_kind == (kind)) sat_prof_mark(st); } while (0)

// ---- programmatic dependent launch (PDL) ---------------------------------------------------------
// The decoder is a long chain of short dependent kernels.  Kernels launched through sat_launch_pdl may be scheduled
// while their predecessor drains; they call SAT_PDL_TRIGGER() first (so their own successor can do the same) and
// SAT_PDL_WAIT() before the first global-memory access that depends on (or could disturb) the predecessor.
#define SAT_PDL_TRIGGER() asm volatile("griddepcontrol.launch_dependents;" ::: "memory")
#define SAT_PDL_WAIT() asm volatile("griddepcontrol.wait;" ::: "memory")
// Kernels on this path read operands that are constant inside a driver's launch chain (annotations, P, packed weights)
// BEFORE SAT_PDL_WAIT().  The single-op entry points (sat_linear, sat_attention_step_fwd) take caller-supplied operands
// that may be the output of the caller's previous launch, so they launch without the attribute (SatNoPdlScope): the
// kernel then starts only after everything before it in the stream has completed.
inline bool& sat_pdl_allowed() {          // one flag per host thread for the whole library (inline: shared by all translation units)
  static thread_local bool allowed = true;      // per host thread: drivers on different threads / streams do not interfere
  return allowed;
}
struct SatNoPdlScope {
  bool prev;
  SatNoPdlScope() : prev(sat_pdl_allowed()) { sat_pdl_allowed() = false; }
  ~SatNoPdlScope() { sat_pdl_allowed() = prev; }      // scopes nest
};
// Optional L2 persistence window for the next launches of this host thread (cudaLaunchAttributeAccessPolicyWindow): the
// attention kernels re-read the same annotation tensor at every time step, and at BASELINE configs[1] it fits the 126 MB
// L2.  The drivers set the window around their time loop; sat_launch_pdl attaches it to every launch while it is set.
struct SatL2Window {
  const void* ptr = nullptr;
  size_t bytes = 0;
  float hit_ratio = 1.0f;
};
inline SatL2Window& sat_l2_window() {
  static thread_local SatL2Window w;
  return w;
}
// one-time per device: reserve the persisting carve-out (returns the window size that may be used, 0 = unsupported / disabled)
size_t sat_l2_persist_limit();

template <typename Kern, typename... Args>
static inline cudaError_t sat_launch_pdl(Kern kern, dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (sat_pdl_allowed()) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  const SatL2Window& w = sat_l2_window();
  if (w.ptr != nullptr && w.bytes > 0) {
    attr[na].id = cudaLaunchAttributeAccessPolicyWindow;
    attr[na].val.accessPolicyWindow.base_ptr = const_cast<void*>(w.ptr);
    attr[na].val.accessPolicyWindow.num_bytes = w.bytes;
    attr[na].val.accessPolicyWindow.hitRatio = w.hit_ratio;
    attr[na].val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    attr[na].val.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  return cudaLaunchKernelEx(&cfg, kern, args...);
}

// same, for kernels that run as thread-block clusters of `cluster_x` CTAs along x (distributed shared memory between the CTAs)
template <typename Kern, typename... Args>
static inline cudaError_t sat_launch_cluster_pdl(Kern kern, dim3 grid, dim3 block, size_t smem, unsigned cluster_x, cudaStream_t st,
                                                 Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  int na = 0;
  attr[na].id = cudaLaunchAttributeClusterDimension;
  attr[na].val.clusterDim.x = cluster_x;
  attr[na].val.clusterDim.y = 1;
  attr[na].val.clusterDim.z = 1;
  ++na;
  if (sat_pdl_allowed()) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  return cudaLaunchKernelEx(&cfg, kern, args...);
}

// ---- typed loads / stores ------------------------------------------------------------
__device__ __forceinline__ float to_f(float v) { return v; }
__device__ __forceinline__ float to_f(bf16 v) { return __bfloat162float(v); }

template <typename T> __device__ __forceinline__ T from_f(float v);
template <> __device__ __forceinline__ float from_f<float>(float v) { return v; }
template <> __device__ __forceinline__ bf16 from_f<bf16>(float v) { return __float2bfloat16_rn(v); }

// 4 consecutive elements -> float4 (pointer must be 16B (float) / 8B (bf16) aligned)
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 ld4(const bf16* p) {
  uint2 r = *reinterpret_cast<const uint2*>(p);
  __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&r.x);
  __nv_bfloat162 b = *reinterpret_cast<__nv_bfloat162*>(&r.y);
  float2 fa = __bfloat1622float2(a), fb = __bfloat1622float2(b);
  return make_float4(fa.x, fa.y, fb.x, fb.y);
}
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void st4(bf16* p, float4 v) {
  __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y);
  __nv_bfloat162 b = __floats2bfloat162_rn(v.z, v.w);
  uint2 r;
  r.x = *reinterpret_cast<uint32_t*>(&a);
  r.y = *reinterpret_cast<uint32_t*>(&b);
  *reinterpret_cast<uint2*>(p) = r;
}

// 16-byte vector of T -> floats (float: 4 values, bf16: 8 values)
template <typename T> struct Vec16;
template <> struct Vec16<float> {
  static constexpr int N = 4;
  __device__ __forceinline__ static void load(const float* p, float* o) {
    float4 v = __ldg(reinterpret_cast<const float4*>(p));
    o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
  }
  __device__ __forceinline__ static void load_shared(const float* p, float* o) {
    float4 v = *reinterpret_cast<const float4*>(p);
    o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
  }
  __device__ __forceinline__ static void store(float* p, const float* o) {
    *reinterpret_cast<float4*>(p) = make_float4(o[0], o[1], o[2], o[3]);
  }
};
template <> struct Vec16<bf16> {
  static constexpr int N = 8;
  __device__ __forceinline__ static void load(const bf16* p, float* o) {
    uint4 r = __ldg(reinterpret_cast<const uint4*>(p));
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&r);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float2 f = __bfloat1622float2(h[i]);
      o[2 * i] = f.x; o[2 * i + 1] = f.y;
    }
  }
  __device__ __forceinline__ static void load_shared(const bf16* p, float* o) {
    uint4 r = *reinterpret_cast<const uint4*>(p);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&r);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float2 f = __bfloat1622float2(h[i]);
      o[2 * i] = f.x; o[2 * i + 1] = f.y;
    }
  }
  __device__ __forceinline__ static void store(bf16* p, const float* o) {
    uint4 r;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&r);
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(o[2 * i], o[2 * i + 1]);
    *reinterpret_cast<uint4*>(p) = r;
  }
};

// ---- math ------------------------------------------------------------------------------
// kExact = true : IEEE-accurate libm paths (fp32 parity mode, 1e-5 vs the CPU oracle)
// kExact = false: MUFU approximations (bf16 throughput mode)
template <bool kExact> __device__ __forceinline__ float sat_tanh(float x) {
  if (kExact) return tanhf(x);
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
template <bool kExact> __device__ __forceinline__ float sat_exp(float x) {
  if (kExact) return expf(x);
  return __expf(x);
}
template <bool kExact> __device__ __forceinline__ float sat_sigmoid(float x) {
  if (kExact) return 1.0f / (1.0f + expf(-x));
  return __fdividef(1.0f, 1.0f + __expf(-x));
}

// A word id as the kernels use it: ids outside [0, V0) (nn.Embedding would raise) are fed and scored as <PAD> (id 0);
// tok_init_kernel flags such a caption in out[6].  The one rule for the fed words and both cross-entropy paths' targets.
__device__ __forceinline__ int sat_word_or_pad(int w, int V0) { return (unsigned)w < (unsigned)V0 ? w : 0; }

// ---- dropout: stateless counter-based masks ------------------------------------------------------
// keep(seed, stream, idx) is a pure function, so the backward pass regenerates the forward masks instead of storing them.
// streams: 1 = InitLSTM mean (model.py:78), 2 = embedding_dropout (model.py:526), 3 = DeepOutput dropout (model.py:130)
__host__ __device__ __forceinline__ uint32_t sat_hash32(uint64_t seed, uint32_t stream, uint64_t idx) {
  uint64_t x = idx * 0x9E3779B97F4A7C15ull + seed + ((uint64_t)stream << 56);
  x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull;
  x ^= x >> 27; x *= 0x94D049BB133111EBull;
  x ^= x >> 31;
  return (uint32_t)(x >> 32);
}
// multiplier of an element under inverted dropout with drop probability p: 0 or 1/(1-p)
__host__ __device__ __forceinline__ float sat_dropout_scale(float p, uint64_t seed, uint32_t stream, uint64_t idx) {
  if (p <= 0.0f) return 1.0f;
  const float u = (float)(sat_hash32(seed, stream, idx) >> 8) * (1.0f / 16777216.0f);
  return u < p ? 0.0f : 1.0f / (1.0f - p);
}
// sampling decoders: uniform in (0, 1) and standard Gumbel noise, pure functions of (seed, stream, idx)
__device__ __forceinline__ float sat_uniform01(uint64_t seed, uint32_t stream, uint64_t idx) {
  return ((float)(sat_hash32(seed, stream, idx) >> 8) + 0.5f) * (1.0f / 16777216.0f);
}
__device__ __forceinline__ float sat_gumbel(uint64_t seed, uint32_t stream, uint64_t idx) {
  return -logf(-logf(sat_uniform01(seed, stream, idx)));
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// block-wide reductions for blockDim.x <= 1024 (scratch: 33 floats of shared memory)
__device__ __forceinline__ float block_sum(float v, float* scratch) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) scratch[wid] = v;
  __syncthreads();
  if (wid == 0) {
    float r = lane < nw ? scratch[lane] : 0.0f;
    r = warp_sum(r);
    if (lane == 0) scratch[32] = r;
  }
  __syncthreads();
  return scratch[32];
}
__device__ __forceinline__ float block_max(float v, float* scratch) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_max(v);
  __syncthreads();
  if (lane == 0) scratch[wid] = v;
  __syncthreads();
  if (wid == 0) {
    float r = lane < nw ? scratch[lane] : -INFINITY;
    r = warp_max(r);
    if (lane == 0) scratch[32] = r;
  }
  __syncthreads();
  return scratch[32];
}
