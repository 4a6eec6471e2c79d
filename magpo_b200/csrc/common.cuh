// Shared helpers for the magpo_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <algorithm>
#include <stdint.h>
#include <stdio.h>

#include "../../include/magpo_b200.h"

namespace magpo {

void set_cuda_error(cudaError_t e, const char* file, int line);
void set_error_text(const char* msg);  // text returned by magpo_last_cuda_error() (also used for NCCL failures)

#define MAGPO_CUDA_OK(expr)                                   \
  do {                                                        \
    cudaError_t _e = (expr);                                  \
    if (_e != cudaSuccess) {                                  \
      ::magpo::set_cuda_error(_e, __FILE__, __LINE__);        \
      return MAGPO_ERR_CUDA;                                  \
    }                                                         \
  } while (0)

void note_launch();
#define MAGPO_LAUNCH_OK()              \
  do {                                 \
    ::magpo::note_launch();            \
    MAGPO_CUDA_OK(cudaGetLastError()); \
  } while (0)

// Optional per-category device timing (CUDA events on the launching stream), used by bench.py for the live
// roofline numbers and the per-kernel breakdown. Off by default; zero cost when off.
enum ProfCat {
  PROF_GEMM_NN = 0, PROF_GEMM_TN, PROF_COLSUM, PROF_ROWOPS, PROF_RET_FWD, PROF_RET_BWD, PROF_GRU, PROF_LOSS, PROF_PACK,
  PROF_OPTIM, PROF_ENV, PROF_SAMPLE, PROF_GAE, PROF_MISC, PROF_GEMM_SMALL /* M < 64 Ki rows: the rollout */, PROF_CHAIN /* fused row chains */, PROF_NUM
};
struct ProfScope {
  int idx;
  cudaStream_t s;
  ProfScope(int cat, cudaStream_t s, double work, double bytes = 0.0);  // bytes: algorithmic HBM bytes when `work` is flops
  ~ProfScope();
};

#define MAGPO_TRY(expr)          \
  do {                           \
    int _r = (expr);             \
    if (_r != MAGPO_OK) return _r; \
  } while (0)

// ---- per-device context (MagpoContext of the C ABI): everything an entry point needs besides its arguments. Created by the caller
// (magpo_context_create), passed to every entry point that forks streams or looks up tensor-core weight images; nothing of it is
// process-global, so several learners (and several devices) can be driven from one process. The only process-wide switches are the
// benchmark / test hooks magpo_prof_*, magpo_debug_set_overlap and magpo_set_chain_kernels; the product path never sets them.
struct ForkJoin {  // a forked stream + the events that fork it off / join it back into the caller's stream
  cudaStream_t s = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
  int init();
  void destroy();
};
struct TcRegion {  // a weight region whose TF32 hi / lo images exist (gemm_tc.cu)
  const float* base;
  int64_t n;
  const float *hi, *lo;
};
}  // namespace magpo
#include <vector>
struct MagpoComm;
struct MagpoContext {
  int device = -1;
  MagpoComm* comm = nullptr;  // data-parallel communicator (comm.cu), attached by magpo_context_set_comm
  magpo::ForkJoin side;   // update: the learner's forward / backward beside the guider's (update.cu)
  magpo::ForkJoin dec;    // guider forward: the decoder's encoder-independent prefix beside the encoder (sable.cu)
  magpo::ForkJoin rside;  // rollout: the learner's GRU push beside the guider step kernel (rollout.cu)
  std::vector<magpo::TcRegion> regions;
};
namespace magpo {
using Context = ::MagpoContext;
// The context of the entry point running on this thread. Entry points that take a MagpoContext* install it with CtxScope for the
// duration of the call; the magpo_test_* hooks, which take none, get a thread-local scratch context.
Context& ctx();
struct CtxScope {
  Context* prev;
  bool ok;
  explicit CtxScope(Context* c);
  ~CtxScope();
};
#define MAGPO_CTX(c)             \
  ::magpo::CtxScope _ctx_scope(c); \
  if (!_ctx_scope.ok) return MAGPO_ERR_ARG
// sum (op 0) / max (op 2) all-reduce of n floats in place over the communicator, enqueued on s; no-op for a single rank
int comm_allreduce(MagpoComm* c, cudaStream_t s, float* buf, int64_t n, int op);
// true exactly once per (device, id): guards cudaFuncSetAttribute, which is per device
bool once_per_device(int id);
enum { ONCE_GEMM_TC = 0, ONCE_GEMM_TN, ONCE_GRU_FWD, ONCE_GRU_BWD, ONCE_RET_FWD, ONCE_RET_BWD, ONCE_SABLE_STEP_1 /* 8 ids: (A - 1) * 2 + (EPW - 1) */,
       ONCE_SABLE_STEP_LAST = ONCE_SABLE_STEP_1 + 7, ONCE_CHAIN_GATE, ONCE_CHAIN_GATE_FFN, ONCE_CHAIN_GATE_PROJ, ONCE_CHAIN_TAIL, ONCE_CHAIN_FRONT_OBS, ONCE_CHAIN_FRONT_EMB, ONCE_CHAIN_BWD_A, ONCE_CHAIN_BWD_B,
       ONCE_NUM };

constexpr int kNumSMs = 148;
constexpr float kF32Min = -3.4028234663852886e+38f;  // jnp.finfo(float32).min

inline cudaStream_t as_stream(magpo_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }
inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Bump allocator over the caller-provided workspace (256-byte aligned slices).
struct Arena {
  char* base;
  size_t cap, off;
  bool overflow;
  Arena(void* p, size_t bytes) : base(static_cast<char*>(p)), cap(bytes), off(0), overflow(false) {}
  template <typename T>
  T* get(size_t n) {
    size_t bytes = (n * sizeof(T) + 255) & ~size_t(255);
    if (off + bytes > cap) {
      overflow = true;
      off += bytes;
      return nullptr;
    }
    T* r = reinterpret_cast<T*>(base + off);
    off += bytes;
    return r;
  }
};

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
// Sum of NV per-lane values across the warp (NV a power of two): afterwards v[0] of lane l holds the warp total of value
// index l >> (5 - log2 NV). NV - 1 + (5 - log2 NV) shuffles instead of 5 NV.
template <int NV>
__device__ __forceinline__ void warp_reduce_scatter(float (&v)[NV], int lane) {
  int bit = 16;
#pragma unroll
  for (int half = NV / 2; half >= 1; half >>= 1, bit >>= 1) {
    const bool up = lane & bit;
#pragma unroll
    for (int i = 0; i < half; ++i) {
      const float send = up ? v[i] : v[i + half];
      const float keep = up ? v[i + half] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, bit);
    }
  }
  for (; bit >= 1; bit >>= 1) v[0] += __shfl_xor_sync(0xffffffffu, v[0], bit);
}
template <int NV> struct Log2 { static constexpr int v = 1 + Log2<NV / 2>::v; };
template <> struct Log2<1> { static constexpr int v = 0; };
__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + __expf(-x)); }
__device__ __forceinline__ float sigmoid_precise(float x) { return 1.0f / (1.0f + expf(-x)); }
// flax nn.gelu(approximate=True)
__device__ __forceinline__ float gelu_tanh(float x) {
  const float c = 0.7978845608028654f;
  float t = tanhf(c * (x + 0.044715f * x * x * x));
  return 0.5f * x * (1.0f + t);
}
__device__ __forceinline__ float gelu_tanh_grad(float x) {
  const float c = 0.7978845608028654f;
  float x2 = x * x;
  float t = tanhf(c * (x + 0.044715f * x * x2));
  float dt = (1.0f - t * t) * c * (1.0f + 3.0f * 0.044715f * x2);
  return 0.5f * (1.0f + t) + 0.5f * x * dt;
}

}  // namespace magpo
