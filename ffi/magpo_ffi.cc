// XLA FFI handlers for every entry point of libmagpo_b200.so (include/magpo_b200.h): the thin `jax.ffi` custom calls BASELINE.json's
// north_star names as the boundary. One handler per C-ABI function, same order as the header; each one only unpacks buffers and
// attributes and forwards to the C function on XLA's stream — no logic lives here.
//
// Build (on a machine that has jaxlib; its include directory is `jax.ffi.include_dir()`):
//     g++ -std=c++17 -O2 -fPIC -shared -I include -I $(python -c 'import jax.ffi; print(jax.ffi.include_dir())') \
//         -I /usr/local/cuda/include ffi/magpo_ffi.cc -L magpo_b200/lib -lmagpo_b200 -lcudart -o magpo_b200/lib/libmagpo_ffi.so
// Registration (Python, see INTEGRATION.md):
//     lib = ctypes.CDLL("libmagpo_ffi.so")
//     for name in MAGPO_FFI_HANDLERS: jax.ffi.register_ffi_target(name, jax.ffi.pycapsule(getattr(lib, name)), platform="CUDA")
// jaxlib (and with it "xla/ffi/api/ffi.h") is NOT installable in the image this repo is built in, so this translation unit is empty
// there (`__has_include`) and has never been compiled against the real header; tests/test_host_logic.py syntax-checks it against
// the compile-only stand-in tests/mock_xla_ffi/, which validates this file's own code (every magpo_* call's arguments), not the header.
//
// Conventions
//   * Operands / results are passed positionally (ffi::RemainingArgs / RemainingRets) in the order documented above each handler;
//     a struct of device pointers of the C ABI (MagpoTimeStep, Magpo<Env>State, MagpoTrajectory, MagpoMinibatch, ...) is a run of
//     consecutive buffers in the struct's field order.
//   * A buffer the C function updates in place (env state, PRNG key, hidden states, parameters, Adam moments, gradient accumulator)
//     is an operand AND a result, tied with `input_output_aliases` in `jax.ffi.ffi_call`; if XLA hands over two different buffers
//     anyway, the handler copies operand -> result first (`inout`).
//   * Scalar configuration travels as attributes; the POD config structs are rebuilt from them.
//   * Workspaces are extra result buffers sized by the matching magpo_*_workspace_bytes() on the Python side.
//   * The per-device MagpoContext is owned by the shim: one per CUDA device, created on first use.
#if defined(__has_include)
#if __has_include("xla/ffi/api/ffi.h")
#define MAGPO_HAVE_XLA_FFI 1
#endif
#endif

#ifdef MAGPO_HAVE_XLA_FFI
#include <cuda_runtime_api.h>

#include <cstdint>
#include <mutex>
#include <string>

#include "magpo_b200.h"
#include "xla/ffi/api/ffi.h"

namespace ffi = xla::ffi;

namespace {

using Args = ffi::RemainingArgs;
using Rets = ffi::RemainingRets;

ffi::Error status(int rc, const char* what) {
  if (rc == MAGPO_OK) return ffi::Error::Success();
  std::string msg = std::string(what) + ": ";
  switch (rc) {
    case MAGPO_ERR_ARG: msg += "bad argument"; break;
    case MAGPO_ERR_UNSUPPORTED: msg += "unsupported configuration"; break;
    case MAGPO_ERR_WORKSPACE: msg += "workspace too small"; break;
    case MAGPO_ERR_CUDA: msg += std::string("CUDA error: ") + magpo_last_cuda_error(); break;
    default: msg += "error " + std::to_string(rc);
  }
  return rc == MAGPO_ERR_ARG ? ffi::Error::InvalidArgument(msg) : ffi::Error::Internal(msg);
}

// one context per device, owned by the shim
MagpoContext* context() {
  static std::mutex mu;
  static MagpoContext* ctx[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  std::lock_guard<std::mutex> lock(mu);
  if (dev >= 0 && dev < 64 && !ctx[dev]) magpo_context_create(dev, &ctx[dev]);
  return (dev >= 0 && dev < 64) ? ctx[dev] : nullptr;
}

// Reads operands / results by position; remembers the first failure.
struct Unpack {
  const Args& args;
  const Rets& rets;
  cudaStream_t stream;
  size_t ia = 0, ir = 0;
  bool ok = true;
  Unpack(const Args& a, const Rets& r, cudaStream_t s) : args(a), rets(r), stream(s) {}
  template <typename T>
  const T* in() {  // next operand
    auto b = args.get<ffi::AnyBuffer>(ia++);
    if (!b.has_value()) { ok = false; return nullptr; }
    return static_cast<const T*>(b->untyped_data());
  }
  template <typename T>
  T* out(size_t* bytes = nullptr) {  // next result
    auto b = rets.get<ffi::AnyBuffer>(ir++);
    if (!b.has_value()) { ok = false; return nullptr; }
    if (bytes) *bytes = (*b)->size_bytes();
    return static_cast<T*>((*b)->untyped_data());
  }
  template <typename T>
  T* inout() {  // next operand aliased to the next result (copied when XLA did not alias them)
    auto a = args.get<ffi::AnyBuffer>(ia++);
    auto b = rets.get<ffi::AnyBuffer>(ir++);
    if (!a.has_value() || !b.has_value()) { ok = false; return nullptr; }
    void* dst = (*b)->untyped_data();
    if (a->untyped_data() != dst) cudaMemcpyAsync(dst, a->untyped_data(), a->size_bytes(), cudaMemcpyDeviceToDevice, stream);
    return static_cast<T*>(dst);
  }
  // a struct whose fields are all device pointers, from consecutive operands / results / in-out pairs
  template <typename S> void in_struct(S* s, int first = 0, int n = (int)(sizeof(S) / sizeof(void*))) {
    void** f = reinterpret_cast<void**>(s);
    for (int i = first; i < first + n; ++i) f[i] = const_cast<void*>(static_cast<const void*>(in<char>()));
  }
  template <typename S> void out_struct(S* s, int first = 0, int n = (int)(sizeof(S) / sizeof(void*))) {
    void** f = reinterpret_cast<void**>(s);
    for (int i = first; i < first + n; ++i) f[i] = out<char>();
  }
  template <typename S> void inout_struct(S* s, int first = 0, int n = (int)(sizeof(S) / sizeof(void*))) {
    void** f = reinterpret_cast<void**>(s);
    for (int i = first; i < first + n; ++i) f[i] = inout<char>();
  }
  ffi::Error bad() const { return ffi::Error::InvalidArgument("magpo ffi: wrong number of operands / results"); }
};
static_assert(sizeof(MagpoTimeStep) == 11 * sizeof(void*) && sizeof(MagpoCoordSumState) == 9 * sizeof(void*) &&
              sizeof(MagpoLbfState) == 13 * sizeof(void*) && sizeof(MagpoRwareState) == 15 * sizeof(void*) &&
              sizeof(MagpoSableHState) == 3 * sizeof(void*) && sizeof(MagpoTrajectory) == 16 * sizeof(void*),
              "the structs of device pointers are unpacked field by field");

MagpoNetCfg net_cfg(int32_t n_agents, int32_t obs_dim, int32_t action_dim, int32_t embed_dim, int32_t n_head, int32_t n_block,
                    int32_t hidden, int32_t timestep_pe, float decay_scaling_factor, int32_t max_step_count) {
  return MagpoNetCfg{n_agents, obs_dim, action_dim, embed_dim, n_head, n_block, hidden, timestep_pe, decay_scaling_factor, max_step_count};
}
#define NET_ATTR_PARAMS                                                                                                          \
  int32_t n_agents, int32_t obs_dim, int32_t action_dim, int32_t embed_dim, int32_t n_head, int32_t n_block, int32_t hidden,     \
      int32_t timestep_pe, float decay_scaling_factor, int32_t max_step_count
#define NET_ATTR_ARGS n_agents, obs_dim, action_dim, embed_dim, n_head, n_block, hidden, timestep_pe, decay_scaling_factor, max_step_count
#define NET_ATTR_BIND                                                                                                            \
  .Attr<int32_t>("n_agents").Attr<int32_t>("obs_dim").Attr<int32_t>("action_dim").Attr<int32_t>("embed_dim").Attr<int32_t>("n_head") \
      .Attr<int32_t>("n_block").Attr<int32_t>("hidden").Attr<int32_t>("timestep_pe").Attr<float>("decay_scaling_factor")          \
      .Attr<int32_t>("max_step_count")

MagpoSysCfg sys_cfg(int32_t num_envs, int32_t update_batch_size, int32_t rollout_length, int32_t ppo_epochs, int32_t num_minibatches,
                    float gamma, float gae_lambda, float clip_eps, float ent_coef, float vf_coef, float max_grad_norm, float clip_gpo,
                    float alpha, float lr, int32_t sable_only) {
  return MagpoSysCfg{num_envs, update_batch_size, rollout_length, ppo_epochs, num_minibatches, gamma, gae_lambda, clip_eps, ent_coef,
                     vf_coef, max_grad_norm, clip_gpo, alpha, lr, sable_only};
}
#define SYS_ATTR_PARAMS                                                                                                          \
  int32_t num_envs, int32_t update_batch_size, int32_t rollout_length, int32_t ppo_epochs, int32_t num_minibatches, float gamma, \
      float gae_lambda, float clip_eps, float ent_coef, float vf_coef, float max_grad_norm, float clip_gpo, float alpha, float lr, \
      int32_t sable_only
#define SYS_ATTR_ARGS \
  num_envs, update_batch_size, rollout_length, ppo_epochs, num_minibatches, gamma, gae_lambda, clip_eps, ent_coef, vf_coef, max_grad_norm, clip_gpo, alpha, lr, sable_only
#define SYS_ATTR_BIND                                                                                                            \
  .Attr<int32_t>("num_envs").Attr<int32_t>("update_batch_size").Attr<int32_t>("rollout_length").Attr<int32_t>("ppo_epochs")      \
      .Attr<int32_t>("num_minibatches").Attr<float>("gamma").Attr<float>("gae_lambda").Attr<float>("clip_eps").Attr<float>("ent_coef") \
      .Attr<float>("vf_coef").Attr<float>("max_grad_norm").Attr<float>("clip_gpo").Attr<float>("alpha").Attr<float>("lr")          \
      .Attr<int32_t>("sable_only")

#define STREAM_ARGS_RETS .Ctx<ffi::PlatformStream<cudaStream_t>>().RemainingArgs().RemainingRets()

// ------------------------------------------------------------------ PRNG (jax.random call sites rec_magpo.py:135,202,373,439-450,642,660)
// operands: key u32[2]; results: out u32[num,2]
ffi::Error PrngSplit(cudaStream_t s, Args a, Rets r, int32_t num) {
  Unpack u(a, r, s);
  const uint32_t* key = u.in<uint32_t>();
  uint32_t* out = u.out<uint32_t>();
  return u.ok ? status(magpo_prng_split(s, key, num, out), "magpo_prng_split") : u.bad();
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_prng_split, PrngSplit, ffi::Ffi::Bind() STREAM_ARGS_RETS.Attr<int32_t>("num"));

// operands: key; results: out u32[n]
ffi::Error PrngRandomBits(cudaStream_t s, Args a, Rets r, int64_t n) {
  Unpack u(a, r, s);
  const uint32_t* key = u.in<uint32_t>();
  uint32_t* out = u.out<uint32_t>();
  return u.ok ? status(magpo_prng_random_bits(s, key, n, out), "magpo_prng_random_bits") : u.bad();
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_prng_random_bits, PrngRandomBits, ffi::Ffi::Bind() STREAM_ARGS_RETS.Attr<int64_t>("n"));

// operands: key; results: out i32[n]
ffi::Error PrngRandint(cudaStream_t s, Args a, Rets r, int64_t n, int32_t minval, int32_t maxval) {
  Unpack u(a, r, s);
  const uint32_t* key = u.in<uint32_t>();
  int32_t* out = u.out<int32_t>();
  return u.ok ? status(magpo_prng_randint(s, key, n, minval, maxval, out), "magpo_prng_randint") : u.bad();
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_prng_randint, PrngRandint,
                              ffi::Ffi::Bind() STREAM_ARGS_RETS.Attr<int64_t>("n").Attr<int32_t>("minval").Attr<int32_t>("maxval"));

// operands: key; results: out f32[n]
ffi::Error PrngGumbel(cudaStream_t s, Args a, Rets r, int64_t n) {
  Unpack u(a, r, s);
  const uint32_t* key = u.in<uint32_t>();
  float* out = u.out<float>();
  return u.ok ? status(magpo_prng_gumbel(s, key, n, out), "magpo_prng_gumbel") : u.bad();
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_prng_gumbel, PrngGumbel, ffi::Ffi::Bind() STREAM_ARGS_RETS.Attr<int64_t>("n"));

// jax.random.normal / truncated_normal(key, (n,)) — the parameter initialisers' draws. operands: key; results: out f32[n]
ffi::Error PrngNormal(cudaStream_t s, Args a, Rets r, int64_t n) {
  Unpack u(a, r, s);
  const uint32_t* key = u.in<uint32_t>();
  float* out = u.out<float>();
  return u.ok ? status(magpo_prng_normal(s, key, n, out), "magpo_prng_normal") : u.bad();
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_prng_normal, PrngNormal, ffi::Ffi::Bind() STREAM_ARGS_RETS.Attr<int64_t>("n"));
ffi::Error PrngTruncatedNormal(cudaStream_t s, Args a, Rets r, int64_t n, float lower, float upper) {
  Unpack u(a, r, s);
  const uint32_t* key = u.in<uint32_t>();
  float* out = u.out<float>();
  return u.ok ? status(magpo_prng_truncated_normal(s, key, n, lower, upper, out), "magpo_prng_truncated_normal") : u.bad();
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_prng_truncated_normal, PrngTruncatedNormal,
                              ffi::Ffi::Bind() STREAM_ARGS_RETS.Attr<int64_t>("n").Attr<float>("lower").Attr<float>("upper"));

// operands: key; results: out i32[n], scratch u32[2n]
ffi::Error PrngPermutation(cudaStream_t s, Args a, Rets r, int32_t n) {
  Unpack u(a, r, s);
  const uint32_t* key = u.in<uint32_t>();
  int32_t* out = u.out<int32_t>();
  uint32_t* scratch = u.out<uint32_t>();
  return u.ok ? status(magpo_prng_permutation(s, key, n, out, scratch), "magpo_prng_permutation") : u.bad();
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_prng_permutation, PrngPermutation, ffi::Ffi::Bind() STREAM_ARGS_RETS.Attr<int32_t>("n"));

// ------------------------------------------------------------------ environments (vmap(env.reset) rec_magpo.py:645-647, vmap(env.step) :162)
// reset — operands: keys u32[B,2]; results: the 9 / 13 / 15 state arrays, then the 11 MagpoTimeStep arrays
// step  — operands: action i32[B,A], then the state arrays (in-out); results: the state arrays (aliased), then the 11 timestep arrays
ffi::Error CoordSumReset(cudaStream_t s, Args a, Rets r, int32_t B, int32_t num_agents, int32_t num_actions, int32_t time_limit, int32_t maxval) {
  Unpack u(a, r, s);
  const MagpoCoordSumCfg cfg{num_agents, num_actions, time_limit, maxval};
  const uint32_t* keys = u.in<uint32_t>();
  MagpoCoordSumState st; MagpoTimeStep ts;
  u.out_struct(&st); u.out_struct(&ts);
  return u.ok ? status(magpo_coordsum_reset(s, &cfg, B, keys, st, ts), "magpo_coordsum_reset") : u.bad();
}
ffi::Error CoordSumStep(cudaStream_t s, Args a, Rets r, int32_t B, int32_t num_agents, int32_t num_actions, int32_t time_limit, int32_t maxval) {
  Unpack u(a, r, s);
  const MagpoCoordSumCfg cfg{num_agents, num_actions, time_limit, maxval};
  const int32_t* action = u.in<int32_t>();
  MagpoCoordSumState st; MagpoTimeStep ts;
  u.inout_struct(&st); u.out_struct(&ts);
  return u.ok ? status(magpo_coordsum_step(s, &cfg, B, action, st, ts), "magpo_coordsum_step") : u.bad();
}
#define COORDSUM_BIND STREAM_ARGS_RETS.Attr<int32_t>("B").Attr<int32_t>("num_agents").Attr<int32_t>("num_actions").Attr<int32_t>("time_limit").Attr<int32_t>("maxval")
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_coordsum_reset, CoordSumReset, ffi::Ffi::Bind() COORDSUM_BIND);
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_coordsum_step, CoordSumStep, ffi::Ffi::Bind() COORDSUM_BIND);

#define LBF_PARAMS int32_t B, int32_t grid_size, int32_t fov, int32_t num_agents, int32_t num_food, int32_t max_agent_level, int32_t force_coop, int32_t time_limit, int32_t agent_mask_rows
#define LBF_CFG const MagpoLbfCfg cfg{grid_size, fov, num_agents, num_food, max_agent_level, force_coop, time_limit, agent_mask_rows}
ffi::Error LbfReset(cudaStream_t s, Args a, Rets r, LBF_PARAMS) {
  Unpack u(a, r, s);
  LBF_CFG;
  const uint32_t* keys = u.in<uint32_t>();
  MagpoLbfState st; MagpoTimeStep ts;
  u.out_struct(&st); u.out_struct(&ts);
  return u.ok ? status(magpo_lbf_reset(s, &cfg, B, keys, st, ts), "magpo_lbf_reset") : u.bad();
}
ffi::Error LbfStep(cudaStream_t s, Args a, Rets r, LBF_PARAMS) {
  Unpack u(a, r, s);
  LBF_CFG;
  const int32_t* action = u.in<int32_t>();
  MagpoLbfState st; MagpoTimeStep ts;
  u.inout_struct(&st); u.out_struct(&ts);
  return u.ok ? status(magpo_lbf_step(s, &cfg, B, action, st, ts), "magpo_lbf_step") : u.bad();
}
#define LBF_BIND STREAM_ARGS_RETS.Attr<int32_t>("B").Attr<int32_t>("grid_size").Attr<int32_t>("fov").Attr<int32_t>("num_agents").Attr<int32_t>("num_food") \
    .Attr<int32_t>("max_agent_level").Attr<int32_t>("force_coop").Attr<int32_t>("time_limit").Attr<int32_t>("agent_mask_rows")
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_lbf_reset, LbfReset, ffi::Ffi::Bind() LBF_BIND);
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_lbf_step, LbfStep, ffi::Ffi::Bind() LBF_BIND);

#define RWARE_PARAMS int32_t B, int32_t column_height, int32_t shelf_rows, int32_t shelf_columns, int32_t num_agents, int32_t sensor_range, int32_t request_queue_size, int32_t time_limit
#define RWARE_CFG const MagpoRwareCfg cfg{column_height, shelf_rows, shelf_columns, num_agents, sensor_range, request_queue_size, time_limit}
ffi::Error RwareReset(cudaStream_t s, Args a, Rets r, RWARE_PARAMS) {
  Unpack u(a, r, s);
  RWARE_CFG;
  const uint32_t* keys = u.in<uint32_t>();
  MagpoRwareState st; MagpoTimeStep ts;
  u.out_struct(&st); u.out_struct(&ts);
  return u.ok ? status(magpo_rware_reset(s, &cfg, B, keys, st, ts), "magpo_rware_reset") : u.bad();
}
ffi::Error RwareStep(cudaStream_t s, Args a, Rets r, RWARE_PARAMS) {
  Unpack u(a, r, s);
  RWARE_CFG;
  const int32_t* action = u.in<int32_t>();
  MagpoRwareState st; MagpoTimeStep ts;
  u.inout_struct(&st); u.out_struct(&ts);
  return u.ok ? status(magpo_rware_step(s, &cfg, B, action, st, ts), "magpo_rware_step") : u.bad();
}
#define RWARE_BIND STREAM_ARGS_RETS.Attr<int32_t>("B").Attr<int32_t>("column_height").Attr<int32_t>("shelf_rows").Attr<int32_t>("shelf_columns") \
    .Attr<int32_t>("num_agents").Attr<int32_t>("sensor_range").Attr<int32_t>("request_queue_size").Attr<int32_t>("time_limit")
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_rware_reset, RwareReset, ffi::Ffi::Bind() RWARE_BIND);
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_rware_step, RwareStep, ffi::Ffi::Bind() RWARE_BIND);

// ------------------------------------------------------------------ GAE (calculate_gae, utils/multistep.py:24-68)
// operands: reward f32[T,B,A], value f32[T,B,A], done u8[T,B], last_value f32[B,A], last_done u8[B]; results: advantages, targets f32[T,B,A]
ffi::Error Gae(cudaStream_t s, Args a, Rets r, int32_t T, int32_t B, int32_t A, float gamma, float gae_lambda) {
  Unpack u(a, r, s);
  const float* reward = u.in<float>();
  const float* value = u.in<float>();
  const uint8_t* done = u.in<uint8_t>();
  const float* last_value = u.in<float>();
  const uint8_t* last_done = u.in<uint8_t>();
  float* adv = u.out<float>();
  float* tgt = u.out<float>();
  return u.ok ? status(magpo_gae(s, T, B, A, reward, value, done, last_value, last_done, gamma, gae_lambda, adv, tgt), "magpo_gae") : u.bad();
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_gae, Gae,
                              ffi::Ffi::Bind() STREAM_ARGS_RETS.Attr<int32_t>("T").Attr<int32_t>("B").Attr<int32_t>("A").Attr<float>("gamma").Attr<float>("gae_lambda"));

// ------------------------------------------------------------------ rollout (lax.scan(_env_step) + bootstrap value, rec_magpo.py:126-208)
// operands: guider f32[n_g], actor f32[n_a], then in-out: key u32[2], the env state arrays (9 / 13 / 15 by env_kind), hs (3), policy_h,
//           the 4 observation arrays of the trajectory (done, agents_view, action_mask, step_count: slot 0 or T holds the current obs);
// results : the aliased in-outs in the same order, then the 11 timestep arrays, the remaining 12 trajectory arrays (action ... last_value),
//           workspace u8[magpo_rollout_workspace_bytes]
ffi::Error Rollout(cudaStream_t s, Args a, Rets r, NET_ATTR_PARAMS, SYS_ATTR_PARAMS, int32_t env_kind, int32_t e0, int32_t e1, int32_t e2,
                   int32_t e3, int32_t e4, int32_t e5, int32_t e6, int32_t e7, int32_t carry_over) {
  Unpack u(a, r, s);
  const MagpoNetCfg net = net_cfg(NET_ATTR_ARGS);
  const MagpoSysCfg sys = sys_cfg(SYS_ATTR_ARGS);
  const int32_t env_attr[8] = {e0, e1, e2, e3, e4, e5, e6, e7};  // the env config struct's int32 fields in order (unused ones 0)
  const float* guider = u.in<float>();
  const float* actor = u.in<float>();
  uint32_t* key = u.inout<uint32_t>();
  MagpoCoordSumState cs; MagpoLbfState lbf; MagpoRwareState rw;
  void* env_state = nullptr;
  if (env_kind == MAGPO_ENV_COORDSUM) { u.inout_struct(&cs); env_state = &cs; }
  else if (env_kind == MAGPO_ENV_LBF) { u.inout_struct(&lbf); env_state = &lbf; }
  else if (env_kind == MAGPO_ENV_RWARE) { u.inout_struct(&rw); env_state = &rw; }
  else return ffi::Error::InvalidArgument("magpo_ffi_rollout: env_kind");
  MagpoSableHState hs;
  u.inout_struct(&hs);
  float* policy_h = u.inout<float>();
  MagpoTrajectory traj;
  u.inout_struct(&traj, 0, 4);
  MagpoTimeStep ts;
  u.out_struct(&ts);
  u.out_struct(&traj, 4, 12);
  size_t ws_bytes = 0;
  void* ws = u.out<char>(&ws_bytes);
  if (!u.ok) return u.bad();
  return status(magpo_rollout(context(), s, &net, &sys, env_kind, env_attr, env_state, ts, guider, actor, key, hs, policy_h, traj, carry_over,
                              ws, ws_bytes), "magpo_rollout");
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_rollout, Rollout,
                              ffi::Ffi::Bind() STREAM_ARGS_RETS NET_ATTR_BIND SYS_ATTR_BIND.Attr<int32_t>("env_kind").Attr<int32_t>("env_cfg0")
                                  .Attr<int32_t>("env_cfg1").Attr<int32_t>("env_cfg2").Attr<int32_t>("env_cfg3").Attr<int32_t>("env_cfg4")
                                  .Attr<int32_t>("env_cfg5").Attr<int32_t>("env_cfg6").Attr<int32_t>("env_cfg7").Attr<int32_t>("carry_over"));

// SableNetwork.get_actions (sable_network.py:443-482), the `sable_action_select_fn` of rec_magpo.py:139-144.
// operands: guider, agents_view f32[B,A,d], action_mask u8[B,A,a], step_count i32[B,A], prev_done u8[B], sample_keys u32[A,2], hs (3, in-out);
// results : hs (3, aliased), action i32[B,A], log_prob f32[B,A], value f32[B,A], logits f32[B,A,a], workspace
ffi::Error SableGetActions(cudaStream_t s, Args a, Rets r, NET_ATTR_PARAMS, int32_t B, int32_t gumbel_rows) {
  Unpack u(a, r, s);
  const MagpoNetCfg net = net_cfg(NET_ATTR_ARGS);
  const float* guider = u.in<float>();
  const float* view = u.in<float>();
  const uint8_t* mask = u.in<uint8_t>();
  const int32_t* step = u.in<int32_t>();
  const uint8_t* prev_done = u.in<uint8_t>();
  const uint32_t* keys = u.in<uint32_t>();
  MagpoSableHState hs;
  u.inout_struct(&hs);
  int32_t* action = u.out<int32_t>();
  float* log_prob = u.out<float>();
  float* value = u.out<float>();
  float* logits = u.out<float>();
  size_t ws_bytes = 0;
  void* ws = u.out<char>(&ws_bytes);
  if (!u.ok) return u.bad();
  return status(magpo_sable_get_actions(context(), s, &net, B, gumbel_rows, guider, view, mask, step, prev_done, keys, hs, action, log_prob, value,
                                        logits, ws, ws_bytes), "magpo_sable_get_actions");
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_sable_get_actions, SableGetActions,
                              ffi::Ffi::Bind() STREAM_ARGS_RETS NET_ATTR_BIND.Attr<int32_t>("B").Attr<int32_t>("gumbel_rows"));

// RecurrentActor.apply with a length-1 time axis (rec_magpo.py:146-159).
// operands: actor, agents_view f32[B,A,d], done u8[B], policy_h (in-out); results: policy_h (aliased), workspace
ffi::Error ActorStep(cudaStream_t s, Args a, Rets r, NET_ATTR_PARAMS, int32_t B) {
  Unpack u(a, r, s);
  const MagpoNetCfg net = net_cfg(NET_ATTR_ARGS);
  const float* actor = u.in<float>();
  const float* view = u.in<float>();
  const uint8_t* done = u.in<uint8_t>();
  float* policy_h = u.inout<float>();
  size_t ws_bytes = 0;
  void* ws = u.out<char>(&ws_bytes);
  if (!u.ok) return u.bad();
  return status(magpo_actor_step(context(), s, &net, B, actor, view, done, policy_h, ws, ws_bytes), "magpo_actor_step");
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_actor_step, ActorStep, ffi::Ffi::Bind() STREAM_ARGS_RETS NET_ATTR_BIND.Attr<int32_t>("B"));

// ------------------------------------------------------------------ update (rec_magpo.py:214-499)
// _update_epoch's shuffle (:439-451). operands: key u32[2] (in-out), hs_perm i32[E] (in-out);
// results: key, hs_perm (aliased), batch_perm i32[E], agent_perm i32[A], env_index, hs_index, env_slot i32[M*U*N], scratch u32[4+2max(E,A)+E]
ffi::Error EpochIndices(cudaStream_t s, Args a, Rets r, SYS_ATTR_PARAMS, int32_t A, int32_t first_epoch) {
  Unpack u(a, r, s);
  const MagpoSysCfg sys = sys_cfg(SYS_ATTR_ARGS);
  uint32_t* key = u.inout<uint32_t>();
  int32_t* hs_perm = u.inout<int32_t>();
  int32_t* batch_perm = u.out<int32_t>();
  int32_t* agent_perm = u.out<int32_t>();
  int32_t* env_index = u.out<int32_t>();
  int32_t* hs_index = u.out<int32_t>();
  int32_t* env_slot = u.out<int32_t>();
  uint32_t* scratch = u.out<uint32_t>();
  if (!u.ok) return u.bad();
  return status(magpo_epoch_indices(s, &sys, A, key, hs_perm, first_epoch, batch_perm, agent_perm, env_index, hs_index, env_slot, scratch),
                "magpo_epoch_indices");
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_epoch_indices, EpochIndices,
                              ffi::Ffi::Bind() STREAM_ARGS_RETS SYS_ATTR_BIND.Attr<int32_t>("A").Attr<int32_t>("first_epoch"));

// operands: advantages f32[T,B,A], env_index i32[n_env]; results: stats f32[U,2], scratch f64[2U]
ffi::Error AdvStats(cudaStream_t s, Args a, Rets r, int32_t T, int32_t B, int32_t A, int32_t n_env, int32_t U) {
  Unpack u(a, r, s);
  const float* adv = u.in<float>();
  const int32_t* env_index = u.in<int32_t>();
  float* stats = u.out<float>();
  void* scratch = u.out<char>();
  return u.ok ? status(magpo_adv_stats(s, T, B, A, adv, env_index, n_env, U, scratch, stats), "magpo_adv_stats") : u.bad();
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_adv_stats, AdvStats,
                              ffi::Ffi::Bind() STREAM_ARGS_RETS.Attr<int32_t>("T").Attr<int32_t>("B").Attr<int32_t>("A").Attr<int32_t>("n_env").Attr<int32_t>("U"));

// The gather of :445-462. operands: the 16 trajectory arrays, advantages, targets f32[T,B,A], env_index, hs_index i32[n_env], agent_perm i32[A];
// results: the 13 minibatch arrays (agents_view ... policy_h0, sable_h0 x3), time-major [T, n_env, A, ...]
void minibatch_from(Unpack& u, MagpoMinibatch* mb, int32_t T, int32_t N, bool as_results) {
  mb->T = T; mb->N = N;
  const void** f[] = {(const void**)&mb->agents_view, (const void**)&mb->action_mask, (const void**)&mb->step_count, (const void**)&mb->done,
                      (const void**)&mb->action, (const void**)&mb->value, (const void**)&mb->log_prob, (const void**)&mb->advantages,
                      (const void**)&mb->targets, (const void**)&mb->policy_h0, (const void**)&mb->sable_h0.encoder,
                      (const void**)&mb->sable_h0.decoder_self, (const void**)&mb->sable_h0.decoder_cross};
  for (auto p : f) *p = as_results ? static_cast<const void*>(u.out<char>()) : static_cast<const void*>(u.in<char>());
}
ffi::Error PackMinibatch(cudaStream_t s, Args a, Rets r, NET_ATTR_PARAMS, SYS_ATTR_PARAMS, int32_t n_env) {
  Unpack u(a, r, s);
  const MagpoNetCfg net = net_cfg(NET_ATTR_ARGS);
  const MagpoSysCfg sys = sys_cfg(SYS_ATTR_ARGS);
  MagpoTrajectory traj;
  u.in_struct(&traj);
  const float* adv = u.in<float>();
  const float* tgt = u.in<float>();
  const int32_t* env_index = u.in<int32_t>();
  const int32_t* hs_index = u.in<int32_t>();
  const int32_t* agent_perm = u.in<int32_t>();
  MagpoMinibatch mb;
  minibatch_from(u, &mb, rollout_length, n_env, true);
  if (!u.ok) return u.bad();
  return status(magpo_pack_minibatch(s, &net, &sys, traj, adv, tgt, env_index, hs_index, agent_perm, n_env, mb), "magpo_pack_minibatch");
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_pack_minibatch, PackMinibatch, ffi::Ffi::Bind() STREAM_ARGS_RETS NET_ATTR_BIND SYS_ATTR_BIND.Attr<int32_t>("n_env"));

// guider_grad_fn + actor_grad_fn (:222-391). operands: guider, actor, the 13 minibatch arrays, env_slot i32[N], adv_stats f32[U,2], grads (in-out);
// results: grads f32[n_g+n_a+8] (aliased: accumulated into), workspace. reduce_grads: all-reduce over the communicator attached to the shim's
// context (magpo_ffi_comm_attach) — the two lax.pmean(..., "device") of :399-409.
ffi::Error MinibatchGrads(cudaStream_t s, Args a, Rets r, NET_ATTR_PARAMS, SYS_ATTR_PARAMS, int32_t T, int32_t N, float inv_tokens, int32_t reduce_grads) {
  Unpack u(a, r, s);
  const MagpoNetCfg net = net_cfg(NET_ATTR_ARGS);
  const MagpoSysCfg sys = sys_cfg(SYS_ATTR_ARGS);
  const float* guider = u.in<float>();
  const float* actor = u.in<float>();
  MagpoMinibatch mb;
  minibatch_from(u, &mb, T, N, false);
  const int32_t* env_slot = u.in<int32_t>();
  const float* stats = u.in<float>();
  float* grads = u.inout<float>();
  size_t ws_bytes = 0;
  void* ws = u.out<char>(&ws_bytes);
  if (!u.ok) return u.bad();
  return status(magpo_minibatch_grads(context(), s, &net, &sys, guider, actor, mb, env_slot, stats, inv_tokens, grads, reduce_grads, ws, ws_bytes),
                "magpo_minibatch_grads");
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_minibatch_grads, MinibatchGrads,
                              ffi::Ffi::Bind() STREAM_ARGS_RETS NET_ATTR_BIND SYS_ATTR_BIND.Attr<int32_t>("T").Attr<int32_t>("N").Attr<float>("inv_tokens")
                                  .Attr<int32_t>("reduce_grads"));

// SableNetwork.__call__ (`sable_apply_fn`, sable_network.py:412-441). operands: guider, the 13 minibatch arrays; results: value f32[T,N,A],
// logits f32[T,N,A,a] (masked), workspace
ffi::Error GuiderForward(cudaStream_t s, Args a, Rets r, NET_ATTR_PARAMS, int32_t T, int32_t N) {
  Unpack u(a, r, s);
  const MagpoNetCfg net = net_cfg(NET_ATTR_ARGS);
  const float* guider = u.in<float>();
  MagpoMinibatch mb;
  minibatch_from(u, &mb, T, N, false);
  float* value = u.out<float>();
  float* logits = u.out<float>();
  size_t ws_bytes = 0;
  void* ws = u.out<char>(&ws_bytes);
  if (!u.ok) return u.bad();
  return status(magpo_guider_forward(context(), s, &net, guider, mb, value, logits, ws, ws_bytes), "magpo_guider_forward");
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_guider_forward, GuiderForward, ffi::Ffi::Bind() STREAM_ARGS_RETS NET_ATTR_BIND.Attr<int32_t>("T").Attr<int32_t>("N"));

// RecurrentActor.apply over T steps (`actor_apply_fn`, rec_magpo.py:243-250). operands: actor, the 13 minibatch arrays; results: logits, workspace
ffi::Error ActorForward(cudaStream_t s, Args a, Rets r, NET_ATTR_PARAMS, int32_t T, int32_t N) {
  Unpack u(a, r, s);
  const MagpoNetCfg net = net_cfg(NET_ATTR_ARGS);
  const float* actor = u.in<float>();
  MagpoMinibatch mb;
  minibatch_from(u, &mb, T, N, false);
  float* logits = u.out<float>();
  size_t ws_bytes = 0;
  void* ws = u.out<char>(&ws_bytes);
  if (!u.ok) return u.bad();
  return status(magpo_actor_forward(context(), s, &net, actor, mb, logits, ws, ws_bytes), "magpo_actor_forward");
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_actor_forward, ActorForward, ffi::Ffi::Bind() STREAM_ARGS_RETS NET_ATTR_BIND.Attr<int32_t>("T").Attr<int32_t>("N"));

// optax.chain(clip_by_global_norm, adam) + apply_updates (:581-589,412-423), with make_learning_rate's schedule when decay_period > 0.
// operands: grads f32[n], then in-out: params, mu, nu f32[n], count i32[]; results: params, mu, nu, count (aliased), scratch f32[1024]
ffi::Error ClipAdam(cudaStream_t s, Args a, Rets r, int64_t n, float grad_scale, float lr, int32_t decay_period, int32_t num_updates, float max_norm) {
  Unpack u(a, r, s);
  const float* grads = u.in<float>();
  float* params = u.inout<float>();
  float* mu = u.inout<float>();
  float* nu = u.inout<float>();
  int32_t* count = u.inout<int32_t>();
  float* scratch = u.out<float>();
  if (!u.ok) return u.bad();
  return status(magpo_clip_adam_sched(s, n, params, grads, mu, nu, count, grad_scale, lr, decay_period, num_updates, max_norm, scratch), "magpo_clip_adam");
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_clip_adam, ClipAdam,
                              ffi::Ffi::Bind() STREAM_ARGS_RETS.Attr<int64_t>("n").Attr<float>("grad_scale").Attr<float>("lr").Attr<int32_t>("decay_period")
                                  .Attr<int32_t>("num_updates").Attr<float>("max_norm"));

// ------------------------------------------------------------------ rec_ippo (mava/systems/ppo/anakin/rec_ippo.py)
// The workspaces are result buffers sized on the Python side by calling the entry point itself with workspace == NULL.
// Rollout. operands: actor f32[n_a], critic f32[n_c], then in-out: key u32[2], the env state arrays, policy_h, critic_h f32[B,A,H], the 4
// observation arrays of the trajectory; results: the aliased in-outs in the same order, the 11 timestep arrays, the remaining 12 trajectory
// arrays (action ... last_value; sable_h0 x3 are 1-element placeholders), critic_h0 f32[B,A,H], workspace
ffi::Error IppoRollout(cudaStream_t s, Args a, Rets r, NET_ATTR_PARAMS, SYS_ATTR_PARAMS, int32_t env_kind, int32_t e0, int32_t e1, int32_t e2,
                       int32_t e3, int32_t e4, int32_t e5, int32_t e6, int32_t e7, int32_t carry_over) {
  Unpack u(a, r, s);
  const MagpoNetCfg net = net_cfg(NET_ATTR_ARGS);
  const MagpoSysCfg sys = sys_cfg(SYS_ATTR_ARGS);
  const int32_t env_attr[8] = {e0, e1, e2, e3, e4, e5, e6, e7};
  const float* actor = u.in<float>();
  const float* critic = u.in<float>();
  uint32_t* key = u.inout<uint32_t>();
  MagpoCoordSumState cs; MagpoLbfState lbf; MagpoRwareState rw;
  void* env_state = nullptr;
  if (env_kind == MAGPO_ENV_COORDSUM) { u.inout_struct(&cs); env_state = &cs; }
  else if (env_kind == MAGPO_ENV_LBF) { u.inout_struct(&lbf); env_state = &lbf; }
  else if (env_kind == MAGPO_ENV_RWARE) { u.inout_struct(&rw); env_state = &rw; }
  else return ffi::Error::InvalidArgument("magpo_ffi_ippo_rollout: env_kind");
  float* policy_h = u.inout<float>();
  float* critic_h = u.inout<float>();
  MagpoTrajectory traj;
  u.inout_struct(&traj, 0, 4);
  MagpoTimeStep ts;
  u.out_struct(&ts);
  u.out_struct(&traj, 4, 12);
  float* critic_h0 = u.out<float>();
  size_t ws_bytes = 0;
  void* ws = u.out<char>(&ws_bytes);
  if (!u.ok) return u.bad();
  return status(magpo_ippo_rollout(context(), s, &net, &sys, env_kind, env_attr, env_state, ts, actor, critic, key, policy_h, critic_h, traj,
                                   critic_h0, carry_over, ws, &ws_bytes), "magpo_ippo_rollout");
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_ippo_rollout, IppoRollout,
                              ffi::Ffi::Bind() STREAM_ARGS_RETS NET_ATTR_BIND SYS_ATTR_BIND.Attr<int32_t>("env_kind").Attr<int32_t>("env_cfg0")
                                  .Attr<int32_t>("env_cfg1").Attr<int32_t>("env_cfg2").Attr<int32_t>("env_cfg3").Attr<int32_t>("env_cfg4")
                                  .Attr<int32_t>("env_cfg5").Attr<int32_t>("env_cfg6").Attr<int32_t>("env_cfg7").Attr<int32_t>("carry_over"));

// Epoch shuffle. operands: key u32[2] (in-out); results: key (aliased), perm i32[E], env_index, env_slot i32[M*U*N], workspace
ffi::Error IppoEpochIndices(cudaStream_t s, Args a, Rets r, SYS_ATTR_PARAMS) {
  Unpack u(a, r, s);
  const MagpoSysCfg sys = sys_cfg(SYS_ATTR_ARGS);
  uint32_t* key = u.inout<uint32_t>();
  int32_t* perm = u.out<int32_t>();
  int32_t* env_index = u.out<int32_t>();
  int32_t* env_slot = u.out<int32_t>();
  size_t ws_bytes = 0;
  void* ws = u.out<char>(&ws_bytes);
  if (!u.ok) return u.bad();
  return status(magpo_ippo_epoch_indices(s, &sys, key, perm, env_index, env_slot, ws, &ws_bytes), "magpo_ippo_epoch_indices");
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_ippo_epoch_indices, IppoEpochIndices, ffi::Ffi::Bind() STREAM_ARGS_RETS SYS_ATTR_BIND);

// Gather. operands: the 16 trajectory arrays, critic_h0 f32[B,A,H], advantages, targets f32[T,B,A], env_index i32[n_env];
// results: the 13 minibatch arrays (sable_h0 x3 are placeholders), critic_h0 f32[n_env,A,H]
ffi::Error IppoPackMinibatch(cudaStream_t s, Args a, Rets r, NET_ATTR_PARAMS, SYS_ATTR_PARAMS, int32_t n_env) {
  Unpack u(a, r, s);
  const MagpoNetCfg net = net_cfg(NET_ATTR_ARGS);
  const MagpoSysCfg sys = sys_cfg(SYS_ATTR_ARGS);
  MagpoTrajectory traj;
  u.in_struct(&traj);
  const float* critic_h0 = u.in<float>();
  const float* adv = u.in<float>();
  const float* tgt = u.in<float>();
  const int32_t* env_index = u.in<int32_t>();
  MagpoMinibatch mb;
  minibatch_from(u, &mb, rollout_length, n_env, true);
  float* out_critic_h0 = u.out<float>();
  if (!u.ok) return u.bad();
  return status(magpo_ippo_pack_minibatch(s, &net, &sys, traj, critic_h0, adv, tgt, env_index, n_env, mb, out_critic_h0),
                "magpo_ippo_pack_minibatch");
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_ippo_pack_minibatch, IppoPackMinibatch,
                              ffi::Ffi::Bind() STREAM_ARGS_RETS NET_ATTR_BIND SYS_ATTR_BIND.Attr<int32_t>("n_env"));

// actor_grad_fn + critic_grad_fn. operands: actor, critic, the 13 minibatch arrays, critic_h0 f32[N,A,H], env_slot i32[N], adv_stats f32[U,2],
// grads (in-out); results: grads f32[n_a+n_c+8] (aliased: accumulated into), workspace
ffi::Error IppoMinibatchGrads(cudaStream_t s, Args a, Rets r, NET_ATTR_PARAMS, SYS_ATTR_PARAMS, int32_t T, int32_t N, float inv_tokens,
                              int32_t reduce_grads) {
  Unpack u(a, r, s);
  const MagpoNetCfg net = net_cfg(NET_ATTR_ARGS);
  const MagpoSysCfg sys = sys_cfg(SYS_ATTR_ARGS);
  const float* actor = u.in<float>();
  const float* critic = u.in<float>();
  MagpoMinibatch mb;
  minibatch_from(u, &mb, T, N, false);
  const float* critic_h0 = u.in<float>();
  const int32_t* env_slot = u.in<int32_t>();
  const float* stats = u.in<float>();
  float* grads = u.inout<float>();
  size_t ws_bytes = 0;
  void* ws = u.out<char>(&ws_bytes);
  if (!u.ok) return u.bad();
  return status(magpo_ippo_minibatch_grads(context(), s, &net, &sys, actor, critic, mb, critic_h0, env_slot, stats, inv_tokens, grads,
                                           reduce_grads, ws, &ws_bytes), "magpo_ippo_minibatch_grads");
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_ippo_minibatch_grads, IppoMinibatchGrads,
                              ffi::Ffi::Bind() STREAM_ARGS_RETS NET_ATTR_BIND SYS_ATTR_BIND.Attr<int32_t>("T").Attr<int32_t>("N").Attr<float>("inv_tokens")
                                  .Attr<int32_t>("reduce_grads"));

// ------------------------------------------------------------------ data-parallel exchange (lax.pmean(..., "device"), :399-409)
// The communicator is created on the host (magpo_ffi_comm_attach below) once per process; this handler sums a buffer over the ranks.
// operands: buf f32[n] (in-out); results: buf (aliased)
MagpoComm* g_comm_for_handlers = nullptr;  // set by magpo_ffi_comm_attach (host side, before tracing); one process = one rank
ffi::Error CommAllreduceSum(cudaStream_t s, Args a, Rets r, int64_t n) {
  Unpack u(a, r, s);
  float* buf = u.inout<float>();
  if (!u.ok) return u.bad();
  return status(magpo_comm_allreduce_sum(g_comm_for_handlers, s, buf, n), "magpo_comm_allreduce_sum");
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(magpo_ffi_comm_allreduce_sum, CommAllreduceSum, ffi::Ffi::Bind() STREAM_ARGS_RETS.Attr<int64_t>("n"));

}  // namespace

// Host-side helpers of the shim (plain C, called through ctypes before tracing — not FFI handlers): create this rank's communicator
// from the 128-byte id and attach it to the shim's context so that magpo_ffi_minibatch_grads(reduce_grads=1) and
// magpo_ffi_comm_allreduce_sum use it. magpo_param_count / magpo_param_tensor / magpo_*_workspace_bytes / magpo_rware_num_shelves /
// magpo_comm_unique_id are host-only queries too and are called directly from Python.
extern "C" int magpo_ffi_comm_attach(int32_t nranks, int32_t rank, const void* id128) {
  MagpoComm* c = nullptr;
  const int rc = magpo_comm_init(nranks, rank, id128, &c);
  if (rc != MAGPO_OK) return rc;
  g_comm_for_handlers = c;
  return magpo_context_set_comm(context(), c);
}

#endif  // MAGPO_HAVE_XLA_FFI
