// C ABI of the B200-native Go2 policy hot path (declared in include/go2policy.h).
// Host side: parse the .onnx once, upload the weights in the layouts the kernels read, own the
// mailbox / streams / scratch, launch the sm_100a kernels.  No CPU compute path exists here.
#include "../../include/go2policy.h"

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <array>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <stdexcept>
#include <thread>
#include <string>
#include <utility>
#include <vector>
#if defined(__x86_64__)
#include <immintrin.h>
#endif

#include "kernels_b1.cuh"
#include "kernels_fp32.cuh"
#include "kernels_tc.cuh"
#include "kernels_wide.cuh"
#include "kernels_pack.cuh"   // after the step-path kernels: their instantiation order (and SASS) stays as it was
#include "onnx_reader.hpp"

using namespace go2p;

static_assert(sizeof(go2p_raw_state) == sizeof(RawStateDev), "raw state layout");
static_assert(sizeof(go2p_motor_cmd) == sizeof(MotorCmdDev), "motor command layout");

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

#define CU_TRY(expr)                                                                              \
  do {                                                                                            \
    cudaError_t e__ = (expr);                                                                     \
    if (e__ != cudaSuccess)                                                                       \
      return fail(GO2P_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__));            \
  } while (0)

inline void cpu_relax() {
#if defined(__x86_64__)
  _mm_pause();
#endif
}

constexpr int64_t kFp32ChunkRows = 131072;
constexpr int64_t kHostChunkRows = 65536;
constexpr int kPipeDepth = 3;

}  // namespace

struct go2p_handle {
  go2p_config cfg{};
  MlpModel model;
  int device = 0, sm_count = 0, cc_major = 0, cc_minor = 0;
  std::vector<void*> dev_owned;                // every device buffer of the handle (owned_alloc), freed by go2p_destroy
  DevModel dm{};
  CtrlConst cc{};
  // tensor-core path
  bool tc_ok = false;
  bool wide_ok = false;                        // bf16 / fp16 on the per-layer GEMMs
  bool split_ok = false;                       // GO2P_PREC_FP32_TC on the per-layer GEMMs (wide.L[l].w3)
  uint16_t* d_wpack[2] = {nullptr, nullptr};   // [0] bf16, [1] fp16
  int k0p = 0;
  size_t tc_off[kMaxLayers] = {};              // layer l's image starts tc_off[l] elements into d_wpack[0] / [1]
  int tc_kp[kMaxLayers] = {};
  double tc_wscale[kMaxLayers] = {}, tc_bscale[kMaxLayers] = {};   // the scales pack_umma_kmajor applied
  std::vector<std::pair<const void*, size_t>> smem_opt_in;   // (kernel, dynamic shared memory it is opted in to): opt_in_smem
  WideModel wide{};
  // activation ping-pong buffers between the per-layer launches of the fp32 path and of the wide path, one pair per
  // stream set: set 0 serves the device-pointer API, sets 1..kPipeDepth the streams of the host-buffer pipeline (which
  // run concurrently)
  struct Scratch { void* buf[2] = {nullptr, nullptr}; int64_t rows = 0; };
  Scratch fp32_scratch[1 + kPipeDepth], wide_scratch[1 + kPipeDepth], split_scratch[1 + kPipeDepth];
  // batch-1
  B1State* d_state = nullptr;
  int32_t* d_step_button = nullptr;   // go2p_step_batch: dead-man buttons extracted by the assembly kernel
  int64_t step_button_rows = 0;
  MailWord* inbox = nullptr;    // host-mapped
  MailWord* outbox = nullptr;   // host-mapped
  int n_in_slots = 0;
  uint32_t seq = 0;
  uint32_t epoch = 0;           // launch counter of the resident kernel (farewell word carries it)
  bool resident = false;
  cudaStream_t b1_stream = nullptr;
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t graph_exec = nullptr;
  size_t b1_smem = 0;
  bool b1_weights_in_smem = false;
  float* bound_obs = nullptr;
  float* bound_act = nullptr;
  size_t n_bound_obs = 0, n_bound_act = 0;
  go2p_b1_stats stats{0, ~0ull, 0, 0};
  // host pipeline
  cudaStream_t pipe_stream[kPipeDepth] = {};
  float* pipe_in[kPipeDepth] = {};
  float* pipe_out[kPipeDepth] = {};
  int last_launches = 0;
  unsigned long long* d_sat = nullptr;         // GO2P_F_SAT_COUNT: saturated fp16 operand blocks since the last read
  // go2p_set_weights: w_gen counts updates; tc_w_gen is the update the first tensor-core launch on w_stream (the
  // stream of the last update) has seen.  w_event marks the end of the last update's packer.
  uint64_t w_gen = 0, tc_w_gen = 0;
  cudaStream_t w_stream = nullptr;
  cudaEvent_t w_event = nullptr;
  float* w_fold = nullptr;                     // layer 0 with the observation normaliser folded in
  float* w_stage = nullptr;                    // go2p_set_weights_host: the caller's tensors on the device
  // ObservationAction ring (go2p_log_enable)
  LogRing* d_log = nullptr;
  uint32_t log_capacity = 0;
  uint64_t log_tail = 0;
  // go2p_step_batch_host: per-robot state resident on the device + staging of the raw states / commands
  struct Fleet {
    int64_t robots = 0;
    float* obs = nullptr; float* vel = nullptr; float* act = nullptr;
    go2p_raw_state* raw[kPipeDepth] = {};
    MotorCmdDev* cmd[kPipeDepth] = {};
    int32_t* button[kPipeDepth] = {};
    uint8_t* reset[kPipeDepth] = {};    // go2p_step_batch_host_ex: the chunk's reset flags
  } fleet;
};

namespace {

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    int cur = -1;
    cudaGetDevice(&cur);
    if (prev >= 0 && cur != prev) cudaSetDevice(prev);
  }
};

// Device memory of the handle.  owned_alloc gives p `bytes` of device memory unless p is already set, and records the
// buffer in dev_owned, which go2p_destroy frees.  To retire an outgrown buffer, clear its member; do not free it:
// cudaFree synchronises the device and would never return while the resident batch-1 kernel runs, and kernels of other
// streams may still read the buffer.  owned_free frees a buffer at once, where no kernel can still use it.
template <class T>
int owned_alloc(go2p_handle* h, T*& p, size_t bytes) {
  if (p) return GO2P_OK;
  void* d = nullptr;
  CU_TRY(cudaMalloc(&d, bytes));
  h->dev_owned.push_back(d);
  p = static_cast<T*>(d);
  return GO2P_OK;
}

void owned_free(go2p_handle* h, void* p) {
  if (!p) return;
  h->dev_owned.erase(std::remove(h->dev_owned.begin(), h->dev_owned.end(), p), h->dev_owned.end());
  cudaFree(p);
}

template <class T>
int dev_upload(go2p_handle* h, const std::vector<T>& v, T** out) {
  T* p = nullptr;
  if (const int rc = owned_alloc(h, p, std::max<size_t>(v.size() * sizeof(T), 16))) return rc;
  CU_TRY(cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  *out = p;
  return GO2P_OK;
}

// Opts kernel fn in to `bytes` of dynamic shared memory.  The opt-in is a per-device function attribute, so the handle
// (bound to one device) remembers it and sets the attribute only when the size it needs changes.
cudaError_t opt_in_smem(go2p_handle* h, const void* fn, size_t bytes) {
  auto it = std::find_if(h->smem_opt_in.begin(), h->smem_opt_in.end(), [fn](const auto& r) { return r.first == fn; });
  if (it != h->smem_opt_in.end() && it->second == bytes) return cudaSuccess;
  const cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) return e;
  if (it != h->smem_opt_in.end()) it->second = bytes;
  else h->smem_opt_in.emplace_back(fn, bytes);
  return cudaSuccess;
}

inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

uint16_t to_bf16(float f) { return __bfloat16_as_ushort(__float2bfloat16_rn(f)); }
uint16_t to_f16(float f) {
  f = std::min(65504.f, std::max(-65504.f, f));
  return __half_as_ushort(__float2half_rn(f));
}

float from_bf16(uint16_t b) { return __bfloat162float(__ushort_as_bfloat16(b)); }
float from_f16(uint16_t b) { return __half2float(__ushort_as_half(b)); }

// 16-bit K-major UMMA "interleaved" (no swizzle) layout: 8x8-element core matrices of 128 contiguous
// bytes, K-adjacent cores contiguous (LBO = 128 B), 8-row groups Kp*16 B apart (SBO).
// Element (n,k): k < L.in -> weight * wscale; k == L.in / L.in+1 -> hi / lo 16-bit halves of bias * bscale (the A
// operand carries constant ones in those two columns); everything else zero.
void pack_umma_kmajor(const MlpLayer& L, int Np, int Kp, bool fp16, double wscale, double bscale, std::vector<uint16_t>& out) {
  const size_t base = out.size();
  out.resize(base + (size_t)Np * Kp, 0);
  auto enc = [&](float v) { return fp16 ? to_f16(v) : to_bf16(v); };
  auto dec = [&](uint16_t b) { return fp16 ? from_f16(b) : from_bf16(b); };
  for (int n = 0; n < Np; ++n)
    for (int k = 0; k < Kp; ++k) {
      uint16_t bits = 0;
      if (n < L.out) {
        if (k < L.in) bits = enc((float)((double)L.weight[(size_t)n * L.in + k] * wscale));
        else if (k == L.in || k == L.in + 1) {
          const float b = (float)((double)L.bias[n] * bscale);
          const uint16_t hi = enc(b);
          bits = (k == L.in) ? hi : enc(b - dec(hi));
        }
      }
      const size_t idx = ((size_t)(n / 8) * (Kp / 8) + (k / 8)) * 64 + (n % 8) * 8 + (k % 8);
      out[base + idx] = bits;
    }
}

int upload_model(go2p_handle* h) {
  const MlpModel& m = h->model;
  DevModel& dm = h->dm;
  dm.n_layers = (int)m.layers.size();
  dm.in_dim = m.in_dim();
  dm.out_dim = m.out_dim();
  dm.max_width = dm.in_dim;
  for (int l = 0; l < dm.n_layers; ++l) {
    const MlpLayer& L = m.layers[l];
    DevLayer& D = dm.L[l];
    D.K = L.in; D.N = L.out;
    D.Kp = round_up(L.in, 4);
    D.Kp8 = round_up(L.in, 8);
    D.Np = round_up(L.out, 128);
    D.has_elu = L.has_elu ? 1 : 0;
    D.alpha = L.elu_alpha;
    dm.max_width = std::max(dm.max_width, L.out);
    std::vector<float> rm((size_t)D.N * D.Kp, 0.f), k4((size_t)D.Kp * D.N, 0.f), kn((size_t)D.Kp8 * D.Np, 0.f), bias(D.Np, 0.f);
    for (int o = 0; o < D.N; ++o)
      for (int k = 0; k < D.K; ++k) {
        const float v = L.weight[(size_t)o * L.in + k];
        rm[(size_t)o * D.Kp + k] = v;
        k4[((size_t)(k / 4) * D.N + o) * 4 + (k % 4)] = v;
        kn[(size_t)k * D.Np + o] = v;
      }
    for (int o = 0; o < D.N; ++o) bias[o] = L.bias[o];
    float *drm, *dk4, *dkn, *db;
    int rc;
    if ((rc = dev_upload(h, rm, &drm)) || (rc = dev_upload(h, k4, &dk4)) || (rc = dev_upload(h, kn, &dkn)) ||
        (rc = dev_upload(h, bias, &db)))
      return rc;
    D.w_rm = drm; D.w_k4 = dk4; D.w_kn = dkn; D.bias = db;
  }
  // controller constants
  for (int i = 0; i < kDof; ++i) h->cc.q0[i] = h->cfg.q0[i];
  h->cc.action_scale = h->cfg.action_scale;
  h->cc.action_limit = h->cfg.action_limit;
  h->cc.kp_deadman = h->cfg.kp_deadman;
  h->cc.foot_threshold = h->cfg.foot_threshold;
  h->cc.H = h->cfg.history;
  h->cc.kp = h->cfg.kp;
  h->cc.kd = h->cfg.kd;

  // ---- tensor-core packing (narrow family: every hidden width 128, in + 2 <= 128, out <= 16: the layer-0 operand
  // with its two constant-one columns has to fit the 64 packed columns of a TMEM buffer; wider inputs take the
  // per-layer GEMM path).  The chain runs
  // in the base-2 exponent domain (kernels_tc.cuh): an ELU layer's pre-activation and output are scaled by log2(e),
  // the next layer's weights carry the inverse factor; biases ride in two extra K rows (hi/lo).
  bool narrow = dm.n_layers >= 2 && dm.in_dim + 2 <= kTcHidden && dm.out_dim <= kTcOutPad;
  for (int l = 0; l + 1 < dm.n_layers; ++l) narrow = narrow && (m.layers[l].out == kTcHidden);
  if (narrow) {
    h->k0p = round_up(dm.in_dim + 2, 16);
    const double kLog2e = 1.4426950408889634074;
    std::vector<uint16_t> wb, wf;
    double in_scale = 1.0;
    for (int l = 0; l < dm.n_layers; ++l) {
      const int Kp = l == 0 ? h->k0p : kTcHidden + kTcBiasK;
      const int Np = l == dm.n_layers - 1 ? kTcOutPad : kTcHidden;
      const double out_scale = m.layers[l].has_elu ? kLog2e : 1.0;
      h->tc_off[l] = wb.size(); h->tc_kp[l] = Kp;
      h->tc_wscale[l] = out_scale / in_scale; h->tc_bscale[l] = out_scale;
      pack_umma_kmajor(m.layers[l], Np, Kp, false, out_scale / in_scale, out_scale, wb);
      pack_umma_kmajor(m.layers[l], Np, Kp, true, out_scale / in_scale, out_scale, wf);
      in_scale = out_scale;
    }
    TcArgs probe{};
    probe.n_layers = dm.n_layers; probe.in_dim = dm.in_dim; probe.k0p = h->k0p;
    if (tc_smem_bytes(probe) <= 227 * 1024) {
      int rc;
      if ((rc = dev_upload(h, wb, &h->d_wpack[0])) || (rc = dev_upload(h, wf, &h->d_wpack[1]))) return rc;
      h->tc_ok = true;
    }
  }
  // the per-layer GEMMs: bf16 / fp16 for the shapes the one-launch kernel does not serve, GO2P_PREC_FP32_TC for every
  // shape they serve
  auto alloc = [h](size_t bytes) { void* p = nullptr; return owned_alloc(h, p, bytes) ? nullptr : p; };
  int rc = wide_prepare(m, alloc, &h->wide, !h->tc_ok, g_err);
  if (rc == 0) { h->wide_ok = !h->tc_ok; h->split_ok = true; }
  else if (rc > 0) return rc;     // CUDA failure; rc < 0 means "shape not served"
  return GO2P_OK;
}

// the Go2 topology keeps its weights in registers (kernels_b1.cuh: B1RegWeights)
bool b1_regs_ok(const go2p_handle* h) { return B1RegWeights::supported(h->dm); }

size_t b1_smem_bytes(const go2p_handle* h, bool resident, bool* weights_fit) {
  const int XW = b1_xw(std::max(h->dm.max_width, h->n_in_slots));
  size_t bytes = (size_t)(2 * XW + kB1Threads + 64) * 4;
  *weights_fit = false;
  if (resident && b1_regs_ok(h)) return bytes + sizeof(B1State) + 4 * 128 * 4;
  if (resident) {
    bytes += sizeof(B1State);
    size_t w = 0;
    for (int l = 0; l < h->dm.n_layers; ++l) w += (size_t)h->dm.L[l].Kp * h->dm.L[l].N + round_up(h->dm.L[l].N, 4);
    if (bytes + w * 4 <= 226 * 1024) { bytes += w * 4; *weights_fit = true; }   // 1 KB left for static shared memory
  }
  return bytes;
}

B1Args make_b1_args(const go2p_handle* h, bool weights_in_smem) {
  B1Args a{};
  a.model = h->dm;
  a.model.max_width = std::max(h->dm.max_width, h->n_in_slots);
  a.cc = h->cc;
  a.gstate = h->d_state;
  a.inbox = h->inbox;
  a.outbox = h->outbox;
  a.n_in_slots = h->n_in_slots;
  a.weights_in_smem = weights_in_smem ? 1 : 0;
  a.idle_ns = (unsigned long long)std::max(0, h->cfg.idle_exit_ms) * 1000000ull;
  a.epoch = h->epoch;
  a.log = h->d_log;
  return a;
}

// one raw state as the kRawWords words of a MSG_STEP message (and of b1_selfdriven_kernel's input)
void raw_to_words(const go2p_raw_state& r, uint32_t* w) {
  std::memcpy(&w[0], r.quat, 16);
  std::memcpy(&w[4], r.gyro, 12);
  std::memcpy(&w[7], r.q, 48);
  std::memcpy(&w[19], r.dq, 48);
  std::memcpy(&w[31], r.axes, 16);
  for (int i = 0; i < 4; ++i) w[35 + i] = (uint32_t)(int32_t)r.foot_force[i];
  w[39] = (uint32_t)(r.joy_valid != 0);
  w[40] = (uint32_t)r.button0;
}

void mail_send(go2p_handle* h, uint32_t type, const uint32_t* words, int n, uint32_t* tag_out) {
  const uint32_t seq = ++h->seq;
  const uint32_t tag = make_tag(seq, type);
  volatile uint64_t* slots = reinterpret_cast<volatile uint64_t*>(h->inbox);
  for (int i = 0; i < h->n_in_slots; ++i) slots[i] = ((uint64_t)tag << 32) | (uint64_t)(i < n ? words[i] : 0u);
  *tag_out = tag;
}

bool resident_said_goodbye(const go2p_handle* h) {
  const volatile uint64_t* slots = reinterpret_cast<const volatile uint64_t*>(h->outbox);
  return slots[kByeSlot] == (((uint64_t)kByeTag << 32) | (uint64_t)h->epoch);
}

int mail_wait(go2p_handle* h, uint32_t tag, int n_words) {
  const volatile uint64_t* slots = reinterpret_cast<const volatile uint64_t*>(h->outbox);
  const auto t0 = std::chrono::steady_clock::now();
  uint64_t spins = 0;
  for (int i = n_words - 1; i >= 0; --i) {
    while ((uint32_t)(slots[i] >> 32) != tag) {
      cpu_relax();
      if ((++spins & 0xFF) == 0 && h->resident && resident_said_goodbye(h)) {
        // the kernel timed out idle while this request was in flight: relaunch, it will pick the request up
        h->resident = false;
        int rc = go2p_persistent_start(h);
        if (rc) return rc;
      }
      if ((spins & 0xFFFF) == 0) {
        const auto dt = std::chrono::duration_cast<std::chrono::milliseconds>(std::chrono::steady_clock::now() - t0).count();
        if (dt > h->cfg.timeout_ms) {
          cudaError_t e = cudaPeekAtLastError();
          if (e == cudaSuccess && h->b1_stream) e = cudaStreamQuery(h->b1_stream);
          return fail(GO2P_ERR_TIMEOUT, std::string("batch-1 kernel did not answer within timeout (cuda: ") +
                                            cudaGetErrorString(e == cudaErrorNotReady ? cudaSuccess : e) + ")");
        }
      }
    }
  }
  std::atomic_thread_fence(std::memory_order_acquire);   // payload reads below stay after the tag polls
  return GO2P_OK;
}

int b1_dispatch(go2p_handle* h) {
  // called after mail_send: make sure some kernel will consume the message
  if (h->cfg.b1_mode == GO2P_B1_PERSISTENT) {
    if (h->resident && resident_said_goodbye(h)) h->resident = false;
    if (!h->resident) return go2p_persistent_start(h);
    return GO2P_OK;
  }
  if (h->cfg.b1_mode == GO2P_B1_GRAPH) {
    if (!h->graph_exec) {
      bool fit;
      const size_t smem = b1_smem_bytes(h, false, &fit);
      CU_TRY(opt_in_smem(h, reinterpret_cast<const void*>(b1_kernel<false>), smem));
      B1Args a = make_b1_args(h, false);
      CU_TRY(cudaStreamBeginCapture(h->b1_stream, cudaStreamCaptureModeThreadLocal));
      b1_kernel<false><<<1, kB1Threads, smem, h->b1_stream>>>(a);
      CU_TRY(cudaStreamEndCapture(h->b1_stream, &h->graph));
      CU_TRY(cudaGraphInstantiate(&h->graph_exec, h->graph, 0));
    }
    CU_TRY(cudaGraphLaunch(h->graph_exec, h->b1_stream));
    return GO2P_OK;
  }
  bool fit;
  const size_t smem = b1_smem_bytes(h, false, &fit);
  CU_TRY(opt_in_smem(h, reinterpret_cast<const void*>(b1_kernel<false>), smem));
  B1Args a = make_b1_args(h, false);
  b1_kernel<false><<<1, kB1Threads, smem, h->b1_stream>>>(a);
  CU_TRY(cudaGetLastError());
  return GO2P_OK;
}

void stats_add(go2p_handle* h, uint64_t ns) {
  h->stats.steps++;
  h->stats.device_ns_sum += ns;
  h->stats.device_ns_min = std::min(h->stats.device_ns_min, ns);
  h->stats.device_ns_max = std::max(h->stats.device_ns_max, ns);
}

int simple_message(go2p_handle* h, uint32_t type, const uint32_t* words, int n) {
  DeviceGuard g(h->device);
  uint32_t tag;
  mail_send(h, type, words, n, &tag);
  int rc = b1_dispatch(h);
  if (rc) return rc;
  return mail_wait(h, tag, 1);
}

// grows both buffers of sc to `rows` rows of `row_bytes`; outgrown buffers retire (owned_alloc)
int ensure_scratch(go2p_handle* h, go2p_handle::Scratch& sc, int64_t rows, size_t row_bytes) {
  if (sc.rows >= rows) return GO2P_OK;
  sc.buf[0] = sc.buf[1] = nullptr;
  sc.rows = 0;
  for (void*& b : sc.buf)
    if (const int rc = owned_alloc(h, b, (size_t)rows * row_bytes)) return rc;
  sc.rows = rows;
  return GO2P_OK;
}

int launch_fp32(go2p_handle* h, int set, const float* d_obs, const int32_t* d_button0, float* d_act, double* d_qdes,
                MotorCmdDev* d_cmd, int64_t B, uint32_t flags, cudaStream_t st) {
  const DevModel& dm = h->dm;
  // the GEMM epilogue stores float4 where the row pitch allows it: the output base has to be 16-byte aligned
  if ((reinterpret_cast<uintptr_t>(d_act) & 15) || (d_qdes && (reinterpret_cast<uintptr_t>(d_qdes) & 15)))
    return fail(GO2P_ERR_INVALID, "fp32 path needs 16-byte aligned act/qdes device pointers");
  const int64_t chunk = std::min<int64_t>(B, kFp32ChunkRows);
  go2p_handle::Scratch& sc = h->fp32_scratch[set];
  int rc = ensure_scratch(h, sc, chunk, (size_t)dm.max_width * sizeof(float));
  if (rc) return rc;
  for (int64_t r0 = 0; r0 < B; r0 += chunk) {
    const int64_t rows = std::min(chunk, B - r0);
    const float* in = d_obs + r0 * dm.in_dim;
    int lda = dm.in_dim;
    for (int l = 0; l < dm.n_layers; ++l) {
      const DevLayer& L = dm.L[l];
      const bool last = l == dm.n_layers - 1;
      float* out = last ? d_act + r0 * dm.out_dim : static_cast<float*>(sc.buf[l & 1]);
      const int ldc = L.N;
      // the narrow output kernel stages 128 whole rows in shared memory: it serves last hidden widths up to ~440;
      // wider ones take the generic GEMM + the elementwise A9/A11 kernel
      const size_t so_smem = ((size_t)kSoRows * (L.K | 1) + (size_t)L.N * L.Kp) * sizeof(float);
      if (last && L.N <= 32 && so_smem <= (size_t)227 * 1024) {
        CU_TRY(opt_in_smem(h, reinterpret_cast<const void*>(small_out_kernel), so_smem));
        small_out_kernel<<<(unsigned)((rows + kSoRows - 1) / kSoRows), kSoRows, so_smem, st>>>(
            in, lda, L.w_rm, L.Kp, L.bias, out, ldc, rows, L.K, L.N, L.has_elu, L.alpha, flags,
            d_button0 ? d_button0 + r0 : nullptr, d_qdes ? d_qdes + r0 * kDof : nullptr, d_cmd ? d_cmd + r0 : nullptr, h->cc);
        h->last_launches++;
      } else {
        dim3 grid((unsigned)((rows + kSgBM - 1) / kSgBM), (unsigned)(L.Np / kSgBN));
        sgemm_bias_act_kernel<<<grid, kSgThreads, 0, st>>>(in, lda, L.w_kn, L.Np, L.bias, out, ldc, (int)rows, L.K, L.N,
                                                          L.has_elu, L.alpha);
        h->last_launches++;
        if (last && flags) {
          const long long total = rows * (long long)dm.out_dim;
          post_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(out, total, dm.out_dim, flags,
                                                                      d_button0 ? d_button0 + r0 : nullptr,
                                                                      d_qdes ? d_qdes + r0 * kDof : nullptr,
                                                                      d_cmd ? d_cmd + r0 : nullptr, h->cc);
          h->last_launches++;
        }
      }
      in = out;
      lda = ldc;
    }
  }
  CU_TRY(cudaGetLastError());
  return GO2P_OK;
}

template <bool kFp16, bool kFused, bool kReset = false, bool kFields = false, bool kSeq = false>
int launch_tc_t(go2p_handle* h, const TcArgs& a, cudaStream_t st) {
  const size_t smem = tc_smem_bytes(a);
  auto kernel = tc_mlp_kernel<kFp16, kFused, kReset, kFields, kSeq>;
  CU_TRY(opt_in_smem(h, reinterpret_cast<const void*>(kernel), smem));
  const long long tiles = (a.B + kTcTileM - 1) / kTcTileM;
  int grid = (int)std::min<long long>(tiles, h->sm_count - (h->resident ? 1 : 0));
  // programmatic stream serialization: the kernel's prologue may overlap the tail of the previous kernel of the stream
  // (it waits for that kernel before touching observations / actions: griddepcontrol.wait in tc_mlp_kernel).  The
  // prologue also issues the weights' bulk copies, so the first launch on the stream of a weight update goes without
  // it: its previous kernel may be the packer (go2p_set_weights).  Other streams reach the new weights through an
  // event or a host synchronisation, which programmatic serialization does not relax.
  const bool after_update = h->tc_w_gen != h->w_gen && st == h->w_stream;
  cudaLaunchConfig_t lc{};
  lc.gridDim = dim3((unsigned)grid); lc.blockDim = dim3(kTcThreads); lc.dynamicSmemBytes = smem; lc.stream = st;
  cudaLaunchAttribute attr{};
  attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr.val.programmaticStreamSerializationAllowed = 1;
  lc.attrs = &attr; lc.numAttrs = after_update ? 0 : 1;
  CU_TRY(cudaLaunchKernelEx(&lc, kernel, a));
  if (after_update) h->tc_w_gen = h->w_gen;
  h->last_launches++;
  CU_TRY(cudaGetLastError());
  return GO2P_OK;
}

// the per-step outputs of tc_mlp_kernel<., true, ., true, true>: T steps, [T,B,.] each (TcArgs)
struct TcSeqOut {
  int T;
  float* act;
  double* qdes;
  MotorCmdDev* cmd;
  float* obs;
};

// raw or fields != null: the fused controller step (A1-A6 in the conversion job) from records or per-field arrays: d_obs
// is the robots' history, updated in place; d_reset (may be null) the robots' reset flags.  seq != null (with fields):
// seq->T steps in one launch, the fields and d_reset holding T*B rows; d_qdes and d_cmd are unused then
int launch_tc(go2p_handle* h, const float* d_obs, const int32_t* d_button0, float* d_act, double* d_qdes,
              MotorCmdDev* d_cmd, int64_t B, bool fp16, uint32_t flags, cudaStream_t st,
              const RawStateDev* raw = nullptr, float* d_vel_cmd = nullptr, const uint8_t* d_reset = nullptr,
              const RawFieldsDev* fields = nullptr, const TcSeqOut* seq = nullptr) {
  if ((reinterpret_cast<uintptr_t>(d_obs) & 15) || (reinterpret_cast<uintptr_t>(d_act) & 15) ||
      (d_qdes && (reinterpret_cast<uintptr_t>(d_qdes) & 15)))
    return fail(GO2P_ERR_INVALID, "tensor-core path needs 16-byte aligned obs/act/qdes device pointers");
  TcArgs a{};
  a.obs = d_obs; a.act = d_act; a.button0 = d_button0; a.qdes = d_qdes; a.B = B;
  a.cmd = d_cmd; a.kp = h->cc.kp; a.kd = h->cc.kd; a.kp_deadman = h->cc.kp_deadman;
  a.sat_count = nullptr;
  if (flags & GO2P_F_SAT_COUNT) {
    if (!h->d_sat) {
      if (const int rc = owned_alloc(h, h->d_sat, sizeof(unsigned long long))) return rc;
      CU_TRY(cudaMemsetAsync(h->d_sat, 0, sizeof(unsigned long long), st));
    }
    a.sat_count = h->d_sat;
  }
  a.wpack = h->d_wpack[fp16 ? 1 : 0];
  a.n_layers = h->dm.n_layers; a.in_dim = h->dm.in_dim; a.k0p = h->k0p; a.out_dim = h->dm.out_dim;
  for (int l = 0; l < h->dm.n_layers; ++l) {
    const float alpha = h->dm.L[l].alpha;
    a.has_elu[l] = !h->dm.L[l].has_elu ? kEluNone : (alpha >= 0.f && alpha <= 1.f) ? kEluMax : kEluSelect;
    a.elu_c[l] = (float)((double)h->dm.L[l].alpha * 1.4426950408889634074);
  }
  a.out_scale = h->dm.L[h->dm.n_layers - 1].has_elu ? 0.69314718055994530942f : 1.0f;
  a.flags = flags;
  a.action_limit = h->cc.action_limit;
  a.action_scale = h->cc.action_scale;
  for (int i = 0; i < kDof; ++i) a.q0[i] = h->cc.q0[i];
  a.trace = nullptr;
#ifdef GO2P_TC_TRACE
  if (const char* e = std::getenv("GO2P_TC_TRACE_PTR")) a.trace = reinterpret_cast<unsigned long long*>(std::strtoull(e, nullptr, 0));
#endif
  a.raw = raw; a.obs_rw = const_cast<float*>(d_obs); a.vel_cmd = d_vel_cmd; a.H = h->cc.H; a.foot_threshold = h->cc.foot_threshold;
  a.reset = raw || fields ? d_reset : nullptr;
  if (fields && seq) {
    a.fields = *fields;
    a.T = seq->T; a.act_seq = seq->act; a.qdes_seq = seq->qdes; a.cmd_seq = seq->cmd; a.obs_seq = seq->obs;
    if (d_reset) return fp16 ? launch_tc_t<true, true, true, true, true>(h, a, st) : launch_tc_t<false, true, true, true, true>(h, a, st);
    return fp16 ? launch_tc_t<true, true, false, true, true>(h, a, st) : launch_tc_t<false, true, false, true, true>(h, a, st);
  }
  if (fields) {
    a.fields = *fields;
    if (d_reset) return fp16 ? launch_tc_t<true, true, true, true>(h, a, st) : launch_tc_t<false, true, true, true>(h, a, st);
    return fp16 ? launch_tc_t<true, true, false, true>(h, a, st) : launch_tc_t<false, true, false, true>(h, a, st);
  }
  if (raw && d_reset) return fp16 ? launch_tc_t<true, true, true>(h, a, st) : launch_tc_t<false, true, true>(h, a, st);
  if (raw) return fp16 ? launch_tc_t<true, true>(h, a, st) : launch_tc_t<false, true>(h, a, st);
  return fp16 ? launch_tc_t<true, false>(h, a, st) : launch_tc_t<false, false>(h, a, st);
}

}  // namespace

struct go2p_fleet {
  std::vector<go2p_handle*> handles;
};

namespace {
// one host thread per device: each drives its own handle (its own streams and scratch) on its shard of the rows
template <class Fn>
int fleet_run(go2p_fleet* f, int64_t B, Fn&& per_shard) {
  const int n = (int)f->handles.size();
  std::vector<int> rc(n, GO2P_OK);
  std::vector<std::string> msg(n);
  std::vector<std::thread> threads;
  for (int i = 0; i < n; ++i) {
    threads.emplace_back([&, i]() {
      int64_t b = 0, e = 0;
      go2p_shard_rows(B, n, i, &b, &e);
      if (e > b) { rc[i] = per_shard(f->handles[i], b, e - b); if (rc[i]) msg[i] = g_err; }   // g_err is thread-local
    });
  }
  for (auto& t : threads) t.join();
  for (int i = 0; i < n; ++i) if (rc[i]) return fail(rc[i], "device shard " + std::to_string(i) + ": " + msg[i]);
  return GO2P_OK;
}

// The host-buffer pipeline: B rows in chunks of kHostChunkRows, round robin over the kPipeDepth pipe streams, so one
// chunk's copies overlap another's kernels.  per_chunk(slot, r0, rows, stream) queues the chunk's copy in, its kernels
// on stream set 1 + slot and its copy out; last_launches ends as the sum over the chunks.
// Not re-entrant: one host thread per handle (the reference's single-threaded executor, controller.cpp:282).
template <class Fn>
int host_pipeline(go2p_handle* h, int64_t B, Fn&& per_chunk) {
  const int64_t chunk = std::min<int64_t>(B, kHostChunkRows);
  int launches = 0, slot = 0;
  for (int64_t r0 = 0; r0 < B; r0 += chunk, slot = (slot + 1) % kPipeDepth) {
    const int rc = per_chunk(slot, r0, std::min(chunk, B - r0), h->pipe_stream[slot]);
    if (rc) return rc;
    launches += h->last_launches;
  }
  for (int i = 0; i < kPipeDepth; ++i) CU_TRY(cudaStreamSynchronize(h->pipe_stream[i]));
  h->last_launches = launches;
  return GO2P_OK;
}
}  // namespace

// =============================================================================================
extern "C" {

int go2p_abi_version(void) { return GO2P_ABI_VERSION; }
const char* go2p_last_error(void) { return g_err.c_str(); }

void go2p_config_default(go2p_config* c) {
  if (!c) return;
  std::memset(c, 0, sizeof(*c));
  c->struct_size = sizeof(go2p_config);
  c->device = 0;
  c->b1_mode = GO2P_B1_PERSISTENT;
  if (const char* e = std::getenv("GO2P_B1_MODE")) {
    if (!std::strcmp(e, "graph")) c->b1_mode = GO2P_B1_GRAPH;
    else if (!std::strcmp(e, "launch")) c->b1_mode = GO2P_B1_LAUNCH;
  }
  c->history = 2;                                   // controller.hpp:15
  c->action_limit = 1000.0f;                        // controller.hpp:16
  c->action_scale = 0.25;                           // controller.cpp:244
  const double q0[12] = {0.1, -0.1, 0.1, -0.1, 0.8, 0.8, 1.0, 1.0, -1.5, -1.5, -1.5, -1.5};   // controller.hpp:165
  std::memcpy(c->q0, q0, sizeof(q0));
  c->foot_threshold = 22;                           // controller.hpp:100-103
  c->kp = 28.0f; c->kd = 0.5f;                      // controller.hpp:119-120
  c->kp_deadman = 5.0f;                             // controller.cpp:246
  c->log_level = 2;
  c->timeout_ms = 2000;
  c->idle_exit_ms = 30000;
  if (const char* e = std::getenv("GO2P_IDLE_EXIT_MS")) c->idle_exit_ms = std::atoi(e);
}

int go2p_create(const char* onnx_path, const go2p_config* cfg_in, go2p_handle** out) {
  if (!onnx_path || !out) return fail(GO2P_ERR_INVALID, "go2p_create: null argument");
  *out = nullptr;
  go2p_config cfg;
  go2p_config_default(&cfg);
  if (cfg_in) {
    if (cfg_in->struct_size != sizeof(go2p_config)) return fail(GO2P_ERR_INVALID, "go2p_config.struct_size mismatch (ABI)");
    cfg = *cfg_in;
  }
  if (cfg.history < 1 || cfg.history > GO2P_MAX_HISTORY) return fail(GO2P_ERR_INVALID, "history must be in [1,8]");

  MlpModel model;
  try {
    model = load_onnx_mlp(onnx_path);
  } catch (const std::exception& e) {
    const std::string w = e.what();
    return fail(w.rfind("io:", 0) == 0 ? GO2P_ERR_IO : GO2P_ERR_MODEL, w);
  }
  if ((int)model.layers.size() > kMaxLayers) return fail(GO2P_ERR_UNSUPPORTED, "more than 8 Gemm layers");

  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(GO2P_ERR_NO_DEVICE, "no CUDA device visible: this library has no CPU fallback");
  }
  if (cfg.device < 0 || cfg.device >= ndev) return fail(GO2P_ERR_INVALID, "device ordinal out of range");
  cudaDeviceProp prop;
  CU_TRY(cudaGetDeviceProperties(&prop, cfg.device));
  if (prop.major != 10)
    return fail(GO2P_ERR_NO_DEVICE, std::string("device '") + prop.name + "' is sm_" + std::to_string(prop.major) +
                                        std::to_string(prop.minor) + "; the kernels are built for sm_100a only (no fallback)");

  auto* h = new go2p_handle();
  h->cfg = cfg;
  h->model = std::move(model);
  h->device = cfg.device;
  h->sm_count = prop.multiProcessorCount;
  h->cc_major = prop.major;
  h->cc_minor = prop.minor;
  DeviceGuard g(h->device);
  int rc = upload_model(h);
  if (rc == GO2P_OK) {
    h->n_in_slots = round_up(std::max(h->dm.in_dim, kRawWords), 32);
    if (h->n_in_slots > kB1Threads) rc = fail(GO2P_ERR_UNSUPPORTED, "batch-1 path supports in_dim <= 512");
    // MSG_ACT answers out_dim words + two timing words, one per thread, below the farewell slot
    else if (h->dm.out_dim + 2 > std::min(kB1Threads, kByeSlot)) rc = fail(GO2P_ERR_UNSUPPORTED, "batch-1 path supports out_dim <= 510");
  }
  auto cuda_part = [&]() -> int {
    CU_TRY(cudaStreamCreateWithFlags(&h->b1_stream, cudaStreamNonBlocking));
    CU_TRY(cudaHostAlloc((void**)&h->inbox, sizeof(MailWord) * kB1Threads, cudaHostAllocMapped));
    CU_TRY(cudaHostAlloc((void**)&h->outbox, sizeof(MailWord) * kOutSlots, cudaHostAllocMapped));
    std::memset(h->inbox, 0, sizeof(MailWord) * kB1Threads);
    std::memset(h->outbox, 0, sizeof(MailWord) * kOutSlots);
    if (const int e = owned_alloc(h, h->d_state, sizeof(B1State))) return e;
    B1State init{};
    init.kp = h->cfg.kp;
    init.kd = h->cfg.kd;
    CU_TRY(cudaMemcpy(h->d_state, &init, sizeof(init), cudaMemcpyHostToDevice));
    for (int i = 0; i < kPipeDepth; ++i) CU_TRY(cudaStreamCreateWithFlags(&h->pipe_stream[i], cudaStreamNonBlocking));
    return GO2P_OK;
  };
  if (rc == GO2P_OK) rc = cuda_part();
  if (rc != GO2P_OK) {
    const std::string keep = g_err;
    go2p_destroy(h);
    g_err = keep;
    return rc;
  }
  *out = h;
  return GO2P_OK;
}

int go2p_destroy(go2p_handle* h) {
  if (!h) return GO2P_OK;
  DeviceGuard g(h->device);
  if (h->resident) go2p_persistent_stop(h);
  if (h->b1_stream) cudaStreamSynchronize(h->b1_stream);
  if (h->graph_exec) cudaGraphExecDestroy(h->graph_exec);
  if (h->graph) cudaGraphDestroy(h->graph);
  for (cudaStream_t s : h->pipe_stream)
    if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); }
  if (h->b1_stream) cudaStreamDestroy(h->b1_stream);
  if (h->w_event) cudaEventDestroy(h->w_event);
  for (void* p : h->dev_owned) cudaFree(p);
  if (h->inbox) cudaFreeHost(h->inbox);
  if (h->outbox) cudaFreeHost(h->outbox);
  delete h;
  return GO2P_OK;
}

int go2p_model_info(const go2p_handle* h, go2p_model_info_t* info) {
  if (!h || !info) return fail(GO2P_ERR_INVALID, "go2p_model_info: null argument");
  std::memset(info, 0, sizeof(*info));
  info->in_dim = h->dm.in_dim;
  info->out_dim = h->dm.out_dim;
  info->n_layers = h->dm.n_layers;
  info->dims[0] = h->dm.in_dim;
  for (int l = 0; l < h->dm.n_layers; ++l) {
    info->dims[l + 1] = h->dm.L[l].N;
    info->has_elu[l] = h->dm.L[l].has_elu;
    info->elu_alpha[l] = h->dm.L[l].alpha;
  }
  info->input_name = h->model.input_name.c_str();
  info->output_name = h->model.output_name.c_str();
  info->n_params = h->model.n_params();
  info->sm_count = h->sm_count;
  info->cc_major = h->cc_major;
  info->cc_minor = h->cc_minor;
  info->tensor_core_path = (h->tc_ok || h->wide_ok) ? 1 : 0;
  return GO2P_OK;
}

int go2p_inspect_model(const char* onnx_path, go2p_model_info_t* info, double* checksum) {
  if (!onnx_path || !info) return fail(GO2P_ERR_INVALID, "go2p_inspect_model: null argument");
  static thread_local MlpModel model;
  try {
    model = load_onnx_mlp(onnx_path);
  } catch (const std::exception& e) {
    const std::string what = e.what();
    return fail(what.rfind("io:", 0) == 0 ? GO2P_ERR_IO : GO2P_ERR_MODEL, what);
  }
  if ((int)model.layers.size() > kMaxLayers) return fail(GO2P_ERR_UNSUPPORTED, "more than 8 Gemm layers");
  std::memset(info, 0, sizeof(*info));
  info->n_layers = (int)model.layers.size();
  info->in_dim = model.layers.front().in;
  info->out_dim = model.layers.back().out;
  info->dims[0] = info->in_dim;
  double sum = 0.0;
  for (int l = 0; l < info->n_layers; ++l) {
    const MlpLayer& L = model.layers[l];
    info->dims[l + 1] = L.out;
    info->has_elu[l] = L.has_elu ? 1 : 0;
    info->elu_alpha[l] = L.elu_alpha;
    size_t i = 0;
    for (float w : L.weight) sum += (double)((i++ % 97) + 1) * (double)w;
    for (float b : L.bias) sum += (double)((i++ % 97) + 1) * (double)b;
  }
  info->input_name = model.input_name.c_str();
  info->output_name = model.output_name.c_str();
  info->n_params = model.n_params();
  if (checksum) *checksum = sum;
  return GO2P_OK;
}

// ------------------------------------------------------------------------------------- batch-1
int go2p_persistent_start(go2p_handle* h) {
  if (!h) return fail(GO2P_ERR_INVALID, "null handle");
  if (h->resident) return GO2P_OK;
  DeviceGuard g(h->device);
  bool fit = false;
  const size_t smem = b1_smem_bytes(h, true, &fit);
  const bool regs = b1_regs_ok(h);
  CU_TRY(opt_in_smem(h, regs ? reinterpret_cast<const void*>(b1_kernel<true, true>) : reinterpret_cast<const void*>(b1_kernel<true, false>), smem));
  ++h->epoch;
  B1Args a = make_b1_args(h, fit);
  if (regs) b1_kernel<true, true><<<1, kB1Threads, smem, h->b1_stream>>>(a);
  else b1_kernel<true, false><<<1, kB1Threads, smem, h->b1_stream>>>(a);
  CU_TRY(cudaGetLastError());
  h->resident = true;
  h->b1_smem = smem;
  h->b1_weights_in_smem = fit;
  return GO2P_OK;
}

int go2p_persistent_stop(go2p_handle* h) {
  if (!h) return fail(GO2P_ERR_INVALID, "null handle");
  if (!h->resident) return GO2P_OK;
  DeviceGuard g(h->device);
  if (resident_said_goodbye(h)) {
    h->resident = false;
    CU_TRY(cudaStreamSynchronize(h->b1_stream));
    return GO2P_OK;
  }
  uint32_t tag;
  mail_send(h, MSG_EXIT, nullptr, 0, &tag);
  int rc = mail_wait(h, tag, 1);
  h->resident = false;
  if (rc) return rc;
  CU_TRY(cudaStreamSynchronize(h->b1_stream));
  return GO2P_OK;
}

int go2p_bind(go2p_handle* h, float* obs, size_t n_obs, float* act, size_t n_act) {
  if (!h || !obs || !act) return fail(GO2P_ERR_INVALID, "go2p_bind: null argument");
  if ((int)n_obs < h->dm.in_dim || (int)n_act < h->dm.out_dim)
    return fail(GO2P_ERR_INVALID, "go2p_bind: buffers smaller than the model's input/output dimension");
  h->bound_obs = obs; h->n_bound_obs = n_obs;
  h->bound_act = act; h->n_bound_act = n_act;
  return GO2P_OK;
}

int go2p_act(go2p_handle* h) {
  if (!h) return fail(GO2P_ERR_INVALID, "null handle");
  if (!h->bound_obs) return fail(GO2P_ERR_STATE, "go2p_act: no buffers bound (go2p_bind)");
  DeviceGuard g(h->device);
  uint32_t tag;
  mail_send(h, MSG_ACT, reinterpret_cast<const uint32_t*>(h->bound_obs), h->dm.in_dim, &tag);
  int rc = b1_dispatch(h);
  if (rc) return rc;
  const int n = h->dm.out_dim;
  rc = mail_wait(h, tag, n + 2);
  if (rc) return rc;
  for (int i = 0; i < n; ++i) {
    const uint32_t bits = h->outbox[i].bits;
    std::memcpy(&h->bound_act[i], &bits, 4);
  }
  stats_add(h, (uint64_t)h->outbox[n].bits | ((uint64_t)h->outbox[n + 1].bits << 32));
  return GO2P_OK;
}

int go2p_step_fused(go2p_handle* h, const go2p_raw_state* raw, go2p_step_out* out) {
  if (!h || !raw || !out) return fail(GO2P_ERR_INVALID, "go2p_step_fused: null argument");
  const int n_obs = GO2P_FRAME * h->cfg.history;
  if (h->dm.in_dim != n_obs || h->dm.out_dim != GO2P_DOF)
    return fail(GO2P_ERR_UNSUPPORTED, "fused step needs a policy with 49*history inputs and 12 outputs");
  DeviceGuard g(h->device);
  uint32_t w[kRawWords];
  raw_to_words(*raw, w);
  uint32_t tag;
  mail_send(h, MSG_STEP, w, kRawWords, &tag);
  int rc = b1_dispatch(h);
  if (rc) return rc;
  rc = mail_wait(h, tag, n_obs + 54);
  if (rc) return rc;
  const MailWord* ob = h->outbox;
  auto f32 = [&](int i) { float f; const uint32_t b = ob[i].bits; std::memcpy(&f, &b, 4); return f; };
  auto f64 = [&](int i) { double d; const uint64_t b = (uint64_t)ob[i].bits | ((uint64_t)ob[i + 1].bits << 32); std::memcpy(&d, &b, 8); return d; };
  for (int i = 0; i < n_obs; ++i) out->observation[i] = f32(i);
  for (int i = 0; i < 12; ++i) {
    out->action_raw[i] = f32(n_obs + i);
    out->action[i] = f32(n_obs + 12 + i);
    out->q_des[i] = f64(n_obs + 24 + 2 * i);
  }
  out->kp = f64(n_obs + 48);
  out->kd = f64(n_obs + 50);
  out->device_ns = (uint64_t)ob[n_obs + 52].bits | ((uint64_t)ob[n_obs + 53].bits << 32);
  stats_add(h, out->device_ns);
  return GO2P_OK;
}

// the send_command arguments of the same step in Unitree motor order (data movement only: the values are the kernel's)
int go2p_step_fused_cmd(go2p_handle* h, const go2p_raw_state* raw, go2p_step_out* out, go2p_motor_cmd* cmd) {
  if (!cmd) return fail(GO2P_ERR_INVALID, "go2p_step_fused_cmd: null argument");
  go2p_step_out local;
  go2p_step_out* o = out ? out : &local;
  const int rc = go2p_step_fused(h, raw, o);
  if (rc) return rc;
  for (int i = 0; i < GO2P_DOF; ++i) cmd->q_des[motor_of_isaac(i)] = o->q_des[i];
  cmd->kp = o->kp;
  cmd->kd = o->kd;
  return GO2P_OK;
}

int go2p_b1_closed_loop(go2p_handle* h, const go2p_raw_state* raws, int n_raws, int steps, uint64_t* host_ns,
                        uint64_t* device_ns, go2p_step_out* last) {
  if (!h || !raws || n_raws < 1 || steps < 0) return fail(GO2P_ERR_INVALID, "go2p_b1_closed_loop: bad argument");
  go2p_step_out out;
  for (int i = 0; i < steps; ++i) {
    const auto t0 = std::chrono::steady_clock::now();
    const int rc = go2p_step_fused(h, &raws[i % n_raws], &out);
    const auto t1 = std::chrono::steady_clock::now();
    if (rc) return rc;
    if (host_ns) host_ns[i] = (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(t1 - t0).count();
    if (device_ns) device_ns[i] = out.device_ns;
  }
  if (last && steps > 0) *last = out;
  return GO2P_OK;
}

int go2p_b1_selfdriven(go2p_handle* h, const go2p_raw_state* raws, int n_raws, int steps, float* last_action,
                       float* elapsed_ms) {
  if (!h || !raws || n_raws < 1 || steps < 1) return fail(GO2P_ERR_INVALID, "go2p_b1_selfdriven: bad argument");
  if (h->dm.in_dim != GO2P_FRAME * h->cfg.history || h->dm.out_dim != GO2P_DOF)
    return fail(GO2P_ERR_UNSUPPORTED, "fused step needs a policy with 49*history inputs and 12 outputs");
  DeviceGuard g(h->device);
  bool fit = false;
  const size_t smem = b1_smem_bytes(h, true, &fit);
  const bool regs = b1_regs_ok(h);
  if (!fit && !regs) return fail(GO2P_ERR_UNSUPPORTED, "weights fit neither the register file nor shared memory");
  std::vector<uint32_t> words((size_t)n_raws * kRawWords);
  for (int r = 0; r < n_raws; ++r) raw_to_words(raws[r], &words[(size_t)r * kRawWords]);
  uint32_t* d_raws = nullptr;
  float* d_out = nullptr;
  B1State* d_st = nullptr;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  auto run = [&]() -> int {
    int rc;
    if ((rc = owned_alloc(h, d_raws, words.size() * 4)) || (rc = owned_alloc(h, d_out, 64)) ||
        (rc = owned_alloc(h, d_st, sizeof(B1State))))
      return rc;
    B1State init{};
    init.kp = h->cfg.kp; init.kd = h->cfg.kd;
    CU_TRY(cudaMemcpy(d_st, &init, sizeof(init), cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(d_raws, words.data(), words.size() * 4, cudaMemcpyHostToDevice));
    CU_TRY(opt_in_smem(h, regs ? reinterpret_cast<const void*>(b1_selfdriven_kernel<true>) : reinterpret_cast<const void*>(b1_selfdriven_kernel<false>), smem));
    B1Args a = make_b1_args(h, true);
    a.gstate = d_st;
    CU_TRY(cudaEventCreate(&e0));
    CU_TRY(cudaEventCreate(&e1));
    CU_TRY(cudaEventRecord(e0, h->pipe_stream[0]));
    if (regs) b1_selfdriven_kernel<true><<<1, kB1Threads, smem, h->pipe_stream[0]>>>(a, d_raws, n_raws, steps, d_out);
    else b1_selfdriven_kernel<false><<<1, kB1Threads, smem, h->pipe_stream[0]>>>(a, d_raws, n_raws, steps, d_out);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaEventRecord(e1, h->pipe_stream[0]));
    CU_TRY(cudaEventSynchronize(e1));
    float ms = 0.f;
    CU_TRY(cudaEventElapsedTime(&ms, e0, e1));
    if (elapsed_ms) *elapsed_ms = ms;
    if (last_action) CU_TRY(cudaMemcpyAsync(last_action, d_out, 48, cudaMemcpyDeviceToHost, h->pipe_stream[0]));
    CU_TRY(cudaStreamSynchronize(h->pipe_stream[0]));
    return GO2P_OK;
  };
  const int rc = run();
  if (e0) cudaEventDestroy(e0);
  if (e1) cudaEventDestroy(e1);
  // while the resident kernel runs, cudaFree would block on it: the buffers then stay until go2p_destroy
  if (!h->resident) for (void* p : {(void*)d_raws, (void*)d_out, (void*)d_st}) owned_free(h, p);
  if (rc == GO2P_OK) h->last_launches = 1;
  return rc;
}

int go2p_reset_history(go2p_handle* h) {
  if (!h) return fail(GO2P_ERR_INVALID, "null handle");
  return simple_message(h, MSG_RESET, nullptr, 0);
}

int go2p_set_gains(go2p_handle* h, float kp, float kd) {
  if (!h) return fail(GO2P_ERR_INVALID, "null handle");
  uint32_t w[2];
  std::memcpy(&w[0], &kp, 4);
  std::memcpy(&w[1], &kd, 4);
  h->cfg.kp = h->cc.kp = kp;       // the batched epilogues read the gains from the handle
  h->cfg.kd = h->cc.kd = kd;
  return simple_message(h, MSG_GAINS, w, 2);
}

int go2p_b1_stats_get(go2p_handle* h, go2p_b1_stats* out, int reset) {
  if (!h || !out) return fail(GO2P_ERR_INVALID, "null argument");
  *out = h->stats;
  if (out->steps == 0) out->device_ns_min = 0;
  if (reset) h->stats = go2p_b1_stats{0, ~0ull, 0, 0};
  return GO2P_OK;
}

// ------------------------------------------------------------------------------------- batched
namespace {
// the per-layer GEMM chain (kernels_wide.cuh) with the activation buffers sc of one stream set
int launch_wide(go2p_handle* h, go2p_handle::Scratch& sc, WdOperands operands, const float* d_obs, const int32_t* d_button0,
                float* d_act, double* d_qdes, MotorCmdDev* cmd, int64_t B, uint32_t flags, cudaStream_t st) {
  const size_t pieces = operands == kWdSplit ? 3 : 1;
  if (ensure_scratch(h, sc, wide_act_rows(B), pieces * h->wide.max_kp * sizeof(uint16_t)))
    return fail(GO2P_ERR_CUDA, "wide_launch: cudaMalloc of the activation buffers failed");
  uint16_t* const act[2] = {static_cast<uint16_t*>(sc.buf[0]), static_cast<uint16_t*>(sc.buf[1])};
  auto opt_in = [h](const void* fn, size_t bytes) { return opt_in_smem(h, fn, bytes); };
  int rc = wide_launch(h->wide, act, d_obs, d_button0, d_act, d_qdes, cmd, B, operands, flags, h->cc, h->sm_count, opt_in, st,
                       &h->last_launches, g_err);
  return rc ? fail(rc, g_err.c_str()) : GO2P_OK;
}

// go2p_infer_batch_cmd with the activation scratch of stream set `set`
int infer_batch_on(go2p_handle* h, int set, const float* d_obs, const int32_t* d_button0, float* d_act, double* d_qdes,
                   go2p_motor_cmd* d_cmd, int64_t B, int precision, uint32_t flags, cudaStream_t st) {
  if (!h) return fail(GO2P_ERR_INVALID, "go2p_infer_batch: null handle");
  if (B < 0) return fail(GO2P_ERR_INVALID, "negative batch");
  if (B == 0) { h->last_launches = 0; return GO2P_OK; }   // empty batch: nothing is read, nothing is launched
  if (!d_obs || !d_act) return fail(GO2P_ERR_INVALID, "go2p_infer_batch: null argument");
  if ((flags & GO2P_F_QDES) && (!d_qdes || h->dm.out_dim != GO2P_DOF))
    return fail(GO2P_ERR_INVALID, "GO2P_F_QDES needs d_qdes and a 12-output policy");
  if ((flags & GO2P_F_MOTOR_CMD) && (!d_cmd || h->dm.out_dim != GO2P_DOF))
    return fail(GO2P_ERR_INVALID, "GO2P_F_MOTOR_CMD needs d_cmd and a 12-output policy");
  if ((flags & GO2P_F_MOTOR_CMD) && (reinterpret_cast<uintptr_t>(d_cmd) & 15))
    return fail(GO2P_ERR_INVALID, "d_cmd must be 16-byte aligned");
  h->last_launches = 0;
  DeviceGuard g(h->device);
  MotorCmdDev* cmd = reinterpret_cast<MotorCmdDev*>(d_cmd);
  switch (precision) {
    case GO2P_PREC_FP32: return launch_fp32(h, set, d_obs, d_button0, d_act, d_qdes, cmd, B, flags, st);
    case GO2P_PREC_BF16:
    case GO2P_PREC_FP16:
      if (h->tc_ok) return launch_tc(h, d_obs, d_button0, d_act, d_qdes, cmd, B, precision == GO2P_PREC_FP16, flags, st);
      if (h->wide_ok)
        return launch_wide(h, h->wide_scratch[set], precision == GO2P_PREC_FP16 ? kWdFp16 : kWdBf16, d_obs, d_button0, d_act,
                           d_qdes, cmd, B, flags, st);
      return fail(GO2P_ERR_UNSUPPORTED, "tensor-core kernels do not serve this layer shape; use GO2P_PREC_FP32");
    case GO2P_PREC_FP32_TC:
      if (h->split_ok) return launch_wide(h, h->split_scratch[set], kWdSplit, d_obs, d_button0, d_act, d_qdes, cmd, B, flags, st);
      return fail(GO2P_ERR_UNSUPPORTED, "GO2P_PREC_FP32_TC serves 2-8 layers, hidden widths that are multiples of 64 and at "
                                        "most 16 outputs; use GO2P_PREC_FP32");
    default: return fail(GO2P_ERR_INVALID, "unknown precision");
  }
}
}  // namespace

int go2p_infer_batch_cmd(go2p_handle* h, const float* d_obs, const int32_t* d_button0, float* d_act, double* d_qdes,
                         go2p_motor_cmd* d_cmd, int64_t B, int precision, uint32_t flags, void* stream) {
  return infer_batch_on(h, 0, d_obs, d_button0, d_act, d_qdes, d_cmd, B, precision, flags, static_cast<cudaStream_t>(stream));
}

int go2p_infer_batch_ex(go2p_handle* h, const float* d_obs, const int32_t* d_button0, float* d_act, double* d_qdes,
                        int64_t B, int precision, uint32_t flags, void* stream) {
  if (flags & GO2P_F_MOTOR_CMD) return fail(GO2P_ERR_INVALID, "GO2P_F_MOTOR_CMD needs go2p_infer_batch_cmd");
  return go2p_infer_batch_cmd(h, d_obs, d_button0, d_act, d_qdes, nullptr, B, precision, flags, stream);
}

int go2p_infer_batch(go2p_handle* h, const float* d_obs, float* d_act, int64_t B, int precision, void* stream) {
  return go2p_infer_batch_cmd(h, d_obs, nullptr, d_act, nullptr, nullptr, B, precision, 0u, stream);
}

int go2p_last_launch_count(const go2p_handle* h) { return h ? h->last_launches : 0; }

// GO2P_F_SAT_COUNT: (row, 32-column operand block) pairs with a saturated fp16 operand in the launches since the last
// reset, read after `stream` has drained
int go2p_saturation_count(go2p_handle* h, uint64_t* count, int reset, void* stream) {
  if (!h || !count) return fail(GO2P_ERR_INVALID, "go2p_saturation_count: null argument");
  *count = 0;
  if (!h->d_sat) return GO2P_OK;                       // no counting launch yet
  DeviceGuard g(h->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned long long v = 0;
  CU_TRY(cudaMemcpyAsync(&v, h->d_sat, sizeof(v), cudaMemcpyDeviceToHost, st));
  if (reset) CU_TRY(cudaMemsetAsync(h->d_sat, 0, sizeof(v), st));
  CU_TRY(cudaStreamSynchronize(st));
  *count = v;
  return GO2P_OK;
}

// Isaac joint index of every Unitree motor (controller.hpp:168-170 vs the SDK's FR, FL, RR, RL x hip, thigh, calf)
int go2p_motor_order(int32_t isaac_of_motor[GO2P_DOF]) {
  if (!isaac_of_motor) return fail(GO2P_ERR_INVALID, "null argument");
  for (int i = 0; i < GO2P_DOF; ++i) isaac_of_motor[motor_of_isaac(i)] = i;
  return GO2P_OK;
}

int go2p_infer_batch_host(go2p_handle* h, const float* h_obs, float* h_act, int64_t B, int precision) {
  if (!h || !h_obs || !h_act) return fail(GO2P_ERR_INVALID, "go2p_infer_batch_host: null argument");
  if (B <= 0) return B == 0 ? GO2P_OK : fail(GO2P_ERR_INVALID, "negative batch");
  DeviceGuard g(h->device);
  const int in = h->dm.in_dim, out = h->dm.out_dim;
  for (int i = 0; i < kPipeDepth; ++i) {
    int rc;
    if ((rc = owned_alloc(h, h->pipe_in[i], (size_t)kHostChunkRows * in * sizeof(float))) ||
        (rc = owned_alloc(h, h->pipe_out[i], (size_t)kHostChunkRows * out * sizeof(float))))
      return rc;
  }
  return host_pipeline(h, B, [&](int slot, int64_t r0, int64_t rows, cudaStream_t st) -> int {
    CU_TRY(cudaMemcpyAsync(h->pipe_in[slot], h_obs + r0 * in, (size_t)rows * in * sizeof(float), cudaMemcpyHostToDevice, st));
    const int rc = infer_batch_on(h, 1 + slot, h->pipe_in[slot], nullptr, h->pipe_out[slot], nullptr, nullptr, rows, precision, 0u, st);
    if (rc) return rc;
    CU_TRY(cudaMemcpyAsync(h_act + r0 * out, h->pipe_out[slot], (size_t)rows * out * sizeof(float), cudaMemcpyDeviceToHost, st));
    return GO2P_OK;
  });
}

int go2p_assemble_batch(go2p_handle* h, const go2p_raw_state* d_raw, const float* d_prev_action, float* d_vel_cmd,
                        float* d_obs, int64_t B, void* stream) {
  if (!h || !d_raw || !d_vel_cmd || !d_obs) return fail(GO2P_ERR_INVALID, "go2p_assemble_batch: null argument");
  if (B <= 0) return B == 0 ? GO2P_OK : fail(GO2P_ERR_INVALID, "negative batch");
  DeviceGuard g(h->device);
  launch_assemble_batch(reinterpret_cast<const RawStateDev*>(d_raw), d_prev_action, d_vel_cmd, d_obs, B, h->cc, nullptr,
                        h->sm_count, static_cast<cudaStream_t>(stream));
  h->last_launches = 1;
  CU_TRY(cudaGetLastError());
  return GO2P_OK;
}

namespace {
bool aligned16(const void* p) { return !(reinterpret_cast<uintptr_t>(p) & 15); }

// whether the fused tensor-core kernel serves this step (the one-launch path)
bool fused_step_ok(const go2p_handle* h, const go2p_raw_state* d_raw, const RawFieldsDev* fields, const float* d_obs,
                   const float* d_action, const double* d_qdes, const go2p_motor_cmd* d_cmd, int precision) {
  TcArgs probe{};
  probe.n_layers = h->dm.n_layers; probe.in_dim = h->dm.in_dim; probe.k0p = h->k0p;
  probe.raw = reinterpret_cast<const RawStateDev*>(d_raw);          // the fused kernel also stages the raw states
  if (fields) probe.fields = *fields;
  // the fused kernel bulk-copies a full tile of records, or of every field, into shared memory
  const bool raw_aligned = fields ? aligned16(fields->quat) && aligned16(fields->gyro) && aligned16(fields->q) &&
                                        aligned16(fields->dq) && aligned16(fields->axes) && aligned16(fields->foot_force) &&
                                        aligned16(fields->joy_valid) && aligned16(fields->button0)
                                  : aligned16(d_raw);
  return h->tc_ok && (precision == GO2P_PREC_FP16 || precision == GO2P_PREC_BF16) && (h->dm.in_dim & 1) == 0 &&
         tc_smem_bytes(probe) <= (size_t)227 * 1024 && raw_aligned &&
         !(reinterpret_cast<uintptr_t>(d_obs) & 15) && !(reinterpret_cast<uintptr_t>(d_action) & 15) &&
         !(d_qdes && (reinterpret_cast<uintptr_t>(d_qdes) & 15)) && !(d_cmd && (reinterpret_cast<uintptr_t>(d_cmd) & 15));
}

// publish() for B robots on device buffers; button_scratch [B] receives the dead-man buttons for the epilogue.
// The raw states are records (d_raw) or per-field arrays (fields); exactly one of the two is non-null.
// d_reset [B] (may be null): robots to start from the initial state, applied by whichever kernel assembles the
// observations (the fused kernel's conversion job or assemble_batch_kernel); the path choice does not depend on it.
// `set`: the stream set whose activation scratch the policy uses.
int step_batch_on(go2p_handle* h, int set, const go2p_raw_state* d_raw, const RawFieldsDev* fields, const uint8_t* d_reset,
                  float* d_vel_cmd, float* d_obs, float* d_action, double* d_qdes, go2p_motor_cmd* d_cmd,
                  int32_t* button_scratch, int64_t B, int precision, cudaStream_t st) {
  const uint32_t all_flags = GO2P_F_CLAMP_MASK | (d_qdes ? GO2P_F_QDES : 0u) | (d_cmd ? GO2P_F_MOTOR_CMD : 0u);
  if (fused_step_ok(h, d_raw, fields, d_obs, d_action, d_qdes, d_cmd, precision)) {
    // ONE launch: A1-A6 run inside the policy kernel's conversion job, the newest frame never round-trips HBM
    h->last_launches = 0;
    return launch_tc(h, d_obs, nullptr, d_action, d_qdes, reinterpret_cast<MotorCmdDev*>(d_cmd), B, precision == GO2P_PREC_FP16,
                     all_flags, st, reinterpret_cast<const RawStateDev*>(d_raw), d_vel_cmd, d_reset, fields);
  }
  // A1-A6: d_action still holds the previous published action here
  launch_assemble_batch(reinterpret_cast<const RawStateDev*>(d_raw), d_action, d_vel_cmd, d_obs, B, h->cc, button_scratch,
                        h->sm_count, st, d_reset, fields);
  CU_TRY(cudaGetLastError());
  // A7 + A9 + A11
  const uint32_t flags = GO2P_F_CLAMP_MASK | (d_qdes ? GO2P_F_QDES : 0u) | (d_cmd ? GO2P_F_MOTOR_CMD : 0u);
  const int rc = infer_batch_on(h, set, d_obs, button_scratch, d_action, d_qdes, d_cmd, B, precision, flags, st);
  if (rc == GO2P_OK) h->last_launches += 1;
  return rc;
}

// the device-buffer step's policy check and its button scratch of B rows, under the handle's device
int step_setup(go2p_handle* h, const char* fn, int64_t B) {
  if (h->dm.in_dim != kFrame * h->cc.H || h->dm.out_dim != kDof)
    return fail(GO2P_ERR_INVALID, std::string(fn) + ": the policy is not a 49*H -> 12 controller policy");
  if (h->step_button_rows < B) {
    h->d_step_button = nullptr;   // retire (owned_alloc)
    h->step_button_rows = 0;
    if (const int rc = owned_alloc(h, h->d_step_button, (size_t)B * sizeof(int32_t))) return rc;
    h->step_button_rows = B;
  }
  return GO2P_OK;
}

// the device-buffer step after its pointer checks: batch and policy checks, the button scratch, stream set 0
int step_batch_device(go2p_handle* h, const char* fn, const go2p_raw_state* d_raw, const RawFieldsDev* fields,
                      const uint8_t* d_reset, float* d_vel_cmd, float* d_obs, float* d_action, double* d_qdes,
                      go2p_motor_cmd* d_cmd, int64_t B, int precision, void* stream) {
  if (B <= 0) return B == 0 ? GO2P_OK : fail(GO2P_ERR_INVALID, "negative batch");
  DeviceGuard g(h->device);
  if (const int rc = step_setup(h, fn, B)) return rc;
  return step_batch_on(h, 0, d_raw, fields, d_reset, d_vel_cmd, d_obs, d_action, d_qdes, d_cmd, h->d_step_button, B,
                       precision, static_cast<cudaStream_t>(stream));
}
}  // namespace

int go2p_step_batch_ex(go2p_handle* h, const go2p_raw_state* d_raw, const uint8_t* d_reset, float* d_vel_cmd, float* d_obs,
                       float* d_action, double* d_qdes, go2p_motor_cmd* d_cmd, int64_t B, int precision, void* stream) {
  if (!h || !d_raw || !d_vel_cmd || !d_obs || !d_action || (!d_qdes && !d_cmd))
    return fail(GO2P_ERR_INVALID, "go2p_step_batch: null argument");
  return step_batch_device(h, "go2p_step_batch", d_raw, nullptr, d_reset, d_vel_cmd, d_obs, d_action, d_qdes, d_cmd, B,
                           precision, stream);
}

namespace {
// the pointer checks of the per-field steps: handle, f and its fields, the state and output pointers in `more` (named
// in the message), then `no_output` (the single step's d_qdes and d_cmd both null), then the fields' alignment
int check_fields_step(const char* fn, const go2p_handle* h, const go2p_raw_fields* f,
                      std::initializer_list<std::pair<const void*, const char*>> more, bool no_output) {
  if (!h) return fail(GO2P_ERR_INVALID, std::string(fn) + ": null handle");
  if (!f) return fail(GO2P_ERR_INVALID, std::string(fn) + ": null go2p_raw_fields");
  const std::pair<const void*, const char*> ptrs[] = {
      {f->quat, "quat"}, {f->gyro, "gyro"}, {f->q, "q"}, {f->dq, "dq"}, {f->axes, "axes"}, {f->foot_force, "foot_force"},
      {f->joy_valid, "joy_valid"}, {f->button0, "button0"}};
  for (const auto& p : ptrs)
    if (!p.first) return fail(GO2P_ERR_INVALID, std::string(fn) + ": null " + p.second);
  for (const auto& p : more)
    if (!p.first) return fail(GO2P_ERR_INVALID, std::string(fn) + ": null " + p.second);
  if (no_output) return fail(GO2P_ERR_INVALID, std::string(fn) + ": d_qdes and d_cmd are both null");
  // the two-kernel chain reads the fields at any alignment of their element type
  const auto addr = [](const void* p) { return reinterpret_cast<uintptr_t>(p); };
  if (((addr(f->quat) | addr(f->gyro) | addr(f->q) | addr(f->dq) | addr(f->axes)) & 3) || (addr(f->foot_force) & 1))
    return fail(GO2P_ERR_INVALID, std::string(fn) + ": a field is not aligned to its element size");
  return GO2P_OK;
}
}  // namespace

int go2p_step_batch_fields(go2p_handle* h, const go2p_raw_fields* f, const uint8_t* d_reset, float* d_vel_cmd,
                           float* d_obs, float* d_action, double* d_qdes, go2p_motor_cmd* d_cmd, int64_t B,
                           int precision, void* stream) {
  const char* fn = "go2p_step_batch_fields";
  if (const int rc = check_fields_step(fn, h, f, {{d_vel_cmd, "d_vel_cmd"}, {d_obs, "d_obs"}, {d_action, "d_action"}},
                                       !d_qdes && !d_cmd))
    return rc;
  const RawFieldsDev fd{f->quat, f->gyro, f->q, f->dq, f->axes, f->foot_force, f->joy_valid, f->button0};
  return step_batch_device(h, fn, nullptr, &fd, d_reset, d_vel_cmd, d_obs, d_action, d_qdes, d_cmd, B, precision, stream);
}

int go2p_step_batch_fields_seq(go2p_handle* h, const go2p_raw_fields* f, int64_t T, const uint8_t* d_reset,
                               float* d_vel_cmd, float* d_obs, float* d_action, float* d_action_seq,
                               double* d_qdes_seq, go2p_motor_cmd* d_cmd_seq, float* d_obs_seq,
                               int64_t B, int precision, void* stream) {
  const char* fn = "go2p_step_batch_fields_seq";
  if (const int rc = check_fields_step(fn, h, f, {{d_vel_cmd, "d_vel_cmd"}, {d_obs, "d_obs"}, {d_action, "d_action"},
                                                  {d_action_seq, "d_action_seq"}}, false))
    return rc;
  if (T < 0 || B < 0) return fail(GO2P_ERR_INVALID, std::string(fn) + ": negative T or B");
  // bounded with the largest history, before anything reads the handle
  if (T > 0 && B > 0 && B > INT64_MAX / (kFrame * kMaxHistory) / T)
    return fail(GO2P_ERR_INVALID, std::string(fn) + ": T * B * 49 * H overflows int64");
  if (T == 0 || B == 0) return GO2P_OK;
  const int64_t frame = (int64_t)kFrame * h->cc.H;
  DeviceGuard g(h->device);
  if (const int rc = step_setup(h, fn, B)) return rc;
  const cudaStream_t st = static_cast<cudaStream_t>(stream);
  const RawFieldsDev fd{f->quat, f->gyro, f->q, f->dq, f->axes, f->foot_force, f->joy_valid, f->button0};

  // ONE launch where the fused kernel serves step 0 and every step's slices stay 16-byte aligned (B % 16 == 0: the
  // one-byte fields), for the 12-output policy without a final activation; a CTA's (tile, step) units must count in int
  const int64_t tiles = (B + kTcTileM - 1) / kTcTileM;
  const int64_t grid = std::max<int64_t>(1, std::min<int64_t>(tiles, h->sm_count - (h->resident ? 1 : 0)));
  const int64_t pairs = ((tiles + grid - 1) / grid + 1) / 2;
  const auto a16 = [](const void* p) { return !(reinterpret_cast<uintptr_t>(p) & 15); };
  if (fused_step_ok(h, nullptr, &fd, d_obs, d_action, d_qdes_seq, d_cmd_seq, precision) && (B & 15) == 0 &&
      a16(d_action_seq) && (!d_obs_seq || a16(d_obs_seq)) && !h->dm.L[h->dm.n_layers - 1].has_elu &&
      T <= INT32_MAX / 2 / pairs) {
    h->last_launches = 0;
    const TcSeqOut seq{(int)T, d_action_seq, d_qdes_seq, reinterpret_cast<MotorCmdDev*>(d_cmd_seq), d_obs_seq};
    const uint32_t flags = GO2P_F_CLAMP_MASK | (d_qdes_seq ? GO2P_F_QDES : 0u) | (d_cmd_seq ? GO2P_F_MOTOR_CMD : 0u);
    return launch_tc(h, d_obs, nullptr, d_action, nullptr, nullptr, B, precision == GO2P_PREC_FP16, flags, st, nullptr,
                     d_vel_cmd, d_reset, &fd, &seq);
  }
  // otherwise the single step T times on the step-t slices, each taking its own path, and copies of the state into the
  // per-step outputs; the launch count is the steps' kernels (the copies are not counted)
  int launches = 0;
  for (int64_t t = 0; t < T; ++t) {
    const int64_t r = t * B;
    const RawFieldsDev ft{fd.quat + r * 4, fd.gyro + r * 3, fd.q + r * kDof, fd.dq + r * kDof, fd.axes + r * 4,
                          fd.foot_force + r * 4, fd.joy_valid + r, fd.button0 + r};
    if (const int rc = step_batch_on(h, 0, nullptr, &ft, d_reset ? d_reset + r : nullptr, d_vel_cmd, d_obs, d_action,
                                     d_qdes_seq ? d_qdes_seq + r * kDof : nullptr, d_cmd_seq ? d_cmd_seq + r : nullptr,
                                     h->d_step_button, B, precision, st))
      return rc;
    launches += h->last_launches;
    CU_TRY(cudaMemcpyAsync(d_action_seq + r * kDof, d_action, (size_t)B * kDof * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (d_obs_seq)
      CU_TRY(cudaMemcpyAsync(d_obs_seq + r * frame, d_obs, (size_t)(B * frame) * sizeof(float), cudaMemcpyDeviceToDevice, st));
  }
  h->last_launches = launches;
  return GO2P_OK;
}

int go2p_step_batch_cmd(go2p_handle* h, const go2p_raw_state* d_raw, float* d_vel_cmd, float* d_obs, float* d_action,
                        double* d_qdes, go2p_motor_cmd* d_cmd, int64_t B, int precision, void* stream) {
  return go2p_step_batch_ex(h, d_raw, nullptr, d_vel_cmd, d_obs, d_action, d_qdes, d_cmd, B, precision, stream);
}

int go2p_step_batch(go2p_handle* h, const go2p_raw_state* d_raw, float* d_vel_cmd, float* d_obs, float* d_action,
                    double* d_qdes, int64_t B, int precision, void* stream) {
  if (!d_qdes) return fail(GO2P_ERR_INVALID, "go2p_step_batch: null argument");
  return go2p_step_batch_cmd(h, d_raw, d_vel_cmd, d_obs, d_action, d_qdes, nullptr, B, precision, stream);
}

// Closed-loop control step for a fleet from HOST buffers: per-robot history / joystick command / previous action stay
// on the device inside the handle, so a step moves 156 B of raw state in and 48 B of action (+ 112 B of motor command
// if asked for) out per robot instead of the 392 + 48 B of go2p_infer_batch_host.  h_reset (may be null): 1 B more per
// robot, staged per chunk next to the raw states.
int go2p_step_batch_host_ex(go2p_handle* h, const go2p_raw_state* h_raw, const uint8_t* h_reset, float* h_action,
                            go2p_motor_cmd* h_cmd, int64_t B, int precision) {
  if (!h || !h_raw || !h_action) return fail(GO2P_ERR_INVALID, "go2p_step_batch_host: null argument");
  if (B <= 0) return B == 0 ? GO2P_OK : fail(GO2P_ERR_INVALID, "negative batch");
  if (h->dm.in_dim != kFrame * h->cc.H || h->dm.out_dim != kDof)
    return fail(GO2P_ERR_INVALID, "go2p_step_batch_host: the policy is not a 49*H -> 12 controller policy");
  DeviceGuard g(h->device);
  go2p_handle::Fleet& f = h->fleet;
  const int n_obs = h->dm.in_dim;
  int rc;
  if (f.robots != B) {
    // (re)create the fleet state: histories 0, joystick command 0, previous action 0 (controller.hpp:132-162); the
    // old buffers retire (owned_alloc)
    f.robots = 0;
    f.obs = f.vel = f.act = nullptr;
    if ((rc = owned_alloc(h, f.obs, (size_t)B * n_obs * sizeof(float))) || (rc = owned_alloc(h, f.vel, (size_t)B * 3 * sizeof(float))) ||
        (rc = owned_alloc(h, f.act, (size_t)B * kDof * sizeof(float))))
      return rc;
    CU_TRY(cudaMemsetAsync(f.obs, 0, (size_t)B * n_obs * sizeof(float), h->pipe_stream[0]));
    CU_TRY(cudaMemsetAsync(f.vel, 0, (size_t)B * 3 * sizeof(float), h->pipe_stream[0]));
    CU_TRY(cudaMemsetAsync(f.act, 0, (size_t)B * kDof * sizeof(float), h->pipe_stream[0]));
    CU_TRY(cudaStreamSynchronize(h->pipe_stream[0]));
    f.robots = B;
  }
  for (int i = 0; i < kPipeDepth; ++i) {
    if ((rc = owned_alloc(h, f.raw[i], (size_t)kHostChunkRows * sizeof(go2p_raw_state))) ||
        (rc = owned_alloc(h, f.cmd[i], (size_t)kHostChunkRows * sizeof(MotorCmdDev))) ||
        (rc = owned_alloc(h, f.button[i], (size_t)kHostChunkRows * sizeof(int32_t))) ||
        (h_reset && (rc = owned_alloc(h, f.reset[i], (size_t)kHostChunkRows))))
      return rc;
  }
  return host_pipeline(h, B, [&](int slot, int64_t r0, int64_t rows, cudaStream_t st) -> int {
    CU_TRY(cudaMemcpyAsync(f.raw[slot], h_raw + r0, (size_t)rows * sizeof(go2p_raw_state), cudaMemcpyHostToDevice, st));
    if (h_reset) CU_TRY(cudaMemcpyAsync(f.reset[slot], h_reset + r0, (size_t)rows, cudaMemcpyHostToDevice, st));
    const int rc = step_batch_on(h, 1 + slot, f.raw[slot], nullptr, h_reset ? f.reset[slot] : nullptr, f.vel + r0 * 3, f.obs + r0 * n_obs,
                                 f.act + r0 * kDof, nullptr, h_cmd ? reinterpret_cast<go2p_motor_cmd*>(f.cmd[slot]) : nullptr,
                                 f.button[slot], rows, precision, st);
    if (rc) return rc;
    CU_TRY(cudaMemcpyAsync(h_action + r0 * kDof, f.act + r0 * kDof, (size_t)rows * kDof * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (h_cmd) CU_TRY(cudaMemcpyAsync(h_cmd + r0, f.cmd[slot], (size_t)rows * sizeof(MotorCmdDev), cudaMemcpyDeviceToHost, st));
    return GO2P_OK;
  });
}

int go2p_step_batch_host(go2p_handle* h, const go2p_raw_state* h_raw, float* h_action, go2p_motor_cmd* h_cmd, int64_t B,
                         int precision) {
  return go2p_step_batch_host_ex(h, h_raw, nullptr, h_action, h_cmd, B, precision);
}

int go2p_step_batch_host_reset(go2p_handle* h) {
  if (!h) return fail(GO2P_ERR_INVALID, "null handle");
  h->fleet.robots = 0;     // the next go2p_step_batch_host call re-creates zeroed state
  return GO2P_OK;
}

// ------------------------------------------------------------------------------------- weight updates
namespace {
int check_weight_args(const char* fn, const go2p_handle* h, const float* const* w, int n_layers, const float* mean,
                      const float* stdv) {
  const std::string f(fn);
  if (!h) return fail(GO2P_ERR_INVALID, f + ": null handle");
  if (n_layers != h->dm.n_layers)
    return fail(GO2P_ERR_INVALID, f + ": n_layers " + std::to_string(n_layers) + " does not match the handle's " +
                                      std::to_string(h->dm.n_layers));
  if (!w) return fail(GO2P_ERR_INVALID, f + ": null weight array");
  for (int l = 0; l < n_layers; ++l)
    if (!w[l]) return fail(GO2P_ERR_INVALID, f + ": null weight pointer for layer " + std::to_string(l));
  if ((mean == nullptr) != (stdv == nullptr)) return fail(GO2P_ERR_INVALID, f + ": obs_mean and obs_std go together");
  return GO2P_OK;
}

// the handle's own streams: the batch-1 stream and the host pipeline's
std::array<cudaStream_t, 1 + kPipeDepth> own_streams(const go2p_handle* h) {
  std::array<cudaStream_t, 1 + kPipeDepth> own = {h->b1_stream};
  for (int i = 0; i < kPipeDepth; ++i) own[1 + i] = h->pipe_stream[i];
  return own;
}

// Before the packer touches the images: the resident batch-1 kernel (which holds the weights in registers or shared
// memory) is stopped -- it saves its state to d_state and is relaunched lazily by the next batch-1 call -- and `st`
// waits for whatever the handle's own streams have queued, the previous update's packer included.
int begin_update(go2p_handle* h, cudaStream_t st) {
  if (h->resident) { const int rc = go2p_persistent_stop(h); if (rc) return rc; }
  if (!h->w_event) CU_TRY(cudaEventCreateWithFlags(&h->w_event, cudaEventDisableTiming));
  for (cudaStream_t s : own_streams(h)) {
    if (s == st) continue;
    CU_TRY(cudaEventRecord(h->w_event, s));
    CU_TRY(cudaStreamWaitEvent(st, h->w_event, 0));
  }
  return GO2P_OK;
}

// The packer (kernels_pack.cuh) on `st`, then the handle's own streams wait for it: a batch-1 call or a host-buffer
// step issued after this returns computes with the new weights without a host synchronisation.
int pack_and_publish(go2p_handle* h, const float* const* w, const float* const* b, const float* mean, const float* stdv,
                     cudaStream_t st) {
  const DevModel& dm = h->dm;
  PackArgs pa{};
  pa.n_layers = dm.n_layers;
  long long widest = 0;
  for (int l = 0; l < dm.n_layers; ++l) {
    const DevLayer& D = dm.L[l];
    PackLayer& P = pa.L[l];
    P.w = w[l]; P.b = b ? b[l] : nullptr;
    P.K = D.K; P.N = D.N; P.Kp = D.Kp; P.Np = D.Np;
    P.w_rm = const_cast<float*>(D.w_rm); P.w_k4 = const_cast<float*>(D.w_k4);
    P.w_kn = const_cast<float*>(D.w_kn); P.bias = const_cast<float*>(D.bias);
    if (h->tc_ok) {
      for (int f = 0; f < 2; ++f) P.tc[f] = h->d_wpack[f] + h->tc_off[l];
      P.tc_Kp = h->tc_kp[l]; P.wscale = h->tc_wscale[l]; P.bscale = h->tc_bscale[l];
    }
    if (h->wide_ok) {
      const WideLayerDev& W = h->wide.L[l];
      for (int f = 0; f < 2; ++f) P.wd[f] = const_cast<uint16_t*>(W.w[f]);
      P.wd_bias = const_cast<float*>(W.bias); P.wd_NT = W.NT; P.wd_Kp = W.Kp;
    }
    if (h->split_ok) {
      const WideLayerDev& W = h->wide.L[l];
      pa.S[l] = PackSplitLayer{const_cast<uint16_t*>(W.w3), const_cast<float*>(W.bias), W.NT3, W.Kp};
    }
    widest = std::max<long long>(widest, (long long)D.N * (D.K + 1));
  }
  if (mean) {
    const int K = dm.L[0].K, N = dm.L[0].N;
    if (const int rc = owned_alloc(h, h->w_fold, ((size_t)N * K + N) * sizeof(float))) return rc;
    fold_normaliser_kernel<<<(N + 127) / 128, 128, 0, st>>>(w[0], b ? b[0] : nullptr, mean, stdv, K, N, h->w_fold,
                                                           h->w_fold + (size_t)N * K);
    CU_TRY(cudaGetLastError());
    pa.L[0].w = h->w_fold;
    pa.L[0].b = h->w_fold + (size_t)N * K;
  }
  const int blocks = (int)std::min<long long>((widest + 255) / 256, (long long)h->sm_count * 4);
  const dim3 grid((unsigned)blocks, (unsigned)dm.n_layers);
  if (h->split_ok) pack_weights_kernel<true><<<grid, 256, 0, st>>>(pa);
  else pack_weights_kernel<false><<<grid, 256, 0, st>>>(pa);
  CU_TRY(cudaGetLastError());
  CU_TRY(cudaEventRecord(h->w_event, st));
  for (cudaStream_t s : own_streams(h))
    if (s != st) CU_TRY(cudaStreamWaitEvent(s, h->w_event, 0));
  ++h->w_gen;
  h->w_stream = st;
  return GO2P_OK;
}
}  // namespace

int go2p_set_weights(go2p_handle* h, const float* const* d_weight, const float* const* d_bias, int n_layers,
                     const float* d_obs_mean, const float* d_obs_std, void* stream) {
  int rc = check_weight_args("go2p_set_weights", h, d_weight, n_layers, d_obs_mean, d_obs_std);
  if (rc) return rc;
  DeviceGuard g(h->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if ((rc = begin_update(h, st))) return rc;
  return pack_and_publish(h, d_weight, d_bias, d_obs_mean, d_obs_std, st);
}

int go2p_set_weights_host(go2p_handle* h, const float* const* h_weight, const float* const* h_bias, int n_layers,
                          const float* h_obs_mean, const float* h_obs_std) {
  int rc = check_weight_args("go2p_set_weights_host", h, h_weight, n_layers, h_obs_mean, h_obs_std);
  if (rc) return rc;
  DeviceGuard g(h->device);
  const DevModel& dm = h->dm;
  size_t floats = 2 * (size_t)dm.in_dim;
  for (int l = 0; l < dm.n_layers; ++l) floats += (size_t)dm.L[l].N * dm.L[l].K + dm.L[l].N;
  if ((rc = owned_alloc(h, h->w_stage, floats * sizeof(float)))) return rc;   // the topology is fixed, so is the size
  cudaStream_t st = h->pipe_stream[0];
  if ((rc = begin_update(h, st))) return rc;
  const float* dw[kMaxLayers] = {};
  const float* db[kMaxLayers] = {};
  float* p = h->w_stage;
  auto stage = [&](const float* src, size_t n, const float** dst) -> int {
    CU_TRY(cudaMemcpyAsync(p, src, n * sizeof(float), cudaMemcpyHostToDevice, st));
    *dst = p;
    p += n;
    return GO2P_OK;
  };
  for (int l = 0; l < dm.n_layers; ++l) {
    if ((rc = stage(h_weight[l], (size_t)dm.L[l].N * dm.L[l].K, &dw[l]))) return rc;
    if (h_bias && h_bias[l] && (rc = stage(h_bias[l], (size_t)dm.L[l].N, &db[l]))) return rc;
  }
  const float *dmean = nullptr, *dstd = nullptr;
  if (h_obs_mean && ((rc = stage(h_obs_mean, (size_t)dm.in_dim, &dmean)) || (rc = stage(h_obs_std, (size_t)dm.in_dim, &dstd))))
    return rc;
  if ((rc = pack_and_publish(h, dw, db, dmean, dstd, st))) return rc;
  CU_TRY(cudaStreamSynchronize(st));
  h->tc_w_gen = h->w_gen;   // the packer has completed: no later launch can overlap it
  return GO2P_OK;
}

// ------------------------------------------------------------------------------------- ObservationAction log
int go2p_log_enable(go2p_handle* h, int capacity) {
  if (!h || capacity < 0) return fail(GO2P_ERR_INVALID, "go2p_log_enable: bad argument");
  DeviceGuard g(h->device);
  const bool was_resident = h->resident;
  if (was_resident) { int rc = go2p_persistent_stop(h); if (rc) return rc; }   // the ring pointer is a launch argument
  owned_free(h, h->d_log);
  h->d_log = nullptr;
  h->log_capacity = 0; h->log_tail = 0;
  if (capacity > 0) {
    const size_t bytes = sizeof(LogRing) + (size_t)capacity * kLogRecFloats * sizeof(float);
    if (const int rc = owned_alloc(h, h->d_log, bytes)) return rc;
    CU_TRY(cudaMemset(h->d_log, 0, bytes));
    LogRing hdr{};
    hdr.head = 0; hdr.capacity = (uint32_t)capacity; hdr.n_obs = (uint32_t)h->dm.in_dim;
    CU_TRY(cudaMemcpy(h->d_log, &hdr, offsetof(LogRing, rec), cudaMemcpyHostToDevice));
    h->log_capacity = (uint32_t)capacity;
  }
  if (h->graph_exec) { cudaGraphExecDestroy(h->graph_exec); h->graph_exec = nullptr; }   // captured arguments are stale
  if (h->graph) { cudaGraphDestroy(h->graph); h->graph = nullptr; }
  if (was_resident) return go2p_persistent_start(h);
  return GO2P_OK;
}

int go2p_log_drain(go2p_handle* h, float* out, int max_records, int* n_records, uint64_t* dropped) {
  if (!h || !out || !n_records || max_records < 0) return fail(GO2P_ERR_INVALID, "go2p_log_drain: bad argument");
  *n_records = 0;
  if (dropped) *dropped = 0;
  if (!h->d_log) return fail(GO2P_ERR_STATE, "go2p_log_drain: logging is off (go2p_log_enable)");
  DeviceGuard g(h->device);
  cudaStream_t st = h->pipe_stream[0];      // a copy stream: works while the resident kernel runs
  unsigned long long head = 0;
  CU_TRY(cudaMemcpyAsync(&head, &h->d_log->head, sizeof(head), cudaMemcpyDeviceToHost, st));
  CU_TRY(cudaStreamSynchronize(st));
  uint64_t tail = h->log_tail;
  if (head - tail > h->log_capacity) {      // the writer lapped the reader: the oldest records are gone
    if (dropped) *dropped = head - tail - h->log_capacity;
    tail = head - h->log_capacity;
  }
  const int n = (int)std::min<uint64_t>(head - tail, (uint64_t)max_records);
  const size_t rec_floats = (size_t)h->dm.in_dim + kDof;        // the message payload: float32[n_obs] + float32[12]
  for (int done = 0; done < n;) {
    const uint64_t idx = (tail + done) % h->log_capacity;
    const int run = (int)std::min<uint64_t>((uint64_t)(n - done), h->log_capacity - idx);
    CU_TRY(cudaMemcpy2DAsync(out + (size_t)done * rec_floats, rec_floats * sizeof(float),
                             h->d_log->rec + idx * kLogRecFloats, (size_t)kLogRecFloats * sizeof(float),
                             rec_floats * sizeof(float), (size_t)run, cudaMemcpyDeviceToHost, st));
    done += run;
  }
  CU_TRY(cudaStreamSynchronize(st));
  h->log_tail = tail + n;
  *n_records = n;
  return GO2P_OK;
}

// ------------------------------------------------------------------------------------- several GPUs, one process
int go2p_shard_rows(int64_t B, int n, int i, int64_t* begin, int64_t* end) {
  if (B < 0 || n < 1 || i < 0 || i >= n || !begin || !end) return fail(GO2P_ERR_INVALID, "go2p_shard_rows: bad argument");
  const int64_t q = B / n, r = B % n;
  *begin = i * q + std::min<int64_t>(i, r);
  *end = *begin + q + (i < r ? 1 : 0);
  return GO2P_OK;
}

int go2p_fleet_create(const char* onnx_path, const go2p_config* cfg_in, const int32_t* devices, int n_devices, go2p_fleet** out) {
  if (!onnx_path || !devices || n_devices < 1 || !out) return fail(GO2P_ERR_INVALID, "go2p_fleet_create: bad argument");
  *out = nullptr;
  auto* f = new go2p_fleet();
  for (int i = 0; i < n_devices; ++i) {
    go2p_config cfg;
    if (cfg_in) cfg = *cfg_in; else go2p_config_default(&cfg);
    cfg.device = devices[i];
    go2p_handle* h = nullptr;
    const int rc = go2p_create(onnx_path, &cfg, &h);
    if (rc) { const std::string keep = g_err; go2p_fleet_destroy(f); g_err = keep; return rc; }
    f->handles.push_back(h);
  }
  *out = f;
  return GO2P_OK;
}

int go2p_fleet_destroy(go2p_fleet* f) {
  if (!f) return GO2P_OK;
  for (go2p_handle* h : f->handles) go2p_destroy(h);
  delete f;
  return GO2P_OK;
}

int go2p_fleet_device_count(const go2p_fleet* f) { return f ? (int)f->handles.size() : 0; }


int go2p_fleet_infer_host(go2p_fleet* f, const float* h_obs, float* h_act, int64_t B, int precision) {
  if (!f || f->handles.empty() || !h_obs || !h_act || B < 0) return fail(GO2P_ERR_INVALID, "go2p_fleet_infer_host: bad argument");
  const int in = f->handles[0]->dm.in_dim, out = f->handles[0]->dm.out_dim;
  return fleet_run(f, B, [&](go2p_handle* h, int64_t r0, int64_t rows) {
    return go2p_infer_batch_host(h, h_obs + r0 * in, h_act + r0 * out, rows, precision);
  });
}

int go2p_fleet_step_host_ex(go2p_fleet* f, const go2p_raw_state* h_raw, const uint8_t* h_reset, float* h_action,
                            go2p_motor_cmd* h_cmd, int64_t B, int precision) {
  if (!f || f->handles.empty() || !h_raw || !h_action || B < 0) return fail(GO2P_ERR_INVALID, "go2p_fleet_step_host: bad argument");
  return fleet_run(f, B, [&](go2p_handle* h, int64_t r0, int64_t rows) {
    return go2p_step_batch_host_ex(h, h_raw + r0, h_reset ? h_reset + r0 : nullptr, h_action + r0 * kDof,
                                   h_cmd ? h_cmd + r0 : nullptr, rows, precision);
  });
}

int go2p_fleet_step_host(go2p_fleet* f, const go2p_raw_state* h_raw, float* h_action, go2p_motor_cmd* h_cmd, int64_t B,
                         int precision) {
  return go2p_fleet_step_host_ex(f, h_raw, nullptr, h_action, h_cmd, B, precision);
}

int go2p_fleet_set_weights_host(go2p_fleet* f, const float* const* h_weight, const float* const* h_bias, int n_layers,
                                const float* h_obs_mean, const float* h_obs_std) {
  if (!f || f->handles.empty()) return fail(GO2P_ERR_INVALID, "go2p_fleet_set_weights_host: null fleet");
  for (size_t i = 0; i < f->handles.size(); ++i) {
    const int rc = go2p_set_weights_host(f->handles[i], h_weight, h_bias, n_layers, h_obs_mean, h_obs_std);
    if (rc) return fail(rc, "device " + std::to_string(i) + ": " + g_err);
  }
  return GO2P_OK;
}

// ------------------------------------------------------------------------------------- helpers
int go2p_dev_alloc(go2p_handle* h, size_t bytes, void** dptr) {
  if (!h || !dptr) return fail(GO2P_ERR_INVALID, "null argument");
  DeviceGuard g(h->device);
  CU_TRY(cudaMalloc(dptr, std::max<size_t>(bytes, 16)));
  return GO2P_OK;
}
int go2p_dev_free(go2p_handle* h, void* dptr) {
  if (!h) return fail(GO2P_ERR_INVALID, "null handle");
  if (h->resident) return fail(GO2P_ERR_STATE, "cudaFree would block on the resident batch-1 kernel; stop it first");
  DeviceGuard g(h->device);
  CU_TRY(cudaFree(dptr));
  return GO2P_OK;
}
int go2p_host_alloc(go2p_handle* h, size_t bytes, void** hptr) {
  if (!h || !hptr) return fail(GO2P_ERR_INVALID, "null argument");
  DeviceGuard g(h->device);
  CU_TRY(cudaHostAlloc(hptr, std::max<size_t>(bytes, 16), cudaHostAllocDefault));
  return GO2P_OK;
}
int go2p_host_free(go2p_handle* h, void* hptr) {
  if (!h) return fail(GO2P_ERR_INVALID, "null handle");
  if (h->resident) return fail(GO2P_ERR_STATE, "cudaFreeHost would block on the resident batch-1 kernel; stop it first");
  DeviceGuard g(h->device);
  CU_TRY(cudaFreeHost(hptr));
  return GO2P_OK;
}
int go2p_memcpy_h2d(go2p_handle* h, void* dptr, const void* hptr, size_t bytes, void* stream) {
  if (!h) return fail(GO2P_ERR_INVALID, "null handle");
  DeviceGuard g(h->device);
  CU_TRY(cudaMemcpyAsync(dptr, hptr, bytes, cudaMemcpyHostToDevice, static_cast<cudaStream_t>(stream)));
  return GO2P_OK;
}
int go2p_memcpy_d2h(go2p_handle* h, void* hptr, const void* dptr, size_t bytes, void* stream) {
  if (!h) return fail(GO2P_ERR_INVALID, "null handle");
  DeviceGuard g(h->device);
  CU_TRY(cudaMemcpyAsync(hptr, dptr, bytes, cudaMemcpyDeviceToHost, static_cast<cudaStream_t>(stream)));
  return GO2P_OK;
}
int go2p_stream_sync(go2p_handle* h, void* stream) {
  if (!h) return fail(GO2P_ERR_INVALID, "null handle");
  DeviceGuard g(h->device);
  CU_TRY(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  return GO2P_OK;
}

int go2p_time_batch(go2p_handle* h, const float* d_obs, const int32_t* d_button0, float* d_act, double* d_qdes,
                    int64_t B, int precision, uint32_t flags, void* stream, int iters, float* total_ms) {
  if (!h || !total_ms || iters < 1) return fail(GO2P_ERR_INVALID, "go2p_time_batch: bad argument");
  DeviceGuard g(h->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaEvent_t e0, e1;
  CU_TRY(cudaEventCreate(&e0));
  CU_TRY(cudaEventCreate(&e1));
  CU_TRY(cudaEventRecord(e0, st));
  int launches = 0;
  for (int i = 0; i < iters; ++i) {
    int rc = go2p_infer_batch_ex(h, d_obs, d_button0, d_act, d_qdes, B, precision, flags, stream);
    if (rc) { cudaEventDestroy(e0); cudaEventDestroy(e1); return rc; }
    launches += h->last_launches;
  }
  CU_TRY(cudaEventRecord(e1, st));
  CU_TRY(cudaEventSynchronize(e1));
  CU_TRY(cudaEventElapsedTime(total_ms, e0, e1));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  h->last_launches = launches;
  return GO2P_OK;
}

}  // extern "C"
