// Batch-1 control-loop kernel: one CTA executes a whole ONNXController::publish() step
//   A1-A6 observation assembly   (reference: controller.cpp:173-212, controller.hpp:45-68,99-103)
//   A7    policy forward         (reference: onnx_actor.cpp:38-48 -> Ort::Session::Run)
//   A9    clamp + dead-man mask  (reference: controller.cpp:217-223)
//   A11   joint targets          (reference: controller.cpp:235-248)
// either as a RESIDENT kernel fed through a host-mapped mailbox (launch-free, weights and
// history stay in shared memory: no HBM round trip per step) or as a one-shot launch / CUDA-graph
// node using the same mailbox protocol.
//
// Mailbox protocol: every 32-bit payload word travels with a 32-bit tag in one naturally aligned
// 8-byte unit (MailWord), written and read with single 8-byte accesses, so a word is valid exactly
// when its tag matches the expected (sequence,type); no system-scope fence is needed in either
// direction and the poll that sees the request already carries its data.
#pragma once
#include "policy_dev.cuh"

namespace go2p {

constexpr int kB1Threads = 512;
constexpr int kRawWords = 41;   // quat4 gyro3 q12 dq12 axes4 foot4 joy_valid button0

enum B1Msg : uint32_t { MSG_ACT = 1, MSG_STEP = 2, MSG_RESET = 3, MSG_GAINS = 4, MSG_EXIT = 5 };

struct MailWord { uint32_t bits, tag; };

__host__ __device__ inline uint32_t make_tag(uint32_t seq, uint32_t type) { return (seq << 3) | type; }

struct B1State {
  float obs[kFrame * kMaxHistory];   // term-major history == the observation itself (controller.cpp:210-212)
  float vel_cmd[4];
  float action[kDof];                // previous published action (controller.cpp:206)
  float kp, kd;
  uint32_t seq;                      // last sequence number served
  uint32_t pad;
};

// ObservationAction log (reference: onnx_interfaces/msg/ObservationAction.msg:1-2, filled at controller.cpp:226-229):
// one record per control step = the observation as fed to the policy + the published action, appended to a ring in
// device memory by the step that produced it; `head` counts records ever written and is stored (release) after the
// record, so a drain that reads head and then the records sees complete records only.
constexpr int kLogRecFloats = kFrame * kMaxHistory + kDof;   // fixed pitch: 49*8 + 12 floats
struct LogRing {
  unsigned long long head;
  uint32_t capacity, n_obs;
  float rec[1];            // [capacity][kLogRecFloats]
};

struct B1Args {
  DevModel model;
  CtrlConst cc;
  B1State* gstate;          // device memory copy of the state (source/sink for the resident kernel)
  const MailWord* inbox;    // host-mapped
  MailWord* outbox;         // host-mapped
  int n_in_slots;           // slots the host fills for every message (multiple of 32)
  int weights_in_smem;      // resident kernel only
  int smem_weight_floats;
  // resident kernel only: leave the SM after this long without a message (0 = never).  The host sees
  // the farewell word {epoch, kByeTag} in outbox[kByeSlot] and relaunches on the next request, so an
  // abandoned handle can never pin an SM (or hang a GPU box) for longer than this.
  unsigned long long idle_ns;
  uint32_t epoch;
  LogRing* log;             // ObservationAction ring in device memory, or null (logging off: no HBM traffic per step)
};
constexpr int kOutSlots = 1024;
constexpr int kByeSlot = kOutSlots - 1;
constexpr uint32_t kByeTag = 0xB1E0B1E0u;

__device__ __forceinline__ uint2 ld_mail(const MailWord* p) {
  uint2 v;
  asm volatile("ld.relaxed.sys.global.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_mail(MailWord* p, uint32_t bits, uint32_t tag) {
  asm volatile("st.relaxed.sys.global.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(bits), "r"(tag) : "memory");
}
__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// gb = quaternion_.inverse() * (0,0,-1), Eigen semantics, fp32, no FMA contraction
// (reference: controller.cpp:182-184).  gravity_all: the three components; gravity_component: component c.
__device__ __forceinline__ void gravity_all(const float* quat_wxyz, float (&g)[3]) {
  const float w = quat_wxyz[0], x = quat_wxyz[1], y = quat_wxyz[2], z = quat_wxyz[3];
  const float n2 = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z)), __fmul_rn(w, w));
  float cw = 0.f, u0 = 0.f, u1 = 0.f, u2 = 0.f;
  if (n2 > 0.0f) { cw = __fdiv_rn(w, n2); u0 = __fdiv_rn(-x, n2); u1 = __fdiv_rn(-y, n2); u2 = __fdiv_rn(-z, n2); }
  const float v0 = 0.f, v1 = 0.f, v2 = -1.f;
  float a0 = __fsub_rn(__fmul_rn(u1, v2), __fmul_rn(u2, v1));
  float a1 = __fsub_rn(__fmul_rn(u2, v0), __fmul_rn(u0, v2));
  float a2 = __fsub_rn(__fmul_rn(u0, v1), __fmul_rn(u1, v0));
  a0 = __fadd_rn(a0, a0); a1 = __fadd_rn(a1, a1); a2 = __fadd_rn(a2, a2);
  const float b0 = __fsub_rn(__fmul_rn(u1, a2), __fmul_rn(u2, a1));
  const float b1 = __fsub_rn(__fmul_rn(u2, a0), __fmul_rn(u0, a2));
  const float b2 = __fsub_rn(__fmul_rn(u0, a1), __fmul_rn(u1, a0));
  g[0] = __fadd_rn(__fadd_rn(v0, __fmul_rn(cw, a0)), b0);
  g[1] = __fadd_rn(__fadd_rn(v1, __fmul_rn(cw, a1)), b1);
  g[2] = __fadd_rn(__fadd_rn(v2, __fmul_rn(cw, a2)), b2);
}
__device__ __forceinline__ float gravity_component(const float* quat_wxyz, int c) {
  float g[3];
  gravity_all(quat_wxyz, g);
  return c == 0 ? g[0] : (c == 1 ? g[1] : g[2]);
}

// vel_cmd from joystick axes (reference: controller.cpp:176-178; double pow path, -0.0f at axes[0]==0)
__device__ __forceinline__ float vel_cmd_component(const float* axes, int c) {
  const float a0 = axes[0], a1 = axes[1], a3 = axes[3];
  if (c == 0) return a1;
  if (c == 1) {
    const double sq = __dmul_rn((double)a0, (double)a0);
    const double sg = (a0 > 0.f) ? 1.0 : -1.0;
    return __double2float_rn(__dmul_rn(__dmul_rn(sq, sg), 0.8));
  }
  return __fmul_rn(a3, a1);
}

// one observation frame: term widths {3,3,3,12,12,12,4} at offsets {0,3,6,9,21,33,45}
__device__ __forceinline__ int frame_width(int t) { return t < 3 ? 3 : (t < 6 ? 12 : 4); }
__device__ __forceinline__ int frame_offset(int t) { return t < 3 ? 3 * t : (t < 6 ? 9 + 12 * (t - 3) : 45); }

// The newest-frame value of observation term t, component c (A1-A4).
__device__ __forceinline__ float current_term_value(int t, int c, const uint32_t* rw, const B1State* st,
                                                    const CtrlConst& cc) {
  const float* rf = reinterpret_cast<const float*>(rw);
  switch (t) {
    case 0: return gravity_component(rf + 0, c);
    case 1: return rf[4 + c];
    case 2: return rw[39] ? vel_cmd_component(rf + 31, c) : st->vel_cmd[c];
    case 3: return __double2float_rn(__dsub_rn((double)rf[7 + c], cc.q0[c]));          // controller.cpp:194-197
    case 4: return rf[19 + c];
    case 5: return st->action[c];
    default: {                                                                           // controller.hpp:99-103
      const int perm = c ^ 1;   // [1,0,3,2]
      return ((int)rw[35 + perm] >= cc.foot_threshold) ? 1.0f : 0.0f;
    }
  }
}

// One Gemm(+Elu) layer for a single row held in shared memory.  All kB1Threads threads call it.
//   N >= 32 : thread (g,o) accumulates a K-slice of output o from the k-group-major weights
//             (conflict-free float4 reads), slices are combined through shared memory in fixed order
//   N <  32 : one warp per output, lanes split K, warp-shuffle reduction
__device__ __forceinline__ void b1_layer(const DevLayer& L, const float* __restrict__ wk4, const float* __restrict__ wrm,
                                         const float* __restrict__ bias, const float* __restrict__ x,
                                         float* __restrict__ y, float* __restrict__ part, int tid) {
  const int K4 = L.Kp >> 2;
  const float4* x4 = reinterpret_cast<const float4*>(x);
  const int Nq = (L.N + 3) & ~3;
  if (L.N >= 32) {
    const int Npad = (L.N + 31) & ~31;
    if (Npad <= kB1Threads) {
      const int G = kB1Threads / Npad;
      const int g = tid / Npad, o = tid - g * Npad;
      const int per = (K4 + G - 1) / G;
      float acc = 0.f;
      if (g < G && o < L.N) {
        const int k0 = g * per, k1 = min(K4, k0 + per);
        const float4* w4 = reinterpret_cast<const float4*>(wk4);
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 8
        for (int k = k0; k < k1; ++k) {
          const float4 w = w4[k * L.N + o];
          const float4 xv = x4[k];
          a0 = fmaf(w.x, xv.x, a0); a1 = fmaf(w.y, xv.y, a1); a2 = fmaf(w.z, xv.z, a2); a3 = fmaf(w.w, xv.w, a3);
        }
        acc = (a0 + a1) + (a2 + a3);
      }
      if (g < G) part[g * Npad + o] = acc;
      block_sync();
      if (tid < Nq) {
        float s = 0.f;
        if (tid < L.N) {
          s = bias[tid];
          for (int gg = 0; gg < G; ++gg) s += part[gg * Npad + tid];
          if (L.has_elu) s = elu_exact(s, L.alpha);
        }
        y[tid] = s;
      }
    } else {
      for (int o = tid; o < Nq; o += kB1Threads) {
        float s = 0.f;
        if (o < L.N) {
          const float4* w4 = reinterpret_cast<const float4*>(wk4);
          float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 4
          for (int k = 0; k < K4; ++k) {
            const float4 w = w4[k * L.N + o];
            const float4 xv = x4[k];
            a0 = fmaf(w.x, xv.x, a0); a1 = fmaf(w.y, xv.y, a1); a2 = fmaf(w.z, xv.z, a2); a3 = fmaf(w.w, xv.w, a3);
          }
          s = bias[o] + ((a0 + a1) + (a2 + a3));
          if (L.has_elu) s = elu_exact(s, L.alpha);
        }
        y[o] = s;
      }
    }
  } else {
    const int warp = tid >> 5, lane = tid & 31;
    for (int o = warp; o < Nq; o += kB1Threads / 32) {
      float s = 0.f;
      if (o < L.N) {
        const float4* w4 = reinterpret_cast<const float4*>(wrm + (size_t)o * L.Kp);
        float a = 0.f;
        for (int k = lane; k < K4; k += 32) {
          const float4 w = w4[k];
          const float4 xv = x4[k];
          a = fmaf(w.x, xv.x, a); a = fmaf(w.y, xv.y, a); a = fmaf(w.z, xv.z, a); a = fmaf(w.w, xv.w, a);
        }
        a = warp_sum(a);
        s = a + bias[o];
        if (L.has_elu) s = elu_exact(s, L.alpha);
      }
      if (lane == 0) y[o] = s;
    }
  }
  block_sync();
}

// Fast GEMV for a 128-wide layer with the weights in shared memory (the resident kernel's case): 512 threads =
// 128 outputs x 4 K-groups.  Warp w owns outputs 8w..8w+7; lane = g*8 + j, so the 8 lanes of a quarter-warp read
// 128 contiguous bytes of the k-group-major weights (conflict-free LDS.128) and one broadcast float4 of x; the four
// partial sums of an output sit in lanes j, j+8, j+16, j+24 and are combined with two shuffles (fixed order).
__device__ __forceinline__ void b1_layer_n128(const float4* __restrict__ w4, const float* __restrict__ bias, int K4,
                                              bool has_elu, float alpha, const float4* __restrict__ x4,
                                              float* __restrict__ y, int tid) {
  const int lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 3, o = warp * 8 + (lane & 7);
  const int per = (K4 + 3) >> 2;
  const int k0 = g * per, k1 = min(K4, k0 + per);
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 4
  for (int k = k0; k < k1; ++k) {
    const float4 w = w4[k * 128 + o];
    const float4 xv = x4[k];
    a0 = fmaf(w.x, xv.x, a0); a1 = fmaf(w.y, xv.y, a1); a2 = fmaf(w.z, xv.z, a2); a3 = fmaf(w.w, xv.w, a3);
  }
  float s = (a0 + a1) + (a2 + a3);
  s += __shfl_xor_sync(0xffffffffu, s, 8);
  s += __shfl_xor_sync(0xffffffffu, s, 16);
  if (g == 0) {
    s += bias[o];
    if (has_elu) s = (s < 0.0f) ? alpha * (__expf(s) - 1.0f) : s;   // ex2.approx based: ~1e-6 relative, inside the 1e-5 budget
    y[o] = s;
  }
  block_sync();
}

// Register-resident weights for the Go2 topology (4 layers, hidden width 128, K0 <= 112, out <= 16): the 47 k fp32
// weights fit in the register file of one 512-thread CTA (96 per thread), so a control step reads no weight from
// shared memory at all -- only the 128-float activation vector, as warp-uniform (broadcast) float4 loads.
// Thread mapping for the hidden layers: warp w -> K-group g = w & 3, output block w >> 2; lane -> output inside the
// block.  K slices, accumulator interleave and the order in which the four partial sums are combined are exactly
// those of b1_layer_n128 / b1_layer, so all batch-1 variants produce identical bits.
struct B1RegWeights {
  float4 w0[7], w1[8], w2[8], w3;

  __host__ __device__ __forceinline__ static bool supported(const DevModel& m) {
    return m.n_layers == 4 && m.L[0].N == 128 && m.L[1].N == 128 && m.L[2].N == 128 && m.L[1].K == 128 && m.L[2].K == 128 &&
           m.L[3].K == 128 && m.L[3].N <= 16 && m.L[0].Kp <= 112;
  }
  __device__ __forceinline__ void load(const DevModel& m, int tid) {
    const int warp = tid >> 5, lane = tid & 31, g = warp & 3, o = (warp >> 2) * 32 + lane;
    const int K4_0 = m.L[0].Kp >> 2;
    const float4* s0 = reinterpret_cast<const float4*>(m.L[0].w_k4);
    const float4* s1 = reinterpret_cast<const float4*>(m.L[1].w_k4);
    const float4* s2 = reinterpret_cast<const float4*>(m.L[2].w_k4);
#pragma unroll
    for (int j = 0; j < 7; ++j) { const int k4 = g * 7 + j; w0[j] = (k4 < K4_0) ? s0[k4 * 128 + o] : make_float4(0.f, 0.f, 0.f, 0.f); }
#pragma unroll
    for (int j = 0; j < 8; ++j) { w1[j] = s1[(g * 8 + j) * 128 + o]; w2[j] = s2[(g * 8 + j) * 128 + o]; }
    w3 = (warp < m.L[3].N) ? reinterpret_cast<const float4*>(m.L[3].w_rm + (size_t)warp * m.L[3].Kp)[lane] : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  template <int kSteps>
  __device__ __forceinline__ static void hidden(const float4 (&w)[kSteps], const float* __restrict__ bias, bool has_elu, float alpha,
                                                const float* __restrict__ x, float* __restrict__ y, float* __restrict__ part, int tid) {
    const int warp = tid >> 5, lane = tid & 31, g = warp & 3, o = (warp >> 2) * 32 + lane;
    const float4* x4 = reinterpret_cast<const float4*>(x) + g * kSteps;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
    for (int j = 0; j < kSteps; ++j) {
      const float4 xv = x4[j];
      a0 = fmaf(w[j].x, xv.x, a0); a1 = fmaf(w[j].y, xv.y, a1); a2 = fmaf(w[j].z, xv.z, a2); a3 = fmaf(w[j].w, xv.w, a3);
    }
    part[g * 128 + o] = (a0 + a1) + (a2 + a3);
    block_sync();
    if (tid < 128) {
      float s = (part[tid] + part[128 + tid]) + (part[256 + tid] + part[384 + tid]);
      s += bias[tid];
      if (has_elu) s = (s < 0.0f) ? alpha * (__expf(s) - 1.0f) : s;
      y[tid] = s;
    }
    block_sync();
  }
  // xa: layer-0 input zero padded to 112 floats.  Returns the buffer holding the policy output.
  __device__ __forceinline__ float* forward(const DevModel& m, const float* __restrict__ bsm, float* xa, float* xb, float* part, int tid) const {
    hidden<7>(w0, bsm, m.L[0].has_elu != 0, m.L[0].alpha, xa, xb, part, tid);
    hidden<8>(w1, bsm + 128, m.L[1].has_elu != 0, m.L[1].alpha, xb, xa, part, tid);
    hidden<8>(w2, bsm + 256, m.L[2].has_elu != 0, m.L[2].alpha, xa, xb, part, tid);
    const int warp = tid >> 5, lane = tid & 31;
    if (warp < ((m.L[3].N + 3) & ~3)) {
      float s = 0.f;
      if (warp < m.L[3].N) {
        const float4 xv = reinterpret_cast<const float4*>(xb)[lane];
        float acc = 0.f;
        acc = fmaf(w3.x, xv.x, acc); acc = fmaf(w3.y, xv.y, acc); acc = fmaf(w3.z, xv.z, acc); acc = fmaf(w3.w, xv.w, acc);
        acc = warp_sum(acc);
        s = acc + bsm[384 + warp];
        if (m.L[3].has_elu) s = elu_exact(s, m.L[3].alpha);
      }
      if (lane == 0) xa[warp] = s;
    }
    block_sync();
    return xa;
  }
};

// Dynamic shared memory layout (floats): xa[XW] xb[XW] part[kB1Threads] raw[64] state weights...
__host__ __device__ inline int b1_xw(int max_width) { return ((max_width + 3) & ~3) + 4; }

template <bool kResident, bool kRegs = false>
__global__ void __launch_bounds__(kB1Threads, 1) b1_kernel(const B1Args a) {
  static_assert(kResident || !kRegs, "register-resident weights only make sense for the resident kernel");
  extern __shared__ __align__(16) float sm[];
  const int tid = threadIdx.x;
  const int XW = b1_xw(a.model.max_width);
  float* xa = sm;
  float* xb = xa + XW;
  float* part = xb + XW;
  uint32_t* rw = reinterpret_cast<uint32_t*>(part + kB1Threads);
  B1State* st = a.gstate;
  const float* wsm = nullptr;
  __shared__ uint32_t s_type;
  __shared__ uint64_t s_t0;
  __shared__ volatile int s_quit;

  if (kResident) {
    B1State* sst = reinterpret_cast<B1State*>(rw + 64);
    for (int i = tid; i < (int)(sizeof(B1State) / 4); i += kB1Threads)
      reinterpret_cast<uint32_t*>(sst)[i] = reinterpret_cast<const uint32_t*>(a.gstate)[i];
    st = sst;
    if (tid == 0) s_quit = 0;
    if (kRegs) {
      // biases of the four layers, 128 floats each (zero padded), right behind the state
      float* b = reinterpret_cast<float*>(sst + 1);
      for (int i = tid; i < 4 * 128; i += kB1Threads) {
        const DevLayer& L = a.model.L[i >> 7];
        b[i] = ((i & 127) < L.N) ? L.bias[i & 127] : 0.f;
      }
      wsm = b;
    } else if (a.weights_in_smem) {
      // weights (in the layout each layer reads) and biases become shared-memory resident for the
      // life of the kernel: a control step touches no global/HBM weight byte.
      float* w = reinterpret_cast<float*>(sst + 1);
      int off = 0;
      for (int l = 0; l < a.model.n_layers; ++l) {
        const DevLayer& L = a.model.L[l];
        const float* src = (L.N >= 32) ? L.w_k4 : L.w_rm;
        const int n = L.Kp * L.N;
        for (int i = tid * 4; i < n; i += kB1Threads * 4)
          *reinterpret_cast<float4*>(w + off + i) = *reinterpret_cast<const float4*>(src + i);
        off += n;
        const int nb = (L.N + 3) & ~3;
        for (int i = tid; i < nb; i += kB1Threads) w[off + i] = (i < L.N) ? L.bias[i] : 0.f;
        off += nb;
      }
      wsm = w;
    }
    block_sync();
  }

  B1RegWeights regw;
  if (kRegs) regw.load(a.model, tid);

  const int H = a.cc.H;
  const int n_obs = kFrame * H;
  // which observation element this thread assembles (loop invariant: hoisted out of the message loop).
  // term offsets H*{0,3,6,9,21,33,45}; widths {3,3,3,12,12,12,4}
  int t = 0, c = 0, wdt = 3;
  bool newest = false;
  if (tid < n_obs) {
    int off;
    if (tid < 9 * H) { t = tid / (3 * H); off = t * 3 * H; wdt = 3; }
    else if (tid < 45 * H) { t = 3 + (tid - 9 * H) / (12 * H); off = 9 * H + (t - 3) * 12 * H; wdt = 12; }
    else { t = 6; off = 45 * H; wdt = 4; }
    const int local = tid - off;
    const int f = local / wdt;
    c = local - f * wdt;
    newest = (f == H - 1);
  }

  for (;;) {
    // ---- ingest: every slot is polled by its own thread until its tag shows the next sequence number
    const uint32_t want = st->seq + 1u;
    uint32_t type = 0;
    if (tid < a.n_in_slots) {
      uint2 mw;
      if (kResident && a.idle_ns != 0ull) {
        uint32_t polls = 0;
        uint64_t idle0 = 0;
        for (;;) {
          mw = ld_mail(a.inbox + tid);
          if ((mw.y >> 3) == (want & 0x1FFFFFFFu) || s_quit) break;
          if (tid == 0 && (++polls & 0xFFu) == 0u) {
            const uint64_t now = globaltimer_ns();
            if (idle0 == 0) idle0 = now;
            else if (now - idle0 > a.idle_ns) { s_quit = 1; break; }
          }
        }
      } else {
        do { mw = ld_mail(a.inbox + tid); } while ((mw.y >> 3) != (want & 0x1FFFFFFFu));
      }
      type = mw.y & 7u;
      if (tid < 64) rw[tid] = mw.x;
      xa[tid] = __uint_as_float(mw.x);   // ACT payload == observation (overwritten for STEP); n_in_slots <= XW
    }
    // message type is uniform across slots; broadcast from thread 0 through shared memory
    if (tid == 0) { s_type = type; s_t0 = globaltimer_ns(); }
    block_sync();
    if (kResident && s_quit) {
      // idle farewell: state goes back to device memory, sequence number untouched -> a message that
      // raced with the timeout is served by the relaunched kernel
      for (int i = tid; i < (int)(sizeof(B1State) / 4); i += kB1Threads)
        reinterpret_cast<uint32_t*>(a.gstate)[i] = reinterpret_cast<const uint32_t*>(st)[i];
      __threadfence();
      block_sync();
      if (tid == 0) st_mail(a.outbox + kByeSlot, a.epoch, kByeTag);
      return;
    }
    type = s_type;
    const uint32_t tag = make_tag(want, type);

    if (type == MSG_EXIT) {
      if (tid == 0) st->seq = want;
      block_sync();
      if (kResident)
        for (int i = tid; i < (int)(sizeof(B1State) / 4); i += kB1Threads)
          reinterpret_cast<uint32_t*>(a.gstate)[i] = reinterpret_cast<const uint32_t*>(st)[i];
      if (tid == 0) st_mail(a.outbox, 0u, tag);
      return;
    }
    if (type == MSG_RESET || type == MSG_GAINS) {
      if (type == MSG_RESET) {                       // controller.hpp:132-162 initial member state
        for (int i = tid; i < kFrame * kMaxHistory; i += kB1Threads) st->obs[i] = 0.f;
        if (tid < 4) st->vel_cmd[tid] = 0.f;
        if (tid < kDof) st->action[tid] = 0.f;
      } else if (tid == 0) {                         // controller.cpp:254-277
        st->kp = __uint_as_float(rw[0]);
        st->kd = __uint_as_float(rw[1]);
      }
      if (tid == 0) { st->seq = want; st_mail(a.outbox, 0u, tag); }
      block_sync();
      if (!kResident) return;
      continue;
    }

    if (type == MSG_STEP) {
      // ---- A1-A6: term-major history shift + newest frame (controller.cpp:173-212)
      // the 49 newest-frame values are produced one term per warp (warp t, lane c): no intra-warp divergence between
      // the gravity projection, the double-precision vel_cmd / q - q0 paths and the plain copies
      {
        const int ft = tid >> 5, fc = tid & 31;
        if (ft < 7 && fc < frame_width(ft)) part[frame_offset(ft) + fc] = current_term_value(ft, fc, rw, st, a.cc);
      }
      block_sync();
      float v = 0.f;
      if (tid < n_obs) v = newest ? part[frame_offset(t) + c] : st->obs[tid + wdt];
      block_sync();
      if (tid < n_obs) {
        st->obs[tid] = v;
        xa[tid] = v;
        if (newest && t == 2) st->vel_cmd[c] = v;
      }
    }
    // zero the K padding of the first layer input
    if (tid >= a.model.in_dim && tid < (kRegs ? 112 : a.model.L[0].Kp)) xa[tid] = 0.f;
    block_sync();

    // ---- A7: Gemm/Elu chain
    float* x = xa;
    float* y = xb;
    int woff = 0;
    if (kRegs) x = regw.forward(a.model, wsm, xa, xb, part, tid);
    else for (int l = 0; l < a.model.n_layers; ++l) {
      const DevLayer& L = a.model.L[l];
      const float* wk4 = L.w_k4; const float* wrm = L.w_rm; const float* bias = L.bias;
      if (kResident && wsm) {
        wk4 = wrm = wsm + woff;
        bias = wsm + woff + L.Kp * L.N;
        woff += L.Kp * L.N + ((L.N + 3) & ~3);
      }
      if (L.N == 128) {   // same code (and bits) whether the weights sit in shared or global memory
        b1_layer_n128(reinterpret_cast<const float4*>(wk4), bias, L.Kp >> 2, L.has_elu != 0, L.alpha,
                      reinterpret_cast<const float4*>(x), y, tid);
        float* tmp = x; x = y; y = tmp;
        continue;
      }
      b1_layer(L, wk4, wrm, bias, x, y, part, tid);
      float* tmp = x; x = y; y = tmp;
    }
    // x now holds the policy output
    const uint64_t t1 = globaltimer_ns();
    const uint64_t dns = t1 - s_t0;
    if (type == MSG_ACT) {
      const int n = a.model.out_dim;
      if (tid < n) st_mail(a.outbox + tid, __float_as_uint(x[tid]), tag);
      if (tid == n) st_mail(a.outbox + n, (uint32_t)dns, tag);
      if (tid == n + 1) st_mail(a.outbox + n + 1, (uint32_t)(dns >> 32), tag);
    } else {
      // ---- A9 + A11 (controller.cpp:217-223, 235-248) and the ObservationAction payload
      MailWord* ob = a.outbox;
      const int button0 = (int)rw[40];
      if (tid < n_obs) st_mail(ob + tid, __float_as_uint(st->obs[tid]), tag);
      if (tid >= 416 && tid < 416 + kDof) {
        const int j = tid - 416;
        const float araw = x[j];
        const float act = clamp_mask(araw, a.cc.action_limit, button0);
        const double qd = joint_target(act, a.cc.q0[j], a.cc.action_scale);
        const unsigned long long qb = (unsigned long long)__double_as_longlong(qd);
        st_mail(ob + n_obs + j, __float_as_uint(araw), tag);
        st_mail(ob + n_obs + 12 + j, __float_as_uint(act), tag);
        st_mail(ob + n_obs + 24 + 2 * j, (uint32_t)qb, tag);
        st_mail(ob + n_obs + 24 + 2 * j + 1, (uint32_t)(qb >> 32), tag);
      }
      if (tid == 448) {
        const double kp = (double)((button0 == 0) ? st->kp : a.cc.kp_deadman);   // controller.cpp:246
        const double kd = (double)st->kd;
        const unsigned long long kpb = (unsigned long long)__double_as_longlong(kp);
        const unsigned long long kdb = (unsigned long long)__double_as_longlong(kd);
        st_mail(ob + n_obs + 48, (uint32_t)kpb, tag); st_mail(ob + n_obs + 49, (uint32_t)(kpb >> 32), tag);
        st_mail(ob + n_obs + 50, (uint32_t)kdb, tag); st_mail(ob + n_obs + 51, (uint32_t)(kdb >> 32), tag);
        st_mail(ob + n_obs + 52, (uint32_t)dns, tag); st_mail(ob + n_obs + 53, (uint32_t)(dns >> 32), tag);
      }
    }
    block_sync();
    if (type == MSG_STEP && tid < kDof) {
      // the published action feeds action_hist_ on the next step (controller.cpp:206)
      const float araw = x[tid];
      st->action[tid] = clamp_mask(araw, a.cc.action_limit, (int)rw[40]);
    }
    if (tid == 0) st->seq = want;
    block_sync();
    if (type == MSG_STEP && a.log) {
      // ObservationAction record of this step (controller.cpp:226-229): the observation as fed + the published action
      LogRing* lg = a.log;
      const unsigned long long head = lg->head;      // only this CTA writes it
      float* rec = lg->rec + (size_t)(head % lg->capacity) * kLogRecFloats;
      if (tid < n_obs) rec[tid] = st->obs[tid];
      if (tid >= 416 && tid < 416 + kDof) rec[n_obs + tid - 416] = st->action[tid - 416];
      __threadfence();
      block_sync();
      if (tid == 0) asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(&lg->head), "l"(head + 1ull) : "memory");
    }
    if (!kResident) return;
  }
}

// Bounded, self-driven variant for profilers: runs `steps` closed-loop steps on raw states read
// from device memory (cycled), no mailbox -- lets ncu report per-step DRAM bytes of the resident
// design (a kernel that never exits cannot be profiled).  Same device functions as b1_kernel.
template <bool kRegs>
__global__ void __launch_bounds__(kB1Threads, 1) b1_selfdriven_kernel(const B1Args a, const uint32_t* __restrict__ raws,
                                                                      int n_raws, int steps, float* __restrict__ out_actions) {
  extern __shared__ __align__(16) float sm[];
  const int tid = threadIdx.x;
  const int XW = b1_xw(a.model.max_width);
  float* xa = sm; float* xb = xa + XW; float* part = xb + XW;
  uint32_t* rw = reinterpret_cast<uint32_t*>(part + kB1Threads);
  B1State* st = reinterpret_cast<B1State*>(rw + 64);
  for (int i = tid; i < (int)(sizeof(B1State) / 4); i += kB1Threads)
    reinterpret_cast<uint32_t*>(st)[i] = reinterpret_cast<const uint32_t*>(a.gstate)[i];
  float* w = reinterpret_cast<float*>(st + 1);
  B1RegWeights regw;
  if (kRegs) {
    regw.load(a.model, tid);
    for (int i = tid; i < 4 * 128; i += kB1Threads) {
      const DevLayer& L = a.model.L[i >> 7];
      w[i] = ((i & 127) < L.N) ? L.bias[i & 127] : 0.f;
    }
  } else {
    int off = 0;
    for (int l = 0; l < a.model.n_layers; ++l) {
      const DevLayer& L = a.model.L[l];
      const float* src = (L.N >= 32) ? L.w_k4 : L.w_rm;
      const int n = L.Kp * L.N;
      for (int i = tid * 4; i < n; i += kB1Threads * 4)
        *reinterpret_cast<float4*>(w + off + i) = *reinterpret_cast<const float4*>(src + i);
      off += n;
      const int nb = (L.N + 3) & ~3;
      for (int i = tid; i < nb; i += kB1Threads) w[off + i] = (i < L.N) ? L.bias[i] : 0.f;
      off += nb;
    }
  }
  block_sync();
  const int H = a.cc.H, n_obs = kFrame * H;
  for (int s = 0; s < steps; ++s) {
    if (tid < kRawWords) rw[tid] = raws[(size_t)(s % n_raws) * kRawWords + tid];
    block_sync();
    float v = 0.f; int t = 0, c = 0, wdt = 3; bool newest = false;
    if (tid < n_obs) {
      int off;
      if (tid < 9 * H) { t = tid / (3 * H); off = t * 3 * H; wdt = 3; }
      else if (tid < 45 * H) { t = 3 + (tid - 9 * H) / (12 * H); off = 9 * H + (t - 3) * 12 * H; wdt = 12; }
      else { t = 6; off = 45 * H; wdt = 4; }
      const int local = tid - off; const int f = local / wdt; c = local - f * wdt;
      newest = (f == H - 1);
    }
    {
      const int ft = tid >> 5, fc = tid & 31;
      if (ft < 7 && fc < frame_width(ft)) part[frame_offset(ft) + fc] = current_term_value(ft, fc, rw, st, a.cc);
    }
    block_sync();
    if (tid < n_obs) v = newest ? part[frame_offset(t) + c] : st->obs[tid + wdt];
    block_sync();
    if (tid < n_obs) { st->obs[tid] = v; xa[tid] = v; if (newest && t == 2) st->vel_cmd[c] = v; }
    if (tid >= a.model.in_dim && tid < (kRegs ? 112 : a.model.L[0].Kp)) xa[tid] = 0.f;
    block_sync();
    float* x = xa; float* y = xb; int woff = 0;
    if (kRegs) x = regw.forward(a.model, w, xa, xb, part, tid);
    else for (int l = 0; l < a.model.n_layers; ++l) {
      const DevLayer& L = a.model.L[l];
      const float* wl = w + woff;
      if (L.N == 128) b1_layer_n128(reinterpret_cast<const float4*>(wl), wl + L.Kp * L.N, L.Kp >> 2, L.has_elu != 0, L.alpha,
                                    reinterpret_cast<const float4*>(x), y, tid);
      else b1_layer(L, wl, wl, wl + L.Kp * L.N, x, y, part, tid);
      woff += L.Kp * L.N + ((L.N + 3) & ~3);
      float* tmp = x; x = y; y = tmp;
    }
    if (tid < kDof) {
      const float act = clamp_mask(x[tid], a.cc.action_limit, (int)rw[40]);
      st->action[tid] = act;
      if (s == steps - 1) out_actions[tid] = act;
    }
    block_sync();
  }
}

}  // namespace go2p
