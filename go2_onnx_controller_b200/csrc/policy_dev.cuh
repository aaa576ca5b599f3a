// Device-side view of a parsed MLP policy + the controller constants, shared by all kernels.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace go2p {

constexpr int kMaxLayers = 8;
constexpr int kDof = 12;
constexpr int kFrame = 49;
constexpr int kMaxHistory = 8;

struct DevLayer {
  const float* w_rm;   // [N][Kp]        row-major, Kp = K rounded up to 4 (zero padded)
  const float* w_k4;   // [Kp/4][N][4]   k-group major: thread o reads float4 #(k4*N + o)
  const float* w_kn;   // [Kp8][Np]      k-major (transposed), Np = N rounded up to 128, Kp8 = K rounded up to 8
  const float* bias;   // [Np]           zero padded
  int K, Kp, N, Np, Kp8;
  int has_elu;
  float alpha;
};

struct DevModel {
  int n_layers, in_dim, out_dim, max_width;
  DevLayer L[kMaxLayers];
};

// reference constants (controller.hpp:13-16,100-103,119-120,165; controller.cpp:244,246)
struct CtrlConst {
  double q0[kDof];
  double action_scale;
  float action_limit;
  float kp_deadman;
  int foot_threshold;
  int H;
  float kp, kd;          // controller.hpp:119-120 (ROS parameters; go2p_set_gains)
};

// Everything publish() reads from the outside world for one robot and one control step (include/go2policy.h:
// go2p_raw_state), read through RawRecordRow below.
struct RawStateDev {
  float quat[4]; float gyro[3]; float q[12]; float dq[12]; float axes[4];
  int16_t foot_force[4]; int32_t joy_valid; int32_t button0;
};
static_assert(sizeof(RawStateDev) == 4 * 35 + 8 + 8, "must match go2p_raw_state");

// The same quantities as one array per field (include/go2policy.h: go2p_raw_fields), row-major, B rows each.  The flags
// are one byte: every reader compares them with 0.
struct RawFieldsDev {
  const float* quat;            // [B,4]
  const float* gyro;            // [B,3]
  const float* q;               // [B,12]
  const float* dq;              // [B,12]
  const float* axes;            // [B,4]
  const int16_t* foot_force;    // [B,4]
  const uint8_t* joy_valid;     // [B]
  const uint8_t* button0;       // [B]
};
// a tile of `rows` robots' fields packed one field after the other (quat, gyro, q, dq, axes, foot_force, joy_valid,
// button0): the shared-memory form.  For rows a multiple of 4 every field starts 16-byte aligned.
__host__ __device__ constexpr int raw_fields_tile_bytes(int rows) { return rows * (35 * 4 + 4 * 2 + 2); }
__host__ __device__ inline RawFieldsDev raw_fields_tile(const void* base, int rows) {
  const uint8_t* p = static_cast<const uint8_t*>(base);
  RawFieldsDev f;
  f.quat = reinterpret_cast<const float*>(p);
  f.gyro = f.quat + rows * 4;
  f.q = f.gyro + rows * 3;
  f.dq = f.q + rows * kDof;
  f.axes = f.dq + rows * kDof;
  f.foot_force = reinterpret_cast<const int16_t*>(f.axes + rows * 4);
  f.joy_valid = reinterpret_cast<const uint8_t*>(f.foot_force + rows * 4);
  f.button0 = f.joy_valid + rows;
  return f;
}

// One robot's raw state, read field by field: the only code that knows where a field sits in either layout.
// RawRecordRow: a go2p_raw_state record as 39 words (quat 0-3, gyro 4-6, q 7-18, dq 19-30, axes 31-34, foot_force 35-36
// as 4 x int16, joy_valid 37, button0 38); any 4-byte alignment.
struct RawRecordRow {
  const uint32_t* w;
  __device__ __forceinline__ float quat(int i) const { return reinterpret_cast<const float*>(w)[i]; }
  __device__ __forceinline__ float gyro(int i) const { return reinterpret_cast<const float*>(w)[4 + i]; }
  __device__ __forceinline__ float q(int i) const { return reinterpret_cast<const float*>(w)[7 + i]; }
  __device__ __forceinline__ float dq(int i) const { return reinterpret_cast<const float*>(w)[19 + i]; }
  __device__ __forceinline__ float axes(int i) const { return reinterpret_cast<const float*>(w)[31 + i]; }
  __device__ __forceinline__ int foot_force(int i) const { return (int)(int16_t)(uint16_t)(w[35 + (i >> 1)] >> (16 * (i & 1))); }
  __device__ __forceinline__ uint32_t joy_valid() const { return w[37]; }
  __device__ __forceinline__ uint32_t button0() const { return w[38]; }
};
// RawFieldRow: row r of a raw_fields_tile of kRows rows in shared memory; each group of 4 floats is one 16-byte load
// and the foot forces one 8-byte load (the compiler merges the loads of one group).
template <int kRows>
struct RawFieldRow {
  const void* tile;
  int r;
  __device__ __forceinline__ RawFieldsDev f() const { return raw_fields_tile(tile, kRows); }
  __device__ __forceinline__ static float pick(const float4& t, int i) { return (i & 3) == 0 ? t.x : (i & 3) == 1 ? t.y : (i & 3) == 2 ? t.z : t.w; }
  __device__ __forceinline__ float quat(int i) const { return pick(reinterpret_cast<const float4*>(f().quat)[r], i); }
  __device__ __forceinline__ float gyro(int i) const { return f().gyro[r * 3 + i]; }
  __device__ __forceinline__ float q(int i) const { return pick(reinterpret_cast<const float4*>(f().q)[r * 3 + (i >> 2)], i); }
  __device__ __forceinline__ float dq(int i) const { return pick(reinterpret_cast<const float4*>(f().dq)[r * 3 + (i >> 2)], i); }
  __device__ __forceinline__ float axes(int i) const { return pick(reinterpret_cast<const float4*>(f().axes)[r], i); }
  __device__ __forceinline__ int foot_force(int i) const {
    const short4 t = reinterpret_cast<const short4*>(f().foot_force)[r];
    return (int)((i & 3) == 0 ? t.x : (i & 3) == 1 ? t.y : (i & 3) == 2 ? t.z : t.w);
  }
  __device__ __forceinline__ uint32_t joy_valid() const { return f().joy_valid[r]; }
  __device__ __forceinline__ uint32_t button0() const { return f().button0[r]; }
};

// What Go2RobotInterface::send_command receives from publish() (controller.cpp:235-251), in UNITREE motor order:
// motor u = leg_u*3 + joint with legs FR, FL, RR, RL and joints hip, thigh, calf, while the policy works in Isaac order
// i = joint*4 + leg_i with legs FL, FR, RL, RR (controller.hpp:168-170) -- the same left/right swap as the foot
// contacts (controller.hpp:100-103).  dq_des and tau_ff are zero in the reference and are not stored.
struct MotorCmdDev {
  double q_des[kDof];
  double kp, kd;         // one value for all 12 joints (controller.cpp:246-247)
};
__host__ __device__ inline int motor_of_isaac(int i) { return (((i & 3) ^ 1) * 3) + (i >> 2); }


// CTA barrier that is safe after thread-divergent code.  Measured on B200 (driver 580, CUDA 12.9): when nvcc
// emits no reconvergence point between an `if (tid < n) {...}` and the following BAR.SYNC, a warp reaches the
// barrier in two pieces and each piece is counted as an arrival of the whole warp, which skews every later
// barrier of that warp by one phase (seen as stale shared-memory reads in the one-shot batch-1 kernel).
// Re-converging the warp first makes the arrival count exact.
__device__ __forceinline__ void block_sync() {
  __syncwarp();
  __syncthreads();
}

// std::clamp(a,-lim,lim) then a *= (button0==0)   (controller.cpp:218-223)
// NaN passes through the clamp (no fminf/fmaxf!), the multiply keeps the sign of zero.
__device__ __forceinline__ float clamp_mask(float a, float lim, int button0) {
  a = (a < -lim) ? -lim : ((lim < a) ? lim : a);
  return __fmul_rn(a, (button0 == 0) ? 1.0f : 0.0f);
}

// q_des = q0 + (double)a * scale   (controller.cpp:244) -- no contraction into an FMA
__device__ __forceinline__ double joint_target(float a, double q0, double scale) {
  return __dadd_rn(q0, __dmul_rn((double)a, scale));
}

// kp = button0 == 0 ? kp_ : 5, kd = kd_   (controller.cpp:246-247)
__device__ __forceinline__ void store_gains(MotorCmdDev* cmd, long long row, int button0, float kp, float kd, float kp_deadman) {
  cmd[row].kp = (double)((button0 == 0) ? kp : kp_deadman);
  cmd[row].kd = (double)kd;
}

// ONNX Elu-6: x < 0 ? alpha*(exp(x)-1) : x ; NaN and -0.0 pass through
__device__ __forceinline__ float elu_exact(float v, float alpha) {
  return (v < 0.0f) ? alpha * (expf(v) - 1.0f) : v;
}

}  // namespace go2p
