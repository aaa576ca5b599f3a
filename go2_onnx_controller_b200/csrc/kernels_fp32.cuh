// Batched policy forward in plain fp32 on the CUDA cores -- the path that has to agree with the
// reference's ONNX Runtime CPU execution to 1e-5 (reference: onnx_actor.cpp:38-48), for any layer
// widths.  One launch per Gemm(+Elu) layer; activations ping-pong through a scratch buffer that stays
// L2 resident for the chunk sizes the host uses.
//   sgemm_bias_act_kernel : C[M,N] = act(A[M,K] * W^T + b), 128x128x8 tiles, 8x8 register tiles,
//                           register-prefetched double buffering
//   small_out_kernel      : the narrow output layer (N <= 32) with the fused A9/A11 epilogue
//                           (clamp + dead-man mask, q_des; reference: controller.cpp:217-223,244)
//   assemble_batch_kernel : A1-A6 for B robots (reference: controller.cpp:173-212)
#pragma once
#include <algorithm>
#include "kernels_b1.cuh"
#include "policy_dev.cuh"

namespace go2p {

constexpr int kSgBM = 128, kSgBN = 128, kSgBK = 8, kSgThreads = 256;

// A: [M,K] row-major (lda), Wkn: [Kp8][Np] k-major zero padded, bias: [Np] zero padded, C: [M,N] (ldc)
__global__ void __launch_bounds__(kSgThreads, 2)
sgemm_bias_act_kernel(const float* __restrict__ A, int lda, const float* __restrict__ Wkn, int Np,
                      const float* __restrict__ bias, float* __restrict__ C, int ldc, int M, int K, int N,
                      int has_elu, float alpha) {
  __shared__ __align__(16) float As[2][kSgBK][kSgBM + 4];
  __shared__ __align__(16) float Bs[2][kSgBK][kSgBN];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;            // 16 x 16 threads, each an 8x8 tile (2x2 blocks of 4x4)
  const int row0 = blockIdx.x * kSgBM, col0 = blockIdx.y * kSgBN;
  // A loader: thread -> (row = tid/2, 4 consecutive k)   B loader: thread -> (k = tid/32, 4 consecutive n)
  const int a_r = tid >> 1, a_k = (tid & 1) * 4;
  const int b_k = tid >> 5, b_n = (tid & 31) * 4;
  const int Kt = (K + kSgBK - 1) / kSgBK;

  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  float ra[4];
  float4 rb;
  auto gload = [&](int kt) {
    const int k0 = kt * kSgBK;
    const int gr = row0 + a_r;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k0 + a_k + j;
      ra[j] = (gr < M && k < K) ? A[(size_t)gr * lda + k] : 0.f;
    }
    rb = *reinterpret_cast<const float4*>(Wkn + (size_t)(k0 + b_k) * Np + col0 + b_n);   // padded: always in range
  };
  auto sstore = [&](int buf) {
#pragma unroll
    for (int j = 0; j < 4; ++j) As[buf][a_k + j][a_r] = ra[j];
    *reinterpret_cast<float4*>(&Bs[buf][b_k][b_n]) = rb;
  };

  gload(0);
  sstore(0);
  block_sync();
  for (int kt = 0; kt < Kt; ++kt) {
    const int buf = kt & 1;
    if (kt + 1 < Kt) gload(kt + 1);
#pragma unroll
    for (int kk = 0; kk < kSgBK; ++kk) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[buf][kk][ty * 4]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[buf][kk][64 + ty * 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][kk][tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Bs[buf][kk][64 + tx * 4]);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    if (kt + 1 < Kt) {
      sstore(buf ^ 1);
      block_sync();
    }
  }
  // epilogue: rows {ty*4..+3, 64+ty*4..+3}, cols {tx*4..+3, 64+tx*4..+3}
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = row0 + ((i < 4) ? ty * 4 + i : 64 + ty * 4 + (i - 4));
    if (r >= M) continue;
#pragma unroll
    for (int jh = 0; jh < 2; ++jh) {
      const int c = col0 + jh * 64 + tx * 4;
      float o[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float v = acc[i][jh * 4 + j] + bias[c + j];
        if (has_elu) v = elu_exact(v, alpha);
        o[j] = v;
      }
      float* dst = C + (size_t)r * ldc + c;
      if (c + 3 < N && ((ldc & 3) == 0)) *reinterpret_cast<float4*>(dst) = make_float4(o[0], o[1], o[2], o[3]);
      else {
#pragma unroll
        for (int j = 0; j < 4; ++j) if (c + j < N) dst[j] = o[j];
      }
    }
  }
}

// Output layer with N <= 32: a CTA stages 128 rows of A in shared memory (odd pitch: conflict-free row
// walks), each thread owns one row and all N outputs; W (row-major [N][Kp]) is read as warp-uniform
// broadcasts.  Epilogue: bias (+ELU) (+clamp/mask) (+q_des).
constexpr int kSoRows = 128;
__global__ void __launch_bounds__(kSoRows, 1)
small_out_kernel(const float* __restrict__ A, int lda, const float* __restrict__ Wrm, int Kp,
                 const float* __restrict__ bias, float* __restrict__ C, int ldc, long long M, int K, int N,
                 int has_elu, float alpha, uint32_t flags, const int32_t* __restrict__ button0,
                 double* __restrict__ qdes, MotorCmdDev* __restrict__ cmd, CtrlConst cc) {
  extern __shared__ __align__(16) float so_sm[];
  const int pitch = K | 1;
  float* As = so_sm;                       // [128][pitch]
  float* Ws = so_sm + kSoRows * pitch;     // [N][Kp]
  const int tid = threadIdx.x;
  const long long row0 = (long long)blockIdx.x * kSoRows;
  const int rows = (int)min((long long)kSoRows, M - row0);
  for (int i = tid; i < rows * K; i += kSoRows) {
    const int r = i / K, k = i - r * K;
    As[r * pitch + k] = A[(size_t)(row0 + r) * lda + k];
  }
  for (int i = tid; i < N * Kp; i += kSoRows) Ws[i] = Wrm[i];
  block_sync();
  if (tid >= rows) return;
  const float* x = As + tid * pitch;
  float acc[32];
#pragma unroll
  for (int n = 0; n < 32; ++n) acc[n] = 0.f;
  for (int k = 0; k < K; ++k) {
    const float xv = x[k];
#pragma unroll
    for (int n = 0; n < 32; ++n)
      if (n < N) acc[n] = fmaf(xv, Ws[n * Kp + k], acc[n]);
  }
  const long long row = row0 + tid;
  const int b0 = (button0 && (flags & 5u)) ? button0[row] : 0;
  if ((flags & 4u) && cmd) store_gains(cmd, row, b0, cc.kp, cc.kd, cc.kp_deadman);
#pragma unroll
  for (int n = 0; n < 32; ++n) {
    if (n >= N) break;
    float v = acc[n] + bias[n];
    if (has_elu) v = elu_exact(v, alpha);
    if (flags & 1u) v = clamp_mask(v, cc.action_limit, b0);
    C[(size_t)row * ldc + n] = v;
    if (n < kDof && (flags & 6u)) {
      const double qd = joint_target(v, cc.q0[n], cc.action_scale);
      if ((flags & 2u) && qdes) qdes[(size_t)row * kDof + n] = qd;
      if ((flags & 4u) && cmd) cmd[row].q_des[motor_of_isaac(n)] = qd;
    }
  }
}

// Elementwise A9/A11 for models whose output layer is too wide for small_out_kernel.
__global__ void post_kernel(float* __restrict__ act, long long total, int out_dim, uint32_t flags,
                            const int32_t* __restrict__ button0, double* __restrict__ qdes, MotorCmdDev* __restrict__ cmd,
                            const __grid_constant__ CtrlConst cc) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long row = i / out_dim;
  const int n = (int)(i - row * out_dim);
  const int b0 = ((flags & 5u) && button0) ? button0[row] : 0;
  float v = act[i];
  if (flags & 1u) { v = clamp_mask(v, cc.action_limit, b0); act[i] = v; }
  if (n < kDof && (flags & 6u)) {
    const double qd = joint_target(v, cc.q0[n], cc.action_scale);
    if ((flags & 2u) && qdes) qdes[row * kDof + n] = qd;
    if ((flags & 4u) && cmd) cmd[row].q_des[motor_of_isaac(n)] = qd;
  }
  if (n == 0 && (flags & 4u) && cmd) store_gains(cmd, row, b0, cc.kp, cc.kd, cc.kp_deadman);
}

// A1-A6 for B robots: one thread per observation element, history kept in the obs rows themselves
// (term-major, oldest frame first; reference: controller.cpp:200-212).  The raw states are records (raw, kFields =
// false) or one array per field (fields, kFields = true; any natural alignment); both are read through the row
// accessors of policy_dev.cuh.

// button0_out (optional): the dead-man button of every robot as int32 [B], the form the batched epilogue reads.
// A warp takes 32 robots at a time:
//   1. their raw states (32 x 156 B of records, or 32 rows of every field) are copied to shared memory with coalesced
//      loads;
//   2. lane r evaluates the newest frame of robot r (49 values: gravity projection, gyro, command, q - q0, dq,
//      previous action, contacts) -- one robot per lane, so the scalar work of a robot is not replicated over a warp --
//      with the same device functions as the batch-1 kernel (kernels_b1.cuh), i.e. bit-identical results;
//   3. the warp walks the 32 observation rows: every lane reads its elements of a row (old frames from the row itself,
//      the newest frame from shared memory), then writes them back shifted -- coalesced 392-byte rows, no block
//      barrier, several rows of loads in flight.
// reset (optional, [B] bytes): a robot whose byte is non-zero starts from the controller's initial state
// (controller.hpp:132-162): its newest frame takes previous action 0 and, without joystick input, joystick command 0
// (written back), and its old-frame elements come out as 0 (selected: nothing the row held reaches the output).
constexpr int kAsmWarps = 4;
constexpr int kAsmRawWords = 39;                        // sizeof(RawStateDev) / 4
constexpr int kAsmRowsInFlight = 4;
static_assert(raw_fields_tile_bytes(32) <= 32 * kAsmRawWords * 4, "a warp's per-field tile fits its record stage");

template <class T>
__device__ __forceinline__ void asm_copy_rows(T* dst, const T* src, int n, int lane) {
  for (int i = lane; i < n; i += 32) dst[i] = src[i];
}

template <int kPerLane, bool kFields = false>
__global__ void __launch_bounds__(kAsmWarps * 32)
assemble_batch_kernel(const RawStateDev* __restrict__ raw, const float* __restrict__ prev_action,
                      float* __restrict__ vel_cmd, float* __restrict__ obs, long long B, CtrlConst cc,
                      int32_t* __restrict__ button0_out, const uint8_t* __restrict__ reset, const RawFieldsDev fields) {
  __shared__ __align__(16) uint32_t s_raw[kAsmWarps][32 * kAsmRawWords];
  __shared__ float s_new[kAsmWarps][32 * kFrame];
  const int H = cc.H, n_obs = kFrame * H;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  uint32_t* my_raw = s_raw[wid];
  float* my_new = s_new[wid];
  // element classification is row-independent.  meta = -1: no element; bit 8 set: old frame, low byte = distance
  // to the value to copy; else newest frame, low byte = index inside the 49-value frame
  int meta[kPerLane];
#pragma unroll
  for (int e = 0; e < kPerLane; ++e) {
    const int tid = e * 32 + lane;
    meta[e] = -1;
    if (tid < n_obs) {
      int t, off, wdt;
      if (tid < 9 * H) { t = tid / (3 * H); off = t * 3 * H; wdt = 3; }
      else if (tid < 45 * H) { t = 3 + (tid - 9 * H) / (12 * H); off = 9 * H + (t - 3) * 12 * H; wdt = 12; }
      else { t = 6; off = 45 * H; wdt = 4; }
      const int local = tid - off; const int f = local / wdt; const int c = local - f * wdt;
      meta[e] = (f != H - 1) ? (0x100 | wdt) : (frame_offset(t) + c);
    }
  }
  const long long n_groups = (B + 31) / 32;
  for (long long grp = (long long)blockIdx.x * kAsmWarps + wid; grp < n_groups; grp += (long long)gridDim.x * kAsmWarps) {
    const long long row0 = grp * 32;
    const int rows = (int)min(32LL, B - row0);
    // 1. raw states of the group -> shared memory (contiguous words, coalesced; per field: a raw_fields_tile of 32 rows)
    if constexpr (kFields) {
      const RawFieldsDev t = raw_fields_tile(my_raw, 32);
      asm_copy_rows(const_cast<float*>(t.quat), fields.quat + row0 * 4, rows * 4, lane);
      asm_copy_rows(const_cast<float*>(t.gyro), fields.gyro + row0 * 3, rows * 3, lane);
      asm_copy_rows(const_cast<float*>(t.q), fields.q + row0 * kDof, rows * kDof, lane);
      asm_copy_rows(const_cast<float*>(t.dq), fields.dq + row0 * kDof, rows * kDof, lane);
      asm_copy_rows(const_cast<float*>(t.axes), fields.axes + row0 * 4, rows * 4, lane);
      asm_copy_rows(const_cast<int16_t*>(t.foot_force), fields.foot_force + row0 * 4, rows * 4, lane);
      asm_copy_rows(const_cast<uint8_t*>(t.joy_valid), fields.joy_valid + row0, rows, lane);
      asm_copy_rows(const_cast<uint8_t*>(t.button0), fields.button0 + row0, rows, lane);
    } else {
      const uint32_t* gr = reinterpret_cast<const uint32_t*>(raw + row0);
      for (int i = lane; i < rows * kAsmRawWords; i += 32) my_raw[i] = gr[i];
    }
    const bool rst = reset != nullptr && lane < rows && reset[row0 + lane] != 0;   // lane r: row r's flag
    const uint32_t rst_rows = __ballot_sync(0xffffffffu, rst);                      // bit r: row r is reset
    __syncwarp();
    // 2. newest frame of robot (row0 + lane)
    if (lane < rows) {
      const long long row = row0 + lane;
      const auto rr = [&] {                                        // records: stride 39 words, conflict-free
        if constexpr (kFields) return RawFieldRow<32>{my_raw, lane};
        else return RawRecordRow{my_raw + lane * kAsmRawWords};
      }();
      float* nf = my_new + lane * kFrame;                          // stride 49 words: conflict-free
      float quat[4] = {rr.quat(0), rr.quat(1), rr.quat(2), rr.quat(3)};
      float g[3];
      gravity_all(quat, g);
      nf[0] = g[0]; nf[1] = g[1]; nf[2] = g[2];
#pragma unroll
      for (int c = 0; c < 3; ++c) nf[3 + c] = rr.gyro(c);
      const int joy_valid = (int)rr.joy_valid();
      float axes[4] = {rr.axes(0), rr.axes(1), rr.axes(2), rr.axes(3)};
      float cmd[3];
      if (joy_valid) {
#pragma unroll
        for (int c = 0; c < 3; ++c) { cmd[c] = vel_cmd_component(axes, c); vel_cmd[row * 3 + c] = cmd[c]; }
      } else if (rst) {
#pragma unroll
        for (int c = 0; c < 3; ++c) { cmd[c] = 0.f; vel_cmd[row * 3 + c] = 0.f; }
      } else {
#pragma unroll
        for (int c = 0; c < 3; ++c) cmd[c] = vel_cmd[row * 3 + c];
      }
#pragma unroll
      for (int c = 0; c < 3; ++c) nf[6 + c] = cmd[c];
#pragma unroll
      for (int c = 0; c < kDof; ++c) nf[9 + c] = __double2float_rn(__dsub_rn((double)rr.q(c), cc.q0[c]));
#pragma unroll
      for (int c = 0; c < kDof; ++c) nf[21 + c] = rr.dq(c);
      if (prev_action && !rst) {
        const float4* pa = reinterpret_cast<const float4*>(prev_action + row * kDof);
#pragma unroll
        for (int q = 0; q < 3; ++q) { const float4 t4 = pa[q]; nf[33 + 4 * q] = t4.x; nf[34 + 4 * q] = t4.y; nf[35 + 4 * q] = t4.z; nf[36 + 4 * q] = t4.w; }
      } else {
#pragma unroll
        for (int c = 0; c < kDof; ++c) nf[33 + c] = 0.f;
      }
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int p = c ^ 1;                                       // [1,0,3,2] (controller.hpp:99-103)
        nf[45 + c] = (rr.foot_force(p) >= cc.foot_threshold) ? 1.0f : 0.0f;
      }
      if (button0_out) button0_out[row] = (int32_t)rr.button0();
    }
    __syncwarp();
    // 3. shift + append, row by row, kAsmRowsInFlight rows of loads in flight
    for (int r0 = 0; r0 < rows; r0 += kAsmRowsInFlight) {
      float v[kAsmRowsInFlight][kPerLane];
#pragma unroll
      for (int i = 0; i < kAsmRowsInFlight; ++i) {
        const int r = r0 + i;
        if (r < rows) {
          const float* o = obs + (row0 + r) * n_obs;
          const bool old_zero = (rst_rows >> r) & 1u;              // reset row: its old frames are not read
#pragma unroll
          for (int e = 0; e < kPerLane; ++e) {
            const int mt = meta[e];
            v[i][e] = mt < 0 ? 0.f : ((mt & 0x100) ? (old_zero ? 0.f : o[e * 32 + lane + (mt & 0xff)]) : my_new[r * kFrame + mt]);
          }
        }
      }
      __syncwarp();      // every lane holds the old values of these rows before any lane overwrites them
#pragma unroll
      for (int i = 0; i < kAsmRowsInFlight; ++i) {
        const int r = r0 + i;
        if (r < rows) {
          float* o = obs + (row0 + r) * n_obs;
#pragma unroll
          for (int e = 0; e < kPerLane; ++e)
            if (meta[e] >= 0) o[e * 32 + lane] = v[i][e];
        }
      }
    }
    __syncwarp();        // shared buffers are reused by the next group
  }
}

// n_obs = 49*H floats per row: 4 elements per lane serve H <= 2, 13 serve H <= 8
// fields != null: the raw states come from these arrays instead of raw
inline void launch_assemble_batch(const RawStateDev* raw, const float* prev_action, float* vel_cmd, float* obs, long long B,
                                  const CtrlConst& cc, int32_t* button0_out, int sm_count, cudaStream_t st,
                                  const uint8_t* reset = nullptr, const RawFieldsDev* fields = nullptr) {
  const long long groups = (B + 31) / 32;
  const unsigned grid = (unsigned)std::min<long long>((groups + kAsmWarps - 1) / kAsmWarps, (long long)sm_count * 16);
  constexpr int kWide = (kFrame * kMaxHistory + 31) / 32;
  const RawFieldsDev f = fields ? *fields : RawFieldsDev{};
  const bool narrow = kFrame * cc.H <= 128;
  auto kernel = fields ? (narrow ? assemble_batch_kernel<4, true> : assemble_batch_kernel<kWide, true>)
                       : (narrow ? assemble_batch_kernel<4> : assemble_batch_kernel<kWide>);
  kernel<<<grid, kAsmWarps * 32, 0, st>>>(raw, prev_action, vel_cmd, obs, B, cc, button0_out, reset, f);
}

}  // namespace go2p
