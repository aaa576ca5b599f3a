// Batched policy forward on the 5th-gen tensor cores (tcgen05 + TMEM), one persistent CTA per SM.
//
//   A7  Gemm/Elu chain   reference: onnx_actor.cpp:38-48 (Ort::Session::Run), here for B rows at once
//   A9  clamp + mask     reference: controller.cpp:217-223   (optional fused epilogue)
//   A11 joint targets    reference: controller.cpp:244       (optional fused epilogue)
//
// Design (see DESIGN.md "tc_mlp_kernel"):
//   * all layer weights live in shared memory for the life of the CTA as 16-bit K-major UMMA
//     "interleaved" core matrices (packed once on the host at create time);
//   * observations stream in as 1-D bulk async copies (TMA engine) of whole 128-row slabs
//     ([128,in] fp32 is contiguous; its 392-byte row pitch rules out a 2-D tensor map) into a
//     2-stage shared-memory ring guarded by mbarriers;
//   * two 128-row tiles are in flight per CTA ("slots").  Each slot owns two 128-column TMEM buffers used
//     in ping-pong: layer l accumulates into one buffer; the epilogue warps read that accumulator with
//     tcgen05.ld, apply ELU, pack to 16 bit and write the result back IN PLACE (the first 16 columns of
//     every 32-column block) with tcgen05.st, where the next layer's tcgen05.mma reads it as its A
//     operand (TS form) while accumulating into the other buffer.  The activation never leaves the SM;
//   * A-operand readiness is one mbarrier per slot (16 arrivals = the 16 worker warps); the slot's control warp
//     waits for it and issues the layer's K steps back to back in a fixed order, so the fp32 accumulation order
//     (every output bit) does not depend on timing;
//   * the bias rides inside the MMA: every A operand carries two constant 1.0 columns and the weight
//     matrix two extra K rows holding hi/lo halves of the bias, so the epilogue has no bias add;
//   * the chain is evaluated in the base-2 exponent domain: layer l produces z' = log2(e)*z, the ELU is
//     h' = z' > 0 ? z' : c*(2^z' - 1) with c = alpha*log2(e), h' = log2(e)*h feeds the next layer whose weights
//     carry the inverse factor (folded on the host);
//   * fp16 path: the ELU runs on packed pairs -- F2FP (pack z'), ex2.approx.f16x2 of -|z'| (2 MUFU + PRMT), one
//     HFMA2 (c*e - c), one HMNMX2.NAN select max(z', e) when 0 <= alpha <= 1: 6 instructions per pair; four pairs in
//     sixteen take a packed-half polynomial 2^x on the FMA pipe instead (elu_neg_poly_f16x2): the MUFU (an ex2.f16x2 is
//     two MUFU.EX2.F16) is what an epilogue job saturates.  bf16 keeps the fp32 exponential;
//   * one elected thread issues every tcgen05.mma and signals completion with tcgen05.commit; ONE pool of 16 worker
//     warps walks the jobs of both slots alternately, so a slot's MMAs run while the pool works on the other slot.
#pragma once
#include "kernels_b1.cuh"      // gravity_all, vel_cmd_component: the same device functions as the batch-1 kernel
#include "policy_dev.cuh"
#include "ptx_sm100.cuh"

namespace go2p {

constexpr int kTcTileM = 128;
constexpr int kTcHidden = 128;     // every hidden width handled by this kernel
constexpr int kTcOutPad = 16;      // last layer N padded to 16 (smallest UMMA N at M=128)
constexpr int kTcBiasK = 16;       // extra K block carrying the two constant-one columns (bias hi / lo)
constexpr int kTcWorkers = 16;     // warps 0..15: one pool, 4 TMEM lane quarters (warp % 4) x 4 column blocks (warp / 4)
constexpr int kTcCtrlWarp0 = 16;      // warps 16,17: per-slot control warp = bulk-copy producer + MMA issuer; warp 16 owns TMEM
constexpr int kTcThreads = (kTcWorkers + 2) * 32;
constexpr int kTcSlotCols = 256;   // TMEM columns per slot: two 128-column ping-pong buffers
constexpr int kTcBlocks = 4;       // 32-column blocks per buffer, each with its own A-ready barrier

struct TcArgs {
  const float* obs;          // [B, in_dim]
  float* act;                // [B, out_dim]
  const int32_t* button0;    // [B] or null
  double* qdes;              // [B, 12] or null
  long long B;
  const uint16_t* wpack;     // per layer: N_l x Kp_l 16-bit, UMMA K-major interleaved layout (bias rows included)
  int n_layers, in_dim, k0p, out_dim;
  int has_elu[kMaxLayers];   // kEluNone / kEluSelect / kEluMax (elu_pack32; the output layer tests != 0 only)
  float elu_c[kMaxLayers];   // alpha * log2(e)
  float out_scale;           // ln(2) if the last layer has an ELU (its output is in the scaled domain), else 1
  uint32_t flags;
  float action_limit;
  double action_scale;
  double q0[kDof];
  MotorCmdDev* cmd;          // [B] send_command arguments in Unitree motor order (flag 4) or null
  float kp, kd, kp_deadman;
  // fp16 operands saturate at +-65504 where the fp32 reference does not (cvt.rn.satfinite): with flag 8 the kernel counts,
  // per launch, the (row, 32-column operand block) pairs in which at least one packed operand -- an observation or a
  // hidden activation -- sits at the largest finite magnitude.  0 = no operand was clipped on the way.
  unsigned long long* sat_count;
  // fused controller step (go2p_step_batch, tc_mlp_kernel<., true>): A1-A6 run in the conversion job.  obs_rw holds
  // every robot's history (== its previous observation) and is updated in place; act holds the previous published
  // action on entry (read by the assembly) and the new one on return; button0 comes from the raw state.
  const RawStateDev* raw;    // [B]
  float* obs_rw;             // [B, 49*H]  (== obs)
  float* vel_cmd;            // [B, 3] last joystick command (in/out)
  int H, foot_threshold;
  unsigned long long* trace;   // debug timeline (GO2P_TC_TRACE): [0] = count, then (event, clock64) pairs; CTA 0 only
  // fused step with resets (tc_mlp_kernel<., true, true>): [B] per-robot flags.  A robot whose byte is non-zero starts
  // this step from the controller's initial state (controller.hpp:132-162): older frames, previous action and stored
  // joystick command 0
  const uint8_t* reset;
  // fused step from per-field arrays (tc_mlp_kernel<., true, ., true>): read instead of raw, every pointer 16-byte aligned
  RawFieldsDev fields;
  // fused step over T steps (tc_mlp_kernel<., true, ., true, true>): fields and reset hold T*B rows, step-major; act,
  // obs_rw and vel_cmd are the state before step 0 on entry and after step T-1 on return.  Per-step outputs [T,B,.]:
  // act_seq (every published action), qdes_seq / cmd_seq / obs_seq (each may be null; flags 2 / 4 follow the first two)
  float* act_seq;
  double* qdes_seq;
  MotorCmdDev* cmd_seq;
  float* obs_seq;
  int T;
};

// kSeq: CTA-local unit i = 2p + s (slot s) is step p % T of the CTA's local tile 2 (p / T) + s -- a slot keeps its tile
// for all T steps (the host rounds a CTA's unit count up to whole pairs: an odd last tile is paired with a tile past the
// batch, which every job treats as a ragged tile without rows).  Otherwise unit i is local tile i, step 0.
template <bool kSeq>
__device__ __forceinline__ long long tc_unit_row0(const TcArgs& a, int i) {
  if constexpr (kSeq) i = 2 * ((i >> 1) / a.T) + (i & 1);
  return (blockIdx.x + (long long)i * gridDim.x) * kTcTileM;
}
template <bool kSeq>
__device__ __forceinline__ int tc_unit_step(const TcArgs& a, int i) { return kSeq ? (i >> 1) % a.T : 0; }

#ifdef GO2P_TC_TRACE
// store-only tracer: every tracing warp owns a 1024-entry lane of the buffer and a local counter (no atomics,
// so a trace point costs a clock read and one fire-and-forget store)
struct TcTracer {
  unsigned long long* base; uint32_t n;
  __device__ void init(const TcArgs& a, int warp) { base = (a.trace && blockIdx.x == 0) ? a.trace + (size_t)warp * 2048 : nullptr; n = 0; }
  __device__ __forceinline__ void put(uint32_t ev) {
    if (base && n < 1023) { base[2 * n] = ev; base[2 * n + 1] = (unsigned long long)clock64(); ++n; base[2046] = n; }
  }
};
#define TC_TRACE_INIT() TcTracer tracer; tracer.init(a, warp)
#define TC_TRACE(ev) tracer.put(ev)
#else
#define TC_TRACE_INIT() do { } while (0)
#define TC_TRACE(ev) do { } while (0)
#endif

// K extent of layer l's MMA (including the bias block) and its N
__host__ __device__ inline int tc_layer_kp(const TcArgs& a, int l) { return l == 0 ? a.k0p : kTcHidden + kTcBiasK; }
__host__ __device__ inline int tc_layer_n(const TcArgs& a, int l) { return l == a.n_layers - 1 ? kTcOutPad : kTcHidden; }
__host__ __device__ inline size_t tc_weight_bytes(const TcArgs& a) {
  size_t s = 0;
  for (int l = 0; l < a.n_layers; ++l) s += (size_t)tc_layer_kp(a, l) * tc_layer_n(a, l) * 2;
  return s;
}
__host__ __device__ inline size_t tc_stage_bytes(const TcArgs& a) { return ((size_t)kTcTileM * a.in_dim * 4 + 127) & ~(size_t)127; }
constexpr int kTcRawWords = 39;                               // sizeof(RawStateDev) / 4
constexpr int kTcRawStageBytes = kTcTileM * kTcRawWords * 4;    // fused step: one tile's raw states (128 x 156 B, contiguous)
static_assert(raw_fields_tile_bytes(kTcTileM) <= kTcRawStageBytes, "the per-field tile shares the raw stage");
__host__ __device__ inline size_t tc_smem_bytes(const TcArgs& a) {
  return tc_weight_bytes(a) + 2 * tc_stage_bytes(a) + 256 + 4 * kTcTileM * 4 + (a.raw || a.fields.quat ? kTcRawStageBytes : 0);
}

// does any half of these packed fp16 words sit at the largest finite magnitude (0x7BFF)?  (h & 0x7FFF) + 0x0401 reaches
// bit 15 exactly then (satfinite conversion never produces Inf; NaN payloads, 0x7C01.., are reported as well)
template <int kN>
__device__ __forceinline__ bool any_saturated_f16x2(const uint32_t (&w)[kN]) {
  uint32_t t = 0u;
#pragma unroll
  for (int j = 0; j < kN; ++j) t |= (w[j] & 0x7FFF7FFFu) + 0x04010401u;
  return (t & 0x80008000u) != 0u;
}

// ---- fused A1-A6: history shift + newest frame of one observation term, in place in the row's shared-memory copy
// (term-major layout, oldest frame first inside a term: controller.hpp:45-68, controller.cpp:200-212).  rst: the
// older frames are the initial state's zeros instead (selected, so whatever the row held -- NaN included -- is dropped)
template <int kW>
__device__ __forceinline__ void tc_shift_append(float* term, int H, const float (&cur)[kW], bool rst) {
#pragma unroll 1
  for (int f = 0; f + 1 < H; ++f) {
#pragma unroll
    for (int j = 0; j < kW; ++j) term[f * kW + j] = rst ? 0.f : term[(f + 1) * kW + j];
  }
#pragma unroll
  for (int j = 0; j < kW; ++j) term[(H - 1) * kW + j] = cur[j];
}

// Column block cb of a lane quarter updates "its" terms of row `srow` (robot `grow`): cb 0 gravity / angular velocity /
// joystick command, cb 1 joint positions, cb 2 joint velocities, cb 3 previous action / foot contacts (+ the dead-man
// button for the output job).  Bit-exact rules as in kernels_b1.cuh (same device functions).
// pa4 (cb 3) / vc (cb 0): the row's previous published action / last joystick command, loaded one job ahead.
// rst: the row's reset flag (every column block shifts terms, so every one needs it); a reset row's previous action
// and stored joystick command are 0, and without joystick input the 0 is written back as the row's command.
// rr: this robot's raw state (RawRecordRow: in the raw stage or, for a ragged tile, global memory; RawFieldRow: in the stage)
template <class Row>
__device__ __forceinline__ void tc_update_terms(const TcArgs& a, int cb, float* srow, const Row& rr, long long grow, int* button_out,
                                                const float4 (&pa4)[3], const float (&vc)[3], bool rst) {
  const int H = a.H;
  if (cb == 0) {
    const float quat[4] = {rr.quat(0), rr.quat(1), rr.quat(2), rr.quat(3)};
    float g[3];
    gravity_all(quat, g);
    const float w[3] = {rr.gyro(0), rr.gyro(1), rr.gyro(2)};
    float cmd[3];
    if (rr.joy_valid()) {                                // joy_ && !axes.empty() (controller.cpp:173)
      const float axes[4] = {rr.axes(0), rr.axes(1), rr.axes(2), rr.axes(3)};
#pragma unroll
      for (int c = 0; c < 3; ++c) { cmd[c] = vel_cmd_component(axes, c); a.vel_cmd[grow * 3 + c] = cmd[c]; }
    } else {
#pragma unroll
      for (int c = 0; c < 3; ++c) cmd[c] = rst ? 0.f : vc[c];
      if (rst) {
#pragma unroll
        for (int c = 0; c < 3; ++c) a.vel_cmd[grow * 3 + c] = 0.f;
      }
    }
    tc_shift_append<3>(srow, H, g, rst);
    tc_shift_append<3>(srow + 3 * H, H, w, rst);
    tc_shift_append<3>(srow + 6 * H, H, cmd, rst);
  } else if (cb == 1) {
    float q[kDof];
#pragma unroll
    for (int c = 0; c < kDof; ++c) q[c] = __double2float_rn(__dsub_rn((double)rr.q(c), a.q0[c]));   // controller.cpp:194-197
    tc_shift_append<kDof>(srow + 9 * H, H, q, rst);
  } else if (cb == 2) {
    float dq[kDof];
#pragma unroll
    for (int c = 0; c < kDof; ++c) dq[c] = rr.dq(c);
    tc_shift_append<kDof>(srow + 21 * H, H, dq, rst);
  } else {
    float pa[kDof];                                                               // previous published action
#pragma unroll
    for (int q = 0; q < 3; ++q) { const float4 t = pa4[q]; pa[4 * q] = t.x; pa[4 * q + 1] = t.y; pa[4 * q + 2] = t.z; pa[4 * q + 3] = t.w; }
    if (rst) {
#pragma unroll
      for (int c = 0; c < kDof; ++c) pa[c] = 0.f;
    }
    float ct[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int p = c ^ 1;                                                          // [1,0,3,2] (controller.hpp:99-103)
      ct[c] = (rr.foot_force(p) >= a.foot_threshold) ? 1.0f : 0.0f;
    }
    tc_shift_append<kDof>(srow + 33 * H, H, pa, rst);
    tc_shift_append<4>(srow + 45 * H, H, ct, rst);
    *button_out = (int)rr.button0();
  }
}
// L2 prefetch of one tile's per-field raw states (rows row0.. of a.fields, up to a.B; a sequence step's rows start foff
// rows in): thread m of the tile's 128 takes the m-th 128-byte line of every field's range (a field holds at most 48 B
// per row: 49 lines with misalignment).  A rolled loop over the fields, the pointers read from the kernel parameters: it
// runs where the pool holds the most registers.
__device__ __forceinline__ void tc_prefetch_fields(const TcArgs& a, long long row0, int m, long long foff = 0) {
  const long long rows = min((long long)kTcTileM, a.B - row0);
  static_assert(sizeof(RawFieldsDev) == 8 * sizeof(void*), "eight field pointers");
#pragma unroll 1
  for (int f = 0; f < 8; ++f) {
    // bytes per row, one byte per field: quat 16, gyro 12, q 48, dq 48, axes 16, foot_force 8, joy_valid 1, button0 1
    const long long row_bytes = (long long)((0x0101081030300C10ull >> (8 * f)) & 0xFFu);
    const uintptr_t lo = reinterpret_cast<uintptr_t>(reinterpret_cast<const void* const*>(&a.fields)[f]) + (uintptr_t)((row0 + foff) * row_bytes);
    const uintptr_t line = (lo & ~(uintptr_t)127) + (uintptr_t)m * 128u;
    if (line < lo + (uintptr_t)(rows * row_bytes)) ptx::prefetch_l2(reinterpret_cast<const void*>(line));
  }
}

// the term ranges (floats) column block cb owns in a row: [lo, hi)
__device__ __forceinline__ void tc_term_range(int cb, int H, int& lo, int& hi) {
  lo = cb == 0 ? 0 : cb == 1 ? 9 * H : cb == 2 ? 21 * H : 33 * H;
  hi = cb == 0 ? 9 * H : cb == 1 ? 21 * H : cb == 2 ? 33 * H : 49 * H;
}

// c*(2^x - 1) for x = -|z| <= 0 on a packed fp16 pair without the MUFU: clamp at -13 (2^-13 is below the resolution of
// the result; the -|.| rides on the clamp's HMNMX2 as a source modifier), split x = -k + r with the 1536 = 1.5*2^10
// rounding trick (k = 0..13 lands in the low mantissa bits of u), degree-3 polynomial for 2*2^r on [-0.5, 0.5] (p's
// exponent field is >= 15 > k, so the packed integer subtraction of k << 10 keeps the result normal and never borrows
// across the halves), then (c/2)*p - c as one HFMA2: 10 instructions after the pack, none on the MUFU.  Max abs error
// 9.1e-4 over all negative fp16 inputs vs 8.4e-4 for a correctly rounded 2^z followed by the same HFMA2; the max.NaN
// select of elu_pack16 keeps both bounds (exhaustive CPU emulation over every fp16 input, scripts/experiments/polyelu.py).
__device__ __forceinline__ uint32_t elu_neg_poly_f16x2(uint32_t z, uint32_t ch2, uint32_t nc2) {
  const uint32_t kM = 0x66006600u;                                              // (1536, 1536)
  const uint32_t xc = ptx::max_f16x2(ptx::negabs_f16x2(z), 0xCA80CA80u);      // max(-|z|, -13)
  const uint32_t u = ptx::sub_f16x2(kM, xc);                                    // 1536 + k, k = round(-xc)
  const uint32_t r = ptx::add_f16x2(xc, ptx::sub_f16x2(u, kM));
  uint32_t p = ptx::fma_f16x2(0x2F102F10u, r, 0x37C337C3u);   // 0.11035 r + 0.48511
  p = ptx::fma_f16x2(p, r, 0x3D8C3D8Cu);                      // ... + 1.38672
  p = ptx::fma_f16x2(p, r, 0x40004000u);                      // ... + 2.0
  p = ptx::mad_lo_u32(u & 0x000F000Fu, 0xFFFFFC00u, p);       // * 2^-k: p - (k << 10) per half, as LOP3 + IMAD
  return ptx::fma_f16x2(p, ch2, nc2);
}

// TcArgs::has_elu of a hidden layer: how elu_pack32 selects between z' and the exponential branch e' = c*2^-|z'| - c
enum : int {
  kEluNone = 0,
  kEluSelect = 1,   // z' < 0 ? e' : z' (HSET2 + LOP3): any alpha
  kEluMax = 2,      // max.NaN(z', e') (one HMNMX2): 0 <= alpha <= 1, where c*(2^z' - 1) >= z' for every z' <= 0
};

// bit j: column pair j of a warp's 16 per job takes the FMA-pipe exponential (4 of 16; DESIGN.md §3.2 lists every mask
// measured)
constexpr uint32_t kTcPolyMask = 0xC0C0u;

// ELU of 16 accumulator columns -> 8 packed words.  fp16: every pair stays packed -- F2FP (pack z'), then either
// ex2.approx.f16x2 of -|z'| (2 MUFU with the -|.| source modifier + PRMT) + HFMA2 (c*e - c) or, for the pairs in kMask,
// the FMA-pipe polynomial above; then the select.  kEluMax is exact: for z' > 0, e' < 0 < z'; for z' <= 0, e' is the
// ELU, which is >= z' when alpha <= 1 (where rounding puts the computed e' below z', z' is the closer of the two to the
// true value); max.NaN keeps a NaN input NaN.  bf16: the fp32 exponential of -|z| (its budget has no room for the fp16
// one) and the same select in bf16x2.  c2, ch2, nc2: c, c/2 and -c as packed fp16 pairs.
template <bool kFp16, int kElu, uint32_t kMask>
__device__ __forceinline__ void elu_pack16(const uint32_t (&v)[16], float c, uint32_t c2, uint32_t ch2, uint32_t nc2, uint32_t (&p)[8]) {
  const float nc = -c;
  if constexpr (kFp16) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint32_t zp = ptx::pack_f16_sat(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
      if constexpr (kElu == kEluNone) {
        p[j] = zp;
      } else {
        const uint32_t e = ((kMask >> j) & 1u) ? elu_neg_poly_f16x2(zp, ch2, nc2)
                                               : ptx::fma_f16x2(ptx::ex2_f16x2(ptx::negabs_f16x2(zp)), c2, nc2);
        p[j] = kElu == kEluMax ? ptx::max_nan_f16x2(zp, e) : ptx::select_neg_f16x2(zp, e);
      }
    }
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float z0 = __uint_as_float(v[2 * j]), z1 = __uint_as_float(v[2 * j + 1]);
      const uint32_t zp = ptx::pack_bf16(z0, z1);
      if constexpr (kElu == kEluNone) {
        p[j] = zp;
      } else {
        const uint32_t e = ptx::pack_bf16(fmaf(ptx::ex2_approx(-fabsf(z0)), c, nc), fmaf(ptx::ex2_approx(-fabsf(z1)), c, nc));
        p[j] = kElu == kEluMax ? ptx::max_nan_bf16x2(zp, e) : ptx::select_neg_bf16x2(zp, e);
      }
    }
  }
}
// a warp's whole job (32 columns = 16 pairs) under ONE branch on the layer's ELU: the compiler interleaves the two
// halves, so the MUFU queue of one half runs under the dependent tail (PRMT, HFMA2, select) of the other
template <bool kFp16, int kElu>
__device__ __forceinline__ void elu_pack32_sel(const uint32_t (&v0)[16], const uint32_t (&v1)[16], float c, uint32_t c2, uint32_t ch2,
                                               uint32_t nc2, uint32_t (&p)[16]) {
  uint32_t p0[8], p1[8];
  elu_pack16<kFp16, kElu, (kTcPolyMask & 0xFFu)>(v0, c, c2, ch2, nc2, p0);
  elu_pack16<kFp16, kElu, ((kTcPolyMask >> 8) & 0xFFu)>(v1, c, c2, ch2, nc2, p1);
#pragma unroll
  for (int j = 0; j < 8; ++j) { p[j] = p0[j]; p[8 + j] = p1[j]; }
}
template <bool kFp16>
__device__ __forceinline__ void elu_pack32(const uint32_t (&v0)[16], const uint32_t (&v1)[16], int elu, float c, uint32_t (&p)[16]) {
  const uint32_t c2 = ptx::pack_f16_sat(c, c), ch2 = ptx::pack_f16_sat(0.5f * c, 0.5f * c), nc2 = ptx::pack_f16_sat(-c, -c);
  if (elu == kEluMax) elu_pack32_sel<kFp16, kEluMax>(v0, v1, c, c2, ch2, nc2, p);
  else if (elu == kEluSelect) elu_pack32_sel<kFp16, kEluSelect>(v0, v1, c, c2, ch2, nc2, p);
  else elu_pack32_sel<kFp16, kEluNone>(v0, v1, c, c2, ch2, nc2, p);
}


// ---- cold paths, kept out of line so the steady-state loop of the kernel stays small in the instruction cache
// (measured: with everything inlined the kernel was 40 KB of SASS, above the 32 KB L1.5 instruction cache, and
// every phase of the 18-warp pipeline paid instruction-fetch misses: ~1000 cycles for a backward branch)

// ragged last tile, per-field raw states: row `grow`'s fields that column block cb reads (tc_update_terms), from global
// memory into row m of the raw stage, which then serves the row as for a full tile (the same thread reads them back)
__device__ __noinline__ void tc_stage_fields_row(const TcArgs& a, int cb, uint32_t* s_raw, long long grow, int m) {
  const RawFieldsDev t = raw_fields_tile(s_raw, kTcTileM), &g = a.fields;
  if (cb == 0) {
    const_cast<float4*>(reinterpret_cast<const float4*>(t.quat))[m] = reinterpret_cast<const float4*>(g.quat)[grow];
    for (int c = 0; c < 3; ++c) const_cast<float*>(t.gyro)[m * 3 + c] = g.gyro[grow * 3 + c];
    const_cast<float4*>(reinterpret_cast<const float4*>(t.axes))[m] = reinterpret_cast<const float4*>(g.axes)[grow];
    const_cast<uint8_t*>(t.joy_valid)[m] = g.joy_valid[grow];
  } else if (cb == 1 || cb == 2) {
    const float4* src = reinterpret_cast<const float4*>(cb == 1 ? g.q : g.dq) + grow * 3;
    float4* dst = const_cast<float4*>(reinterpret_cast<const float4*>(cb == 1 ? t.q : t.dq)) + m * 3;
    for (int j = 0; j < 3; ++j) dst[j] = src[j];
  } else {
    const_cast<short4*>(reinterpret_cast<const short4*>(t.foot_force))[m] = reinterpret_cast<const short4*>(g.foot_force)[grow];
    const_cast<uint8_t*>(t.button0)[m] = g.button0[grow];
  }
}

// layer-0 A operand of one row for a ragged last tile (read from global memory) or an odd input width
template <bool kFp16>
__device__ __noinline__ void tc_conv_slow(const TcArgs& a, const float* rowp, bool live, int c8_lo, int c8_hi, uint32_t a0_t) {
  for (int c8 = c8_lo; c8 < c8_hi; ++c8) {
    uint32_t q[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = c8 * 16 + 2 * j;
      float lo = 0.f, hi = 0.f;
      if (k < a.in_dim) { if (live) lo = rowp[k]; } else if (k <= a.in_dim + 1) lo = 1.f;
      if (k + 1 < a.in_dim) { if (live) hi = rowp[k + 1]; } else if (k + 1 <= a.in_dim + 1) hi = 1.f;
      q[j] = kFp16 ? ptx::pack_f16_sat(lo, hi) : ptx::pack_bf16(lo, hi);
    }
    ptx::tmem_st_x8(a0_t + (uint32_t)(32 * (c8 >> 1) + 8 * (c8 & 1)), q);
  }
}

// output epilogue for anything but the plain 12-output, no-activation case: one warp per lane quarter (half 0)
__device__ __noinline__ void tc_out_generic(const TcArgs& a, uint32_t o_t, long long row, bool live) {
  uint32_t v[16];
  ptx::tmem_ld_x16(o_t, v);
  ptx::tc_wait_ld();
  if (!live) return;
  const int L = a.n_layers - 1;
  const int b0 = (a.flags & 5u) && a.button0 ? a.button0[row] : 0;
  float* dst = a.act + row * a.out_dim;
#pragma unroll 1
  for (int j = 0; j < a.out_dim; ++j) {
    float x = __uint_as_float(v[0]);
#pragma unroll
    for (int q = 1; q < 16; ++q) if (q == j) x = __uint_as_float(v[q]);
    if (a.has_elu[L]) x = ((x < 0.f) ? fmaf(ptx::ex2_approx(x), a.elu_c[L], -a.elu_c[L]) : x) * a.out_scale;
    if (a.flags & 1u) x = clamp_mask(x, a.action_limit, b0);
    dst[j] = x;
    if (j < kDof && (a.flags & 6u)) {
      const double qd = joint_target(x, a.q0[j], a.action_scale);
      if ((a.flags & 2u) && a.qdes) a.qdes[row * kDof + j] = qd;
      if ((a.flags & 4u) && a.cmd) a.cmd[row].q_des[motor_of_isaac(j)] = qd;
    }
  }
  if ((a.flags & 4u) && a.cmd) store_gains(a.cmd, row, b0, a.kp, a.kd, a.kp_deadman);
}

// kReset (fused step only): the step reads a.reset.  A separate instantiation, so that the step without a mask runs
// exactly the code it ran before resets existed (the per-element selects cost 2 % even when every flag is 0).
// kFields (fused step only): the raw states come from a.fields (one array per field) instead of a.raw (records).
// kSeq (per-field fused step only): a.T consecutive steps (tc_unit_row0); each slot keeps its tile's observation stage in
// shared memory from step 0 to step T-1, and the previous action of step t+1 is the one step t left in that stage.
template <bool kFp16, bool kFused, bool kReset = false, bool kFields = false, bool kSeq = false>
__global__ void __launch_bounds__(kTcThreads, 1) tc_mlp_kernel(const __grid_constant__ TcArgs a) {
  static_assert(kFused || !kReset, "resets belong to the fused controller step");
  static_assert(kFused || !kFields, "per-field raw states belong to the fused controller step");
  static_assert(kFields || !kSeq, "the step sequence reads per-field raw states");
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  const size_t wbytes = tc_weight_bytes(a);
  const size_t stage_bytes = tc_stage_bytes(a);
  uint8_t* w_smem = smem;
  uint8_t* stage0 = smem + wbytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(stage0 + 2 * stage_bytes);
  uint64_t* obs_full = bars;        // [2]
  uint64_t* acc_full = bars + 4;    // [2]
  uint64_t* a_blk = bars + 6;       // [2][4], entry [s][0] used: A operand of slot s's next layer ready (16 arrivals)
  uint64_t* w_full = bars + 14;     // [kMaxLayers]  layer weights landed in shared memory (completes once)
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 14 + kMaxLayers);
  // fused step: ONE stage for the raw states of the tile whose conversion comes next (the two slots convert alternately)
  uint32_t* s_raw = reinterpret_cast<uint32_t*>(stage0 + 2 * stage_bytes + 256 + 4 * kTcTileM * 4);
  uint64_t* raw_full = bars + 2;    // raw states of CTA-local tile i landed (phase i & 1)
  int* s_button = reinterpret_cast<int*>(stage0 + 2 * stage_bytes + 256);   // [2 slots][2 tile parities][128] fused step: the rows' dead-man buttons
  // (the conversion of a slot's next tile may run, in the column block that has no output work, while the other column
  // blocks still read the current tile's buttons: consecutive tiles of a slot use different halves)

  // ---- one-time setup: barriers, TMEM; the weights arrive as one bulk async copy per layer, each with its own
  // mbarrier, so the first tile's conversion and layer-0 MMA do not wait for the deeper layers' weights (matters for
  // small batches, where a CTA sees a single tile)
  if (warp == kTcCtrlWarp0) {
    if (lane == 0) {
      for (int s = 0; s < 2; ++s) {
        ptx::mbar_init(&obs_full[s], 1);
        if (s == 0) ptx::mbar_init(raw_full, 1);
        ptx::mbar_init(&acc_full[s], 1);
        ptx::mbar_init(&a_blk[s * kTcBlocks], kTcWorkers);   // one A-ready barrier per slot: every worker warp arrives once per job
      }
      for (int l = 0; l < a.n_layers; ++l) ptx::mbar_init(&w_full[l], 1);
      ptx::fence_mbar_init();
      uint32_t off = 0;
      for (int l = 0; l < a.n_layers; ++l) {
        const uint32_t bytes = (uint32_t)(tc_layer_kp(a, l) * tc_layer_n(a, l) * 2);
        ptx::mbar_arrive_expect_tx(&w_full[l], bytes);
        ptx::bulk_g2s(w_smem + off, reinterpret_cast<const uint8_t*>(a.wpack) + off, bytes, &w_full[l]);
        off += bytes;
      }
    }
    __syncwarp();
    ptx::tmem_alloc<512>(tmem_ptr);
  }
  ptx::tc_fence_before();
  block_sync();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  // Programmatic dependent launch: everything above (barriers, TMEM, the weights' bulk copies) may run while the
  // previous kernel of the stream drains; observations are read and actions written only after that kernel has
  // completed.  The weights are read before the wait, so the previous kernel must not be one that writes them: the
  // host launches the first tensor-core kernel after a weight update (go2p_set_weights) on the update's stream without
  // programmatic serialization (capi.cu: launch_tc_t).  The next launch may start its own prologue as soon as
  // this CTA's SM is free (a short batch per GPU, e.g. 1/8 of a sharded step, is otherwise launch-gap bound).
  // While the previous kernel drains, pull this CTA's first two observation slabs into L2 (prefetch only: L2 is the
  // point of coherence, so a line the previous kernel still rewrites is simply updated there).  Matters for short
  // launches -- 1/8 of a sharded step is 7 tiles per CTA, and the first slab's HBM latency is part of every launch.
  {
    const long long tiles_all = (a.B + kTcTileM - 1) / kTcTileM;
    const long long slab_lines = ((long long)kTcTileM * a.in_dim * 4 + 127) / 128;
    for (int t = 0; t < 2; ++t) {
      const long long tile = blockIdx.x + (long long)t * gridDim.x;
      if (tile >= tiles_all) break;
      const uint8_t* base = reinterpret_cast<const uint8_t*>(a.obs + tile * kTcTileM * a.in_dim);
      const long long lim = min(slab_lines, (((a.B - tile * kTcTileM) * a.in_dim * 4) + 127) / 128);
      for (long long i = tid; i < lim; i += blockDim.x) ptx::prefetch_l2(base + i * 128);
    }
  }
  ptx::grid_dependency_wait();
  ptx::grid_launch_dependents();

  const long long n_tiles = (a.B + kTcTileM - 1) / kTcTileM;
  const int n_local = (int)((n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x);   // tiles b, b+G, ...
  const int n_units = kSeq ? 2 * a.T * ((n_local + 1) / 2) : n_local;              // (tile, step) units, see tc_unit_row0
  const uint32_t tile_bytes = (uint32_t)(kTcTileM * a.in_dim * 4);
  TC_TRACE_INIT();

  if (warp >= kTcCtrlWarp0) {
    // ================= control warp of slot s: bulk-copy producer + MMA issuer =================
    // One warp per slot walks that slot's tiles and layers: it waits for the A-ready barriers of the four 32-column
    // blocks and issues the layer's K steps back to back in a fixed order, which keeps the fp32 accumulation order
    // (every output bit) independent of timing.  Layer 0's first K step overwrites the buffer the previous tile's
    // output epilogue reads -- safe, because a warp signals its conversion block only after that read; at that
    // point the observation stage of this slot is free as well, so the next tile's bulk copy is issued right there.
    const int s = warp - kTcCtrlWarp0;
    const uint32_t fmt = kFp16 ? ptx::FMT_F16 : ptx::FMT_BF16;
    const uint32_t w_base = ptx::smem_u32(w_smem);
    uint64_t* blk = &a_blk[s * kTcBlocks];
    uint8_t* stage = stage0 + s * stage_bytes;
    uint32_t par = 0u;                       // all four block barriers of a slot advance one phase per layer
    auto load_tile = [&](int i) {            // i = CTA-local tile index (slot s owns i = s, s+2, ...)
      const long long row0 = tc_unit_row0<kSeq>(a, i);
      // kSeq: steps after the first find the stage as the slot's previous unit (the same tile) left it
      if (a.B - row0 >= kTcTileM && tc_unit_step<kSeq>(a, i) == 0) {
        TC_TRACE(0x100u | (uint32_t)s);
        ptx::mbar_arrive_expect_tx(&obs_full[s], tile_bytes);
        ptx::bulk_g2s(stage, a.obs + row0 * a.in_dim, tile_bytes, &obs_full[s]);
      } else {
        ptx::mbar_arrive(&obs_full[s]);      // ragged last tile: the pool reads global memory directly
      }
    };
    // fused step: tile i's raw states (contiguous 19,968 B, or one bulk copy per field: 19,200 B laid out as
    // raw_fields_tile) -> the raw stage; issued when conversion i-1 (the other slot's) has signalled, i.e. when every
    // warp is done with the stage
    auto load_raw = [&](int i) {
      const long long row0 = tc_unit_row0<kSeq>(a, i);
      if (a.B - row0 >= kTcTileM) {
        if constexpr (kFields) {
          const RawFieldsDev t = raw_fields_tile(s_raw, kTcTileM);
          const long long fr0 = row0 + (long long)tc_unit_step<kSeq>(a, i) * a.B;   // the step's rows of the fields
          ptx::mbar_arrive_expect_tx(raw_full, (uint32_t)raw_fields_tile_bytes(kTcTileM));
          ptx::bulk_g2s(const_cast<float*>(t.quat), a.fields.quat + fr0 * 4, kTcTileM * 4 * 4, raw_full);
          ptx::bulk_g2s(const_cast<float*>(t.gyro), a.fields.gyro + fr0 * 3, kTcTileM * 3 * 4, raw_full);
          ptx::bulk_g2s(const_cast<float*>(t.q), a.fields.q + fr0 * kDof, kTcTileM * kDof * 4, raw_full);
          ptx::bulk_g2s(const_cast<float*>(t.dq), a.fields.dq + fr0 * kDof, kTcTileM * kDof * 4, raw_full);
          ptx::bulk_g2s(const_cast<float*>(t.axes), a.fields.axes + fr0 * 4, kTcTileM * 4 * 4, raw_full);
          ptx::bulk_g2s(const_cast<int16_t*>(t.foot_force), a.fields.foot_force + fr0 * 4, kTcTileM * 4 * 2, raw_full);
          ptx::bulk_g2s(const_cast<uint8_t*>(t.joy_valid), a.fields.joy_valid + fr0, kTcTileM, raw_full);
          ptx::bulk_g2s(const_cast<uint8_t*>(t.button0), a.fields.button0 + fr0, kTcTileM, raw_full);
        } else {
          ptx::mbar_arrive_expect_tx(raw_full, (uint32_t)kTcRawStageBytes);
          ptx::bulk_g2s(s_raw, a.raw + row0, (uint32_t)kTcRawStageBytes, raw_full);
        }
      } else {
        ptx::mbar_arrive(raw_full);          // ragged last tile: the pool reads global memory directly
      }
    };
    if (s < n_units && ptx::elect_one_sync()) {
      load_tile(s);
      if (kFused && s == 0) load_raw(0);
    }
    __syncwarp();
    int phi = 0;
    for (int i = s; i < n_units; i += 2, phi ^= 1) {
      uint32_t w_off = 0;
      for (int l = 0; l < a.n_layers; ++l) {
        const int kp = tc_layer_kp(a, l), nl = tc_layer_n(a, l);
        const uint32_t idesc = ptx::make_idesc(fmt, kTcTileM, (uint32_t)nl);
        // K step of 16 elements = two 8x16B core matrices along K (LBO = 128 B apart); 8-row groups are
        // kp*16 B apart (SBO); consecutive K steps are 256 B apart (+16 in the descriptor's address field)
        const uint64_t bdesc0 = ptx::make_smem_desc_nosw(w_base + w_off, 128u, (uint32_t)kp * 16u);
        const uint32_t src = tmem_base + (uint32_t)s * kTcSlotCols + 128u * (uint32_t)((phi + l) & 1);
        const uint32_t dst = tmem_base + (uint32_t)s * kTcSlotCols + 128u * (uint32_t)((phi + l + 1) & 1);
        ptx::mbar_wait(&w_full[l], 0u);      // completes once; later waits return at the first probe
        if (l == 0) {
          ptx::mbar_wait(&blk[0], par);
          ptx::tc_fence_after();
          if (ptx::elect_one_sync()) {
            if (!kFused && i + 2 < n_units) load_tile(i + 2);
            if (kFused && i + 1 < n_units) load_raw(i + 1);
            TC_TRACE(0x200u | (uint32_t)(l << 4) | (uint32_t)s);
            const int ksteps = kp / 16;      // A chunk j sits at 32*(j/2) + 8*(j%2), ones inside the data
            for (int j = 0; j < ksteps; ++j)
              ptx::mma_f16_ts(dst, src + (uint32_t)(32 * (j >> 1) + 8 * (j & 1)), bdesc0 + (uint64_t)(j * 16), idesc, j > 0 ? 1u : 0u);
            ptx::mma_commit(&acc_full[s]);
            TC_TRACE(0x300u | (uint32_t)(l << 4) | (uint32_t)s);
            if constexpr (kFused) {
              // fused step: the stage now holds the tile's UPDATED observation rows (every pool warp fenced its
              // writes towards the async proxy before it signalled): send them back to the caller's history buffer
              // with one bulk copy, and refill the stage only when the copy has read it.  This warp has ~3,000
              // cycles until the slot's next MMA group; the pool never waits for the copy.
              const long long row0 = tc_unit_row0<kSeq>(a, i);
              if (a.B - row0 >= kTcTileM) {
                if constexpr (kSeq) {
                  // every step to obs_seq, the last one also to the history; the stage stays for the next step.  The
                  // output job of this step writes into the stage only after bulk_wait_read below: it waits for the
                  // output layer's commit, which this thread issues after it
                  const int t = tc_unit_step<kSeq>(a, i);
                  if (a.obs_seq) ptx::bulk_s2g(a.obs_seq + ((long long)t * a.B + row0) * a.in_dim, stage, tile_bytes);
                  if (t == a.T - 1) ptx::bulk_s2g(a.obs_rw + row0 * a.in_dim, stage, tile_bytes);
                } else {
                  ptx::bulk_s2g(a.obs_rw + row0 * a.in_dim, stage, tile_bytes);
                }
                ptx::bulk_wait_read();
              }
              if (i + 2 < n_units) load_tile(i + 2);
            }
          }
          __syncwarp();
        } else {
          // all four blocks, then the nine K steps back to back in the fixed order (block 0, bias, blocks 1..3).  The
          // 16 pool warps finish a job within ~300 cycles of each other, so issuing block by block gained nothing and
          // cost ~120 cycles of control-warp latency per MMA (wait + fence + elect per block) against ~55 when the
          // MMAs are issued in one go -- enough to make the pool wait for the accumulator at every job.
          ptx::mbar_wait(&blk[0], par);
          ptx::tc_fence_after();
          if (ptx::elect_one_sync()) {
            TC_TRACE(0x200u | (uint32_t)(l << 4) | (uint32_t)s);
#pragma unroll
            for (int cb = 0; cb < kTcBlocks; ++cb) {
              ptx::mma_f16_ts(dst, src + (uint32_t)(32 * cb), bdesc0 + (uint64_t)(2 * cb * 16), idesc, cb == 0 ? 0u : 1u);
              ptx::mma_f16_ts(dst, src + (uint32_t)(32 * cb + 8), bdesc0 + (uint64_t)((2 * cb + 1) * 16), idesc, 1u);
              if (cb == 0) ptx::mma_f16_ts(dst, src + 16u, bdesc0 + (uint64_t)(8 * 16), idesc, 1u);   // bias K step
            }
            ptx::mma_commit(&acc_full[s]);
            TC_TRACE(0x300u | (uint32_t)(l << 4) | (uint32_t)s);
          }
          __syncwarp();
        }
        par ^= 1u;
        w_off += (uint32_t)(kp * nl * 2);
      }
    }
  } else {
    // ================= worker warps: one pool of 16 warps walks the job list of both slots =================
    // pool = 4 TMEM lane quarters x 4 column blocks (warp = cb*4 + quarter): every warp owns one 32-column block.
    // Job order: see below (E jobs alternate between the slots, output and conversion jobs are interleaved).
    // While the pool works on one slot, the other slot's next-layer MMAs are issued and complete.
    const int quarter = warp & 3;            // TMEM lane quarter this warp may touch (== warp % 4)
    const int cb = warp >> 2;                // 32-column block
    const uint32_t lane_addr = ((uint32_t)(quarter * 32)) << 16;
    const int m = quarter * 32 + lane;       // row inside the tile
    const uint32_t one2 = kFp16 ? 0x3C003C00u : 0x3F803F80u;   // packed (1.0, 1.0)
    const int L = a.n_layers - 1;            // index of the output layer
    const bool out12 = a.out_dim == 12;
    const int n8 = a.k0p / 16;               // layer-0 A operand: chunks of 8 packed columns (16 elements)
    const bool even = (a.in_dim & 1) == 0;

    uint32_t par_acc[2] = {0u, 0u};
    uint32_t n_sat = 0u;                     // flag 8: (row, operand block) pairs with a saturated fp16 operand seen by this thread
    const bool masked = (a.flags & 5u) && a.button0 != nullptr;   // the clamp/mask and the kp selection read the button
    int b0_s0 = 0, b0_s1 = 0;                // dead-man buttons of this thread's row in the two slots' tiles
    // fused step: the row's previous published action (column block 3) / last joystick command (column block 0) for the
    // NEXT conversion job, requested in the output job that precedes it (global loads, ~1 us under load)
    float4 pf_act[3] = {make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f)};
    float pf_vel[3] = {0.f, 0.f, 0.f};
    bool pf_rst = false;                                  // kReset: the row's reset flag (every column block)
    auto prefetch_state = [&](int pair, int s) {          // for conv_job(pair, s)
      const long long row = tc_unit_row0<kSeq>(a, pair * 2 + s) + m;
      const int t = tc_unit_step<kSeq>(a, pair * 2 + s);
      pf_rst = false;
      if (row < a.B) {
        if constexpr (kReset) pf_rst = a.reset[row + (long long)t * a.B] != 0;
        if (cb == 3 && t == 0) {                           // kSeq, t > 0: the conversion reads it from the stage
          const float4* p4 = reinterpret_cast<const float4*>(a.act + row * kDof);
#pragma unroll
          for (int q = 0; q < 3; ++q) pf_act[q] = p4[q];
        } else if (cb == 0) {
#pragma unroll
          for (int c = 0; c < 3; ++c) pf_vel[c] = a.vel_cmd[row * 3 + c];
        }
      }
    };
    // ---- conv(s): fp32 observation rows -> 16-bit layer-0 A operand, constant ones at K = in_dim, in_dim+1.
    //      chunk c8 (16 K elements = 8 columns) lands at 32*(c8/2) + 8*(c8%2) of buffer phi: block cb = chunks 2cb, 2cb+1
    auto conv_job = [&](int pair, int s) {
      const int phi = pair & 1;
      const long long row0 = tc_unit_row0<kSeq>(a, pair * 2 + s);
      const int valid = (int)min((long long)kTcTileM, a.B - row0);
      const uint32_t a0_t = tmem_base + (uint32_t)s * kTcSlotCols + lane_addr + 128u * (uint32_t)phi;
      ptx::mbar_wait(&obs_full[s], (uint32_t)(pair & 1));
      TC_TRACE(0x400u | (uint32_t)s);
      const int c8_hi = min(n8, 2 * cb + 2);
      bool conv_sat = false;
      if constexpr (kFused) {
        // ---- A1-A6 (controller.cpp:173-212): the stage holds the tile's previous observations (== histories);
        // shift them by one frame and append the newest frame from the raw states, in place, then send the rows
        // back to the caller's history buffer with one bulk copy per lane quarter while the layers run
        float* srow = reinterpret_cast<float*>(stage0 + s * stage_bytes) + (size_t)m * a.in_dim;
        const bool full = valid == kTcTileM;
        ptx::mbar_wait(raw_full, (uint32_t)(s & 1));       // CTA-local tile i = 2*pair + s: phase i & 1
        TC_TRACE(0xA00u | (uint32_t)s);
        const int t = tc_unit_step<kSeq>(a, pair * 2 + s);
        if (m < valid) {
          int lo, hi;
          tc_term_range(cb, a.H, lo, hi);
          if constexpr (kSeq) {
            // the previous step's output job left the published action in the oldest frame of the action term
            if (cb == 3 && t > 0) {
              const float* pa = srow + 33 * a.H;
#pragma unroll
              for (int q = 0; q < 3; ++q) pf_act[q] = make_float4(pa[4 * q], pa[4 * q + 1], pa[4 * q + 2], pa[4 * q + 3]);
            }
          }
          if (!full) for (int k = lo; k < hi; ++k) srow[k] = a.obs_rw[(row0 + m) * a.in_dim + k];   // ragged tile: no bulk load
          if constexpr (kFields) {
            if (!full) tc_stage_fields_row(a, cb, s_raw, row0 + (long long)t * a.B + m, m);
            tc_update_terms(a, cb, srow, RawFieldRow<kTcTileM>{s_raw, m}, row0 + m, &s_button[(s * 2 + (pair & 1)) * kTcTileM + m], pf_act,
                            pf_vel, pf_rst);
          } else {
            const RawRecordRow rr{full ? s_raw + m * kTcRawWords : reinterpret_cast<const uint32_t*>(a.raw + row0 + m)};
            tc_update_terms(a, cb, srow, rr, row0 + m, &s_button[(s * 2 + (pair & 1)) * kTcTileM + m], pf_act, pf_vel,
                            pf_rst);
          }
          if (!full) for (int k = lo; k < hi; ++k) a.obs_rw[(row0 + m) * a.in_dim + k] = srow[k];
          if constexpr (kSeq) {
            if (!full && a.obs_seq)
              for (int k = lo; k < hi; ++k) a.obs_seq[((long long)t * a.B + row0 + m) * a.in_dim + k] = srow[k];
          }
        }
        TC_TRACE(0xB00u | (uint32_t)s);
        ptx::fence_proxy_async_smem();     // the control warp bulk-copies the stage to global memory once all warps signalled
        __syncwarp();
        asm volatile("bar.sync %0, 128;" ::"r"(1 + quarter) : "memory");       // the quarter's four column blocks: the
                                                                               // conversion below reads their columns
        TC_TRACE(0xC00u | (uint32_t)s);
      }
      if ((valid == kTcTileM || kFused) && even) {
        // full tile in shared memory, rows 8-byte aligned: vector loads, uniform per-pair classification
        const float2* r2 = reinterpret_cast<const float2*>(reinterpret_cast<const float*>(stage0 + s * stage_bytes) + (size_t)m * a.in_dim);
#pragma unroll 2
        for (int c8 = 2 * cb; c8 < c8_hi; ++c8) {
          uint32_t q[8];
          if (c8 * 16 + 16 <= a.in_dim) {
#pragma unroll
            for (int j = 0; j < 8; ++j) { const float2 t = r2[c8 * 8 + j]; q[j] = kFp16 ? ptx::pack_f16_sat(t.x, t.y) : ptx::pack_bf16(t.x, t.y); }
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int k = c8 * 16 + 2 * j;
              float2 t = make_float2(0.f, 0.f);
              if (k < a.in_dim) t = r2[k >> 1]; else if (k == a.in_dim) t = make_float2(1.f, 1.f);
              q[j] = kFp16 ? ptx::pack_f16_sat(t.x, t.y) : ptx::pack_bf16(t.x, t.y);
            }
          }
          ptx::tmem_st_x8(a0_t + (uint32_t)(32 * (c8 >> 1) + 8 * (c8 & 1)), q);
          if (kFp16 && a.sat_count && m < valid) conv_sat = conv_sat || any_saturated_f16x2(q);
        }
        n_sat += conv_sat ? 1u : 0u;
      } else {
        const float* rowp = (valid == kTcTileM || kFused) ? reinterpret_cast<const float*>(stage0 + s * stage_bytes) + (size_t)m * a.in_dim
                                                          : a.obs + (row0 + m) * a.in_dim;
        tc_conv_slow<kFp16>(a, rowp, m < valid, 2 * cb, c8_hi, a0_t);
      }
      ptx::tc_wait_st();
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&a_blk[s * kTcBlocks]);
      TC_TRACE(0x500u | (uint32_t)s);
    };

    // ---- out(s) (bias already inside the accumulator): (+ELU) (+clamp/mask) (+q_des) -> global
    auto out_job = [&](int pair, int s) {
      const int phi = pair & 1;
      const long long row0 = tc_unit_row0<kSeq>(a, pair * 2 + s);
      const int t = tc_unit_step<kSeq>(a, pair * 2 + s);
      const int valid = (int)min((long long)kTcTileM, a.B - row0);
      const uint32_t o_t = tmem_base + (uint32_t)s * kTcSlotCols + lane_addr + 128u * (uint32_t)((phi + 1 + L) & 1);
      ptx::mbar_wait(&acc_full[s], par_acc[s]);
      par_acc[s] ^= 1u;
      ptx::tc_fence_after();
      TC_TRACE(0x800u | (uint32_t)s);
      if (out12 && !a.has_elu[L]) {
        // the policy's case: 12 outputs, no activation -- column block cb < 3 stores one float4 of every row
        if (cb < 3) {
          uint32_t v[4];
          ptx::tmem_ld_x4(o_t + (uint32_t)(cb * 4), v);
          ptx::tc_wait_ld();
          if (m < valid) {
            const long long row = row0 + m + (long long)t * a.B;
            float o[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) o[j] = __uint_as_float(v[j]);
            if (a.flags & 1u) {
              // loaded two jobs ahead (see the E loop); fused step: taken from the raw state by the conversion job
              const int b0 = kFused ? s_button[(s * 2 + (pair & 1)) * kTcTileM + m] : (s ? b0_s1 : b0_s0);
#pragma unroll
              for (int j = 0; j < 4; ++j) o[j] = clamp_mask(o[j], a.action_limit, b0);
            }
            if constexpr (kSeq) {
              reinterpret_cast<float4*>(a.act_seq + row * 12)[cb] = make_float4(o[0], o[1], o[2], o[3]);
              if (t == a.T - 1) {
                reinterpret_cast<float4*>(a.act + (row0 + m) * 12)[cb] = make_float4(o[0], o[1], o[2], o[3]);
              } else {
                // the next step's previous action, into the oldest frame of the row's action term in the stage (that
                // conversion discards the frame; the bulk stores of this step's stage have been read, see the control
                // warp).  Not at the last step: the next tile's observations may be landing in the stage by then
                float* pa = reinterpret_cast<float*>(stage0 + s * stage_bytes) + (size_t)m * a.in_dim + 33 * a.H + cb * 4;
#pragma unroll
                for (int j = 0; j < 4; ++j) pa[j] = o[j];
              }
            } else {
              reinterpret_cast<float4*>(a.act + row * 12)[cb] = make_float4(o[0], o[1], o[2], o[3]);
            }
            if (a.flags & 6u) {
              double qd[4];
#pragma unroll
              for (int j = 0; j < 4; ++j) qd[j] = joint_target(o[j], a.q0[cb * 4 + j], a.action_scale);
              // kSeq: the step's slices of the per-step outputs (row includes t*B)
              if ((a.flags & 2u) && (kSeq ? a.qdes_seq : a.qdes)) {
                double2* q2 = reinterpret_cast<double2*>((kSeq ? a.qdes_seq : a.qdes) + row * kDof + cb * 4);
                q2[0] = make_double2(qd[0], qd[1]);
                q2[1] = make_double2(qd[2], qd[3]);
              }
              if ((a.flags & 4u) && (kSeq ? a.cmd_seq : a.cmd)) {
                // Isaac joint 4*cb + j = joint type cb of leg j -> Unitree motor (j ^ 1)*3 + cb
                MotorCmdDev* c = (kSeq ? a.cmd_seq : a.cmd) + row;
#pragma unroll
                for (int j = 0; j < 4; ++j) c->q_des[(j ^ 1) * 3 + cb] = qd[j];
                if (cb == 0) store_gains(kSeq ? a.cmd_seq : a.cmd, row, kFused ? s_button[(s * 2 + (pair & 1)) * kTcTileM + m] : (s ? b0_s1 : b0_s0), a.kp, a.kd, a.kp_deadman);
              }
            }
          }
        }
      } else if (cb == 0 && !kSeq) {          // kSeq serves the 12-output, no-activation case only (the host checks)
        tc_out_generic(a, o_t, row0 + m, m < valid);
      }
      ptx::tc_fence_before();
      TC_TRACE(0x900u | (uint32_t)s);
    };

    // Job order: conv(s0) conv(s1) of the first pair, then per pair  E(l,s0) E(l,s1) for every hidden layer |
    // out(s0) conv'(s0) out(s1) conv'(s1)  where conv' converts the NEXT pair's tile of that slot.  Interleaving the
    // output and conversion jobs of the two slots gives the output-layer MMA of slot 1 and the layer-0 MMA of slot 0
    // a whole job of cover each (they used to be waited for).  Hazards: conv'(s) writes the buffer that held A(L),
    // consumed by the MMA out(s) has just waited for; the layer-0 MMA of the new tile overwrites the buffer out(s)
    // reads, but it is issued only after ALL warps signalled conv'(s), i.e. after their out(s) reads.
    for (int s = 0; s < min(2, n_units); ++s) {
      if constexpr (kFused) prefetch_state(0, s);
      conv_job(0, s);
    }
    for (int pair = 0; pair * 2 < n_units; ++pair) {
      const int ns = min(2, n_units - pair * 2);
      const int ns_next = max(0, min(2, n_units - (pair + 1) * 2));
      const int phi = pair & 1;

      // ---- E(l,s): accumulator block -> ELU -> 16-bit A operand of the next layer, in place
      for (int l = 0; l < L; ++l) {
        const int elu = a.has_elu[l];
        const float c = a.elu_c[l];
        if (l == L - 1 && masked) {
          // the output jobs of this pair need the rows' dead-man buttons: request them two jobs ahead, so the global
          // load is not waited for in the output job (it was 9 % of the pool's time)
          const long long r0 = (blockIdx.x + (long long)(pair * 2) * gridDim.x) * kTcTileM + m;
          const long long r1 = r0 + (long long)gridDim.x * kTcTileM;
          b0_s0 = r0 < a.B ? __ldg(a.button0 + r0) : 0;
          b0_s1 = r1 < a.B ? __ldg(a.button0 + r1) : 0;
        }
        if constexpr (kFused) {
          if (l == 0) {
            // the next pair's conversion jobs read these robots' raw states and previous actions: pull them into L2 now,
            // two layers ahead (no registers held, nothing waited for)
            const long long r0 = tc_unit_row0<kSeq>(a, pair * 2 + 2 + (cb & 1)) + m;
            if (r0 < a.B) {
              if (cb < 2) {
                if constexpr (kFields) tc_prefetch_fields(a, r0 - m, m, (long long)tc_unit_step<kSeq>(a, pair * 2 + 2 + (cb & 1)) * a.B);
                else { ptx::prefetch_l2(a.raw + r0); ptx::prefetch_l2(reinterpret_cast<const uint8_t*>(a.raw + r0) + sizeof(RawStateDev) - 1); }
              }
              else { ptx::prefetch_l2(a.act + r0 * kDof); ptx::prefetch_l2(a.vel_cmd + r0 * 3); }
            }
          }
        }
        for (int s = 0; s < ns; ++s) {
          const uint32_t d_t = tmem_base + (uint32_t)s * kTcSlotCols + lane_addr + 128u * (uint32_t)((phi + 1 + l) & 1) + (uint32_t)(cb * 32);
          ptx::mbar_wait(&acc_full[s], par_acc[s]);
          par_acc[s] ^= 1u;
          ptx::tc_fence_after();
          TC_TRACE(0x600u | (uint32_t)(l << 4) | (uint32_t)s);
          // the block's 32 accumulator columns in two loads, the 16 packed words in one store, in place: they land on
          // columns 0..15, whose accumulator values are already in registers
          uint32_t cur[16], nxt[16];
          ptx::tmem_ld_x16(d_t, cur);
          ptx::tmem_ld_x16(d_t + 16u, nxt);
          ptx::tc_wait_ld();
          TC_TRACE(0xF00u | (1u << 4) | (uint32_t)s);
          uint32_t pk[16];
          elu_pack32<kFp16>(cur, nxt, elu, c, pk);
          TC_TRACE(0xF00u | (3u << 4) | (uint32_t)s);
          ptx::tmem_st_x16(d_t, pk);
          if (kFp16 && a.sat_count) n_sat += any_saturated_f16x2(pk) ? 1u : 0u;
          if (cb == 0) {   // constant-one columns (K = 128,129; zeros up to 143) in the dead half of block 0
            const uint32_t ones[8] = {one2, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
            ptx::tmem_st_x8(d_t + 16u, ones);
          }
          ptx::tc_wait_st();
          TC_TRACE(0xF00u | (4u << 4) | (uint32_t)s);
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&a_blk[s * kTcBlocks]);
          TC_TRACE(0x700u | (uint32_t)(l << 4) | (uint32_t)s);
        }
      }

      for (int s = 0; s < ns; ++s) {
        if constexpr (kFused) { if (s < ns_next) prefetch_state(pair + 1, s); }   // lands while the output job runs
        out_job(pair, s);
        // With an even number of hidden layers the output accumulator shares its TMEM buffer with the next tile's
        // layer-0 operand: the four warps of a lane quarter (the only ones touching these lanes) meet before any of
        // them converts the next tile, so no conversion store can overtake a sibling's output read.  (Odd counts --
        // the Go2 policy -- use the other buffer and skip this.)
        // kSeq: the same meeting orders the action stores of column blocks 0-2 into the stage before column block 3's
        // read of them in the conversion of the tile's next step.
        if (kSeq || (L & 1) == 0) {
          __syncwarp();
          asm volatile("bar.sync %0, 128;" ::"r"(1 + quarter) : "memory");
        }
        if (s < ns_next) conv_job(pair + 1, s);
      }
    }
    if (kFp16 && a.sat_count) {
      uint32_t n = n_sat;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
      if (lane == 0 && n) atomicAdd(a.sat_count, (unsigned long long)n);
    }
  }

  // ---- teardown
  if constexpr (kFused) ptx::bulk_wait_all();      // this thread's bulk stores of updated observation rows are complete
  ptx::tc_fence_before();
  block_sync();
  if (warp == kTcCtrlWarp0) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<512>(tmem_base);
  }
}

}  // namespace go2p
