// Batched forward for policies whose layers are too wide for the all-in-shared-memory kernel (kernels_tc.cuh), e.g.
// BASELINE.json configs[4]: 245 -> 1024 -> 512 -> 256 -> 12 with a 5-frame observation history.
//
//   A7  Gemm/Elu chain   reference: onnx_actor.cpp:38-48 (Ort::Session::Run), one tcgen05 GEMM launch per layer
//   A9/A11 epilogue      reference: controller.cpp:217-223,244 (fused into the last layer's epilogue)
//
// Design:
//   * activations travel between layers as 16-bit values in a TILE-BLOCKED layout in global memory (they stay L2
//     resident for the chunk sizes the host uses): tiles of 128 rows x 64 K-columns, each tile stored exactly as the
//     UMMA K-major no-swizzle core-matrix image the tensor core reads from shared memory (8x8-element cores of 128
//     contiguous bytes, K-adjacent cores contiguous, 8-row groups 1024 B apart).  A tile is therefore ONE contiguous
//     16 KB chunk: a single 1-D bulk async copy (TMA engine) brings it in, no tensor map and no relayout;
//   * weights are packed on the host the same way per (N-tile, K-chunk);
//   * wide_gemm_kernel: persistent CTAs over (row tile, N tile); warp 0 = producer (3-stage mbarrier ring of A/B
//     chunks), warp 1 = MMA issuer (SS-form tcgen05.mma, M=128, N=NT, four K steps per 64-wide chunk, accumulators
//     double-buffered in TMEM so the epilogue of one tile overlaps the MMAs of the next), warps 2-17 = epilogue
//     (tcgen05.ld -> +bias -> ELU -> 16-bit -> blocked store for the next layer, or the fused A9/A11 output epilogue);
//   * obs_to_blocked_kernel converts the fp32 [B,in] observations into the blocked 16-bit layout (zero padded).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <string>
#include <vector>

#include "onnx_reader.hpp"
#include "policy_dev.cuh"
#include "ptx_sm100.cuh"

namespace go2p {

constexpr int kWdTileM = 128;
constexpr int kWdChunkK = 64;                       // K columns per pipeline stage (4 MMA K steps)
constexpr int kWdATileBytes = kWdTileM * kWdChunkK * 2;   // 16 KB
// operand ring depth: as many stages as fit in ~192 KB (the L2 round trip under load is ~4,000 cycles, so the bytes in
// flight, not the stage count, set the delivered bandwidth), at most 8.  split: a stage holds three bf16 pieces of each
// operand (GO2P_PREC_FP32_TC)
__host__ __device__ constexpr int wd_stages(int nt, bool split) {
  const int stage = (split ? 3 : 1) * (128 * 64 * 2 + nt * 64 * 2);
  const int n = (192 * 1024) / stage;
  return n > 8 ? 8 : n;
}
constexpr int kWdEpiWarps = 16;                     // kWdEpiWarps/4 per TMEM lane quarter, each takes a share of the tile's columns
constexpr int kWdEpiParts = kWdEpiWarps / 4;
constexpr int kWdThreads = (2 + kWdEpiWarps) * 32;  // producer, MMA issuer, epilogue warps

// byte offset of element (r, c) inside a [rows x 64] blocked tile (rows multiple of 8)
__host__ __device__ inline uint32_t wd_tile_offset(int r, int c) {
  return (uint32_t)(((r >> 3) * 8 + (c >> 3)) * 128 + (r & 7) * 16 + (c & 7) * 2);
}

// ---- GO2P_PREC_FP32_TC: every fp32 operand as three bf16 pieces (DESIGN.md §3.3c).  A split tile group is the hi, mid
// and lo tiles of one (row or N tile, K chunk), 16-bit blocked images as above, stored one after the other.
//
// Activations (the A operand): x = h + m + l, h = bf16_rn(x), m = bf16_rn(x - h), l = x - h - m (exact in bf16): 24
// significand bits, fp32's exponent range.  +-Inf and NaN ride in h alone with m = l = 0 (x - h would be NaN); a finite
// x beyond bf16's largest finite value is truncated into h instead of rounding to Inf.
__device__ __forceinline__ void wd_split_act(float x, float& h, float& m, float& l) {
  const bool fin = fabsf(x) <= 3.40282347e38f;
  float t = __bfloat162float(__float2bfloat16_rn(x));
  if (fin && isinf(t)) t = __bfloat162float(__float2bfloat16_rz(x));
  const float r = fin ? __fsub_rn(x, t) : 0.f;
  h = t;
  m = __bfloat162float(__float2bfloat16_rn(r));
  l = __fsub_rn(r, m);
}

// Weights (the B operand): W = h + m + l with h = bf16_rz(W), m = bf16_rz(W - h), l = W - h - m, so every piece has W's
// sign, and for W != 0 a piece that would be 0 holds bf16_rz(W * 2^-32) instead (2^-32 of W: far below the contract).
// An Inf activation then meets three products of one sign and no zero -- Inf * W stays +-Inf as in the reference instead
// of turning into Inf - Inf or Inf * 0 = NaN.  Every operation is exact, so the host packer and the device packer
// (kernels_pack.cuh) agree bit for bit without explicit rounding modes.
__host__ __device__ inline void wd_split_weight(float w, uint16_t p[3]) {
  const __nv_bfloat16 h = __float2bfloat16_rz(w);
  const float r = w - __bfloat162float(h);
  const __nv_bfloat16 m = __float2bfloat16_rz(r);
  const __nv_bfloat16 l = __float2bfloat16_rz(r - __bfloat162float(m));
  const uint16_t tiny = __bfloat16_as_ushort(__float2bfloat16_rz(w * 0x1p-32f));
  const bool nz = w != 0.f;
  p[0] = __bfloat16_as_ushort(h);
  p[1] = (nz && __bfloat162float(m) == 0.f) ? tiny : __bfloat16_as_ushort(m);
  p[2] = (nz && __bfloat162float(l) == 0.f) ? tiny : __bfloat16_as_ushort(l);
}

struct WideLayerDev {
  const uint16_t* w[2];    // [0] bf16, [1] fp16: per (n tile, k chunk) blocked image, NT rows x 64 (null for a model
                           // the one-launch kernel serves: only the split images are built for it)
  const uint16_t* w3;      // GO2P_PREC_FP32_TC: per (n tile, k chunk) the hi, mid and lo bf16 images, NT3 rows x 64 each
  const float* bias;       // [Npad]
  int K, N, Kp, Np, NT;    // Kp multiple of 64, Np multiple of NT
  int NT3;                 // N tile of the split images (Np is a multiple of it too)
  int has_elu;
  float alpha;
};

struct WideModel {
  int n_layers = 0;
  int in_dim = 0, out_dim = 0;
  WideLayerDev L[kMaxLayers];
  int max_kp = 0;          // widest blocked activation (in K columns)
};

struct WideGemmArgs {
  const uint16_t* a;        // blocked activations [Mp/128][Kp/64] tiles
  const uint16_t* w;        // blocked weights     [Np/NT][Kp/64] tiles
  const float* bias;
  uint16_t* out_blocked;    // next layer's blocked activations (Kp_next = Np), or null for the output layer
  float* out_rows;          // [M, out_dim] fp32 (output layer)
  const int32_t* button0;
  double* qdes;
  MotorCmdDev* cmd;         // send_command arguments in Unitree motor order (flag 4) or null
  float kp, kd, kp_deadman;
  long long M;              // valid rows
  int m_tiles, n_tiles, k_chunks;
  int N, out_dim, has_elu;
  float alpha;
  uint32_t flags;
  float action_limit;
  double action_scale;
  double q0[kDof];
};

// fp32 [B, in] row-major -> blocked 16-bit tiles, zero padded to (m_tiles*128) x Kp.
// A warp converts 8 rows x 32 columns: lane = (column group of 8) * 8 + (row & 7), so its 32 16-byte stores are the four
// K-adjacent cores of one 8-row group -- 512 contiguous bytes (the first version walked along a row: every lane's
// 16 bytes went to a different 128-byte line, and the conversion took 34 us of a 195-us pass).
// kSplit: the three bf16 pieces of every value into the row tile's split tile group (wd_split_act)
template <bool kFp16, bool kSplit = false>
__global__ void obs_to_blocked_kernel(const float* __restrict__ obs, uint16_t* __restrict__ out, long long B, int in_dim, int Kp,
                                      long long m_tiles) {
  const int kg4 = Kp / 32;                                           // groups of four 8-column cores per row
  const long long items = m_tiles * (kWdTileM / 8) * kg4;            // one warp per (8-row group, 32 columns)
  const int lane = threadIdx.x & 31;
  const int r8 = lane & 7, cgl = lane >> 3;
  // programmatic dependent launch: the previous pass may still be reading the buffer this kernel rewrites
  ptx::grid_dependency_wait();
  ptx::grid_launch_dependents();
  const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long it = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; it < items; it += warps) {
    const long long rg = it / kg4;                                   // global 8-row group
    const int kg = (int)(it % kg4) * 4 + cgl;                        // this lane's 8-column core
    const long long row = rg * 8 + r8;
    const float* src = obs + row * in_dim + kg * 8;
    if constexpr (kSplit) {
      uint32_t p[3][4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int k = kg * 8 + 2 * j;
        const float x0 = (row < B && k < in_dim) ? src[2 * j] : 0.f;
        const float x1 = (row < B && k + 1 < in_dim) ? src[2 * j + 1] : 0.f;
        float s0[3], s1[3];
        wd_split_act(x0, s0[0], s0[1], s0[2]);
        wd_split_act(x1, s1[0], s1[1], s1[2]);
#pragma unroll
        for (int q = 0; q < 3; ++q) p[q][j] = ptx::pack_bf16(s0[q], s1[q]);
      }
      const long long mt = row / kWdTileM;
      const int r = (int)(row % kWdTileM);
      const int kc = (kg * 8) / kWdChunkK, c = (kg * 8) % kWdChunkK;
      uint8_t* dst = reinterpret_cast<uint8_t*>(out) + ((mt * (Kp / kWdChunkK) + kc) * 3 * (long long)kWdATileBytes) + wd_tile_offset(r, c);
#pragma unroll
      for (int q = 0; q < 3; ++q) *reinterpret_cast<uint4*>(dst + q * kWdATileBytes) = make_uint4(p[q][0], p[q][1], p[q][2], p[q][3]);
      continue;
    }
    uint32_t p[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = kg * 8 + 2 * j;
      const float lo = (row < B && k < in_dim) ? src[2 * j] : 0.f;
      const float hi = (row < B && k + 1 < in_dim) ? src[2 * j + 1] : 0.f;
      p[j] = kFp16 ? ptx::pack_f16_sat(lo, hi) : ptx::pack_bf16(lo, hi);
    }
    const long long mt = row / kWdTileM;
    const int r = (int)(row % kWdTileM);
    const int kc = (kg * 8) / kWdChunkK, c = (kg * 8) % kWdChunkK;
    uint8_t* dst = reinterpret_cast<uint8_t*>(out) + ((mt * (Kp / kWdChunkK) + kc) * (long long)kWdATileBytes) + wd_tile_offset(r, c);
    *reinterpret_cast<uint4*>(dst) = make_uint4(p[0], p[1], p[2], p[3]);
  }
}

// kSplit (GO2P_PREC_FP32_TC, bf16): a and w are split tile groups (wd_split_act / wd_split_weight).  A stage
// holds the three A pieces and the three B pieces of one K chunk, and per K16 step the MMA warp issues the six products
// whose size is at least 2^-16 of the leading term from that one stage: hi*hi into the main accumulator, hi*mid,
// mid*hi, hi*lo, lo*hi, mid*mid into a second one (the dropped mid*lo, lo*mid, lo*lo are <= 2^-23 relative).  The
// epilogue adds the two accumulators, then the bias in fp32; a hidden layer stores the three pieces of its output.
template <int NT, bool kFp16, bool kSplit = false>
__global__ void __launch_bounds__(kWdThreads, 1) wide_gemm_kernel(const WideGemmArgs a) {
  static_assert(!kSplit || (!kFp16 && NT <= 128), "the split operands are bf16, N tile <= 128");
  extern __shared__ __align__(128) uint8_t smem[];
  constexpr int kBTileBytes = NT * kWdChunkK * 2;
  constexpr int kStageBytes = (kSplit ? 3 : 1) * (kWdATileBytes + kBTileBytes);
  constexpr int kStages = wd_stages(NT, kSplit);
  constexpr uint32_t kAccCols = NT < 32 ? 32 : NT;               // TMEM columns per accumulator
  constexpr uint32_t kAccs = kSplit ? 2 : 1;                     // accumulators per buffer
  constexpr uint32_t kTmemCols = 2 * kAccs * kAccCols;           // 64 .. 512, a power of two
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kStages * kStageBytes);
  uint64_t* full = bars;                 // [kStages] chunk landed
  uint64_t* empty = bars + kStages;    // [kStages] chunk consumed by the tensor core
  uint64_t* acc_full = bars + 2 * kStages;       // [2]
  uint64_t* acc_empty = bars + 2 * kStages + 2;  // [2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);

  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < kStages; ++s) { ptx::mbar_init(&full[s], 1); ptx::mbar_init(&empty[s], 1); }
      for (int b = 0; b < 2; ++b) { ptx::mbar_init(&acc_full[b], 1); ptx::mbar_init(&acc_empty[b], kWdEpiWarps); }
      ptx::fence_mbar_init();
    }
    __syncwarp();
    ptx::tmem_alloc<kTmemCols>(tmem_ptr);
  }
  ptx::tc_fence_before();
  block_sync();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  // Programmatic dependent launch: barriers and TMEM are set up while the previous layer's launch drains; its
  // activations are read (and the buffer two layers back is overwritten) only after that launch has completed.  The
  // next layer's launch may begin its own set-up as soon as this CTA's SM is free.  (5 launches per 18,944-row pass:
  // the gaps between them were a quarter of the wide policy's time.)  Weights and biases, like activations, are read
  // only after the wait (the producer warp's bulk copies and the epilogue's bias loads below), so a launch may follow
  // the weight packer of go2p_set_weights on the same stream with programmatic serialization; obs_to_blocked_kernel
  // reads no weights at all.
  ptx::grid_dependency_wait();
  ptx::grid_launch_dependents();

  // job = (row tile, N tile), N tile fastest: the A tiles stay in L2 for the next N tile.  job < m_tiles * n_tiles, so
  // mt < m_tiles: the producer's clamp and the epilogue's row-tile test below are redundant.  They stay because without
  // them ptxas schedules the epilogues differently (other register counts), and this is the code DESIGN.md §3.3b measured.
  const long long job0 = blockIdx.x, job_stride = gridDim.x;
  const long long n_jobs = (long long)a.m_tiles * a.n_tiles;
  if (warp == 0) {
    // ================= producer =================
    uint32_t it = 0;
    for (long long job = job0; job < n_jobs; job += job_stride) {
      const long long mt = min(job / a.n_tiles, (long long)a.m_tiles - 1);
      const int nt = (int)(job % a.n_tiles);
      for (int kc = 0; kc < a.k_chunks; ++kc, ++it) {
        const int s = it % kStages;
        ptx::mbar_wait(&empty[s], ((it / kStages) & 1u) ^ 1u);
        if constexpr (kSplit) {
          if (ptx::elect_one_sync()) {
            uint8_t* st = smem + s * kStageBytes;
            ptx::mbar_arrive_expect_tx(&full[s], (uint32_t)kStageBytes);
            const uint8_t* asrc = reinterpret_cast<const uint8_t*>(a.a) + (mt * a.k_chunks + kc) * 3 * (long long)kWdATileBytes;
            const uint8_t* wsrc = reinterpret_cast<const uint8_t*>(a.w) + ((long long)nt * a.k_chunks + kc) * 3 * (long long)kBTileBytes;
#pragma unroll
            for (int q = 0; q < 3; ++q) ptx::bulk_g2s(st + q * kWdATileBytes, asrc + q * kWdATileBytes, kWdATileBytes, &full[s]);
#pragma unroll
            for (int q = 0; q < 3; ++q)
              ptx::bulk_g2s(st + 3 * kWdATileBytes + q * kBTileBytes, wsrc + q * kBTileBytes, kBTileBytes, &full[s]);
          }
          __syncwarp();
          continue;
        }
        if (ptx::elect_one_sync()) {
          uint8_t* st = smem + s * kStageBytes;
          ptx::mbar_arrive_expect_tx(&full[s], (uint32_t)kStageBytes);
          ptx::bulk_g2s(st, reinterpret_cast<const uint8_t*>(a.a) + (mt * a.k_chunks + kc) * (long long)kWdATileBytes, kWdATileBytes, &full[s]);
          const uint8_t* wsrc = reinterpret_cast<const uint8_t*>(a.w) + ((long long)nt * a.k_chunks + kc) * (long long)kBTileBytes;
          ptx::bulk_g2s(st + kWdATileBytes, wsrc, kBTileBytes, &full[s]);
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    const uint32_t idesc = ptx::make_idesc(kFp16 ? ptx::FMT_F16 : ptx::FMT_BF16, kWdTileM, (uint32_t)NT);
    uint32_t it = 0, tile_i = 0;
    for (long long job = job0; job < n_jobs; job += job_stride, ++tile_i) {
      const uint32_t buf = tile_i & 1u;
      ptx::mbar_wait(&acc_empty[buf], ((tile_i >> 1) & 1u) ^ 1u);
      ptx::tc_fence_after();
      const uint32_t d_t = tmem_base + buf * kAccs * kAccCols;
      for (int kc = 0; kc < a.k_chunks; ++kc, ++it) {
        const int s = it % kStages;
        ptx::mbar_wait(&full[s], (it / kStages) & 1u);
        ptx::tc_fence_after();
        if constexpr (kSplit) {
          if (ptx::elect_one_sync()) {
            const uint32_t sa = ptx::smem_u32(smem + s * kStageBytes);
            uint64_t ad[3], bd[3];
#pragma unroll
            for (int q = 0; q < 3; ++q) {
              ad[q] = ptx::make_smem_desc_nosw(sa + q * kWdATileBytes, 128u, 1024u);
              bd[q] = ptx::make_smem_desc_nosw(sa + 3 * kWdATileBytes + q * kBTileBytes, 128u, 1024u);
            }
#pragma unroll
            for (int j = 0; j < kWdChunkK / 16; ++j) {
              const uint64_t o = (uint64_t)(j * 16);
              const uint32_t acc = (kc | j) ? 1u : 0u;
              ptx::mma_f16_ss(d_t, ad[0] + o, bd[0] + o, idesc, acc);                 // hi * hi
              ptx::mma_f16_ss(d_t + kAccCols, ad[0] + o, bd[1] + o, idesc, acc);      // hi * mid
              ptx::mma_f16_ss(d_t + kAccCols, ad[1] + o, bd[0] + o, idesc, 1u);       // mid * hi
              ptx::mma_f16_ss(d_t + kAccCols, ad[0] + o, bd[2] + o, idesc, 1u);       // hi * lo
              ptx::mma_f16_ss(d_t + kAccCols, ad[2] + o, bd[0] + o, idesc, 1u);       // lo * hi
              ptx::mma_f16_ss(d_t + kAccCols, ad[1] + o, bd[1] + o, idesc, 1u);       // mid * mid
            }
            ptx::mma_commit(&empty[s]);
            if (kc == a.k_chunks - 1) ptx::mma_commit(&acc_full[buf]);
          }
          __syncwarp();
          continue;
        }
        if (ptx::elect_one_sync()) {
          const uint32_t sa = ptx::smem_u32(smem + s * kStageBytes);
          const uint64_t adesc = ptx::make_smem_desc_nosw(sa, 128u, 1024u);
          const uint64_t bdesc = ptx::make_smem_desc_nosw(sa + kWdATileBytes, 128u, 1024u);
#pragma unroll
          for (int j = 0; j < kWdChunkK / 16; ++j)
            ptx::mma_f16_ss(d_t, adesc + (uint64_t)(j * 16), bdesc + (uint64_t)(j * 16), idesc, (kc | j) ? 1u : 0u);
          ptx::mma_commit(&empty[s]);                  // frees the stage when these MMAs have read it
          if (kc == a.k_chunks - 1) ptx::mma_commit(&acc_full[buf]);
        }
        __syncwarp();
      }
    }
  } else {
    // ================= epilogue warps (lane quarter = warp % 4) =================
    const int quarter = warp & 3;
    const int half = (warp - 2) >> 2;                // which share of the N tile's columns this warp converts
    const uint32_t lane_addr = ((uint32_t)(quarter * 32)) << 16;
    const int r = quarter * 32 + lane;               // row inside the tile
    uint32_t tile_i = 0;
    for (long long job = job0; job < n_jobs; job += job_stride, ++tile_i) {
      const long long mt = job / a.n_tiles;
      const bool past_end = mt >= a.m_tiles;           // never true (see the job mapping above)
      const int nt = (int)(job % a.n_tiles);
      const uint32_t buf = tile_i & 1u;
      ptx::mbar_wait(&acc_full[buf], (tile_i >> 1) & 1u);
      ptx::tc_fence_after();
      const uint32_t acc_t = tmem_base + buf * kAccs * kAccCols + lane_addr;
      const long long row = mt * kWdTileM + r;
      if (past_end) {
        // nothing to store; the accumulator is simply released
      } else if (kSplit && a.out_blocked) {
        if constexpr (kSplit) {   // discarded in the 16-bit instantiations, whose code stays as it was
          // hidden layer: 16 columns at a time -> both accumulators + bias + ELU -> three bf16 pieces -> two 16-byte
          // stores into each of the next layer's three tiles
          const long long next_chunks = (long long)a.n_tiles * (NT / kWdChunkK);
          constexpr int kShare = (NT / kWdEpiParts) < 16 ? 16 : (NT / kWdEpiParts);
#pragma unroll 1
          for (int c0 = half * kShare; c0 < (half + 1) * kShare && c0 < NT; c0 += 16) {
            uint32_t v[16], u[16];
            ptx::tmem_ld_x16(acc_t + (uint32_t)c0, v);
            ptx::tmem_ld_x16(acc_t + kAccCols + (uint32_t)c0, u);
            ptx::tc_wait_ld();
            float x[16];
            {
              const float4* b4 = reinterpret_cast<const float4*>(a.bias + nt * NT + c0);
#pragma unroll
              for (int j4 = 0; j4 < 4; ++j4) {
                const float4 b = __ldg(b4 + j4);
                const float bl[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
                  x[4 * j4 + i] = (__uint_as_float(v[4 * j4 + i]) + __uint_as_float(u[4 * j4 + i])) + bl[i];
              }
            }
            // the activation test is hoisted out of the unrolled loop, as in the 16-bit epilogue below
            if (a.has_elu) {
              const float alpha = a.alpha, nalpha = -a.alpha;
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const float e = fmaf(alpha, ptx::ex2_approx(x[i] * 1.4426950408889634f), nalpha);
                x[i] = (x[i] < 0.f) ? e : x[i];
              }
            }
            uint32_t p[3][8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float s0[3], s1[3];
              wd_split_act(x[2 * j], s0[0], s0[1], s0[2]);
              wd_split_act(x[2 * j + 1], s1[0], s1[1], s1[2]);
#pragma unroll
              for (int q = 0; q < 3; ++q) p[q][j] = ptx::pack_bf16(s0[q], s1[q]);
            }
            const int kn = nt * NT + c0;                 // K index of the next layer
            uint8_t* dst = reinterpret_cast<uint8_t*>(a.out_blocked) + ((mt * next_chunks + kn / kWdChunkK) * 3 * (long long)kWdATileBytes) +
                           wd_tile_offset(r, kn % kWdChunkK);
#pragma unroll
            for (int q = 0; q < 3; ++q)
#pragma unroll
              for (int c = 0; c < 2; ++c)                // consecutive 8-column cores are 128 B apart inside the tile
                *reinterpret_cast<uint4*>(dst + q * kWdATileBytes + c * 128) =
                    make_uint4(p[q][4 * c], p[q][4 * c + 1], p[q][4 * c + 2], p[q][4 * c + 3]);
          }
        }
      } else if (a.out_blocked) {
        // hidden layer: 32 columns at a time -> bias + ELU -> 16 bit -> four 16-byte stores into the next layer's tile
        const int kcn_per_tile = NT / kWdChunkK;       // 64-column chunks of the next layer covered by this N tile
        const long long next_chunks = (long long)a.n_tiles * kcn_per_tile;
        constexpr int kShare = (NT / kWdEpiParts) < 32 ? 32 : (NT / kWdEpiParts);   // columns per warp, whole 32-column groups
#pragma unroll 1
        for (int c0 = half * kShare; c0 < (half + 1) * kShare && c0 < NT; c0 += 32) {
          uint32_t v[32];
          ptx::tmem_ld_x32(acc_t + (uint32_t)c0, v);
          ptx::tc_wait_ld();
          // the 32 biases of this column group as eight 16-byte loads (warp-uniform address, 128-byte aligned)
          float bl[32];
          {
            const float4* b4 = reinterpret_cast<const float4*>(a.bias + nt * NT + c0);
#pragma unroll
            for (int j = 0; j < 8; ++j) { const float4 t = __ldg(b4 + j); bl[4 * j] = t.x; bl[4 * j + 1] = t.y; bl[4 * j + 2] = t.z; bl[4 * j + 3] = t.w; }
          }
          uint32_t p[16];
          // the activation test is hoisted out of the unrolled loop: inside it nvcc emitted a branch with its
          // reconvergence bookkeeping and a constant-bank reload of alpha per PAIR (15+ instead of 11 instructions)
          if (a.has_elu) {
            const float alpha = a.alpha, nalpha = -a.alpha;
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              float x0 = __uint_as_float(v[2 * j]) + bl[2 * j];
              float x1 = __uint_as_float(v[2 * j + 1]) + bl[2 * j + 1];
              const float e0 = fmaf(alpha, ptx::ex2_approx(x0 * 1.4426950408889634f), nalpha);
              const float e1 = fmaf(alpha, ptx::ex2_approx(x1 * 1.4426950408889634f), nalpha);
              x0 = (x0 < 0.f) ? e0 : x0;
              x1 = (x1 < 0.f) ? e1 : x1;
              p[j] = kFp16 ? ptx::pack_f16_sat(x0, x1) : ptx::pack_bf16(x0, x1);
            }
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const float x0 = __uint_as_float(v[2 * j]) + bl[2 * j];
              const float x1 = __uint_as_float(v[2 * j + 1]) + bl[2 * j + 1];
              p[j] = kFp16 ? ptx::pack_f16_sat(x0, x1) : ptx::pack_bf16(x0, x1);
            }
          }
          const int kn = nt * NT + c0;                 // K index of the next layer
          uint8_t* dst = reinterpret_cast<uint8_t*>(a.out_blocked) + ((mt * next_chunks + kn / kWdChunkK) * (long long)kWdATileBytes) +
                         wd_tile_offset(r, kn % kWdChunkK);
#pragma unroll
          for (int q = 0; q < 4; ++q)                  // consecutive 8-column cores are 128 B apart inside the tile
            *reinterpret_cast<uint4*>(dst + q * 128) = make_uint4(p[4 * q], p[4 * q + 1], p[4 * q + 2], p[4 * q + 3]);
        }
      } else {
        // output layer (NT == 16): bias (+ELU) (+clamp/mask) (+q_des) -> fp32 rows
        uint32_t v[16];
        ptx::tmem_ld_x16(acc_t, v);
        if constexpr (kSplit) {
          uint32_t u[16];
          ptx::tmem_ld_x16(acc_t + kAccCols, u);
          ptx::tc_wait_ld();
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(u[j]));
        }
        ptx::tc_wait_ld();
        if (row < a.M && half == 0) {
          const int b0 = ((a.flags & 5u) && a.button0) ? a.button0[row] : 0;
          float* dst = a.out_rows + row * a.out_dim;
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            if (j < a.out_dim) {
              float x = __uint_as_float(v[j]) + a.bias[j];
              if (a.has_elu) x = (x < 0.f) ? fmaf(a.alpha, ptx::ex2_approx(x * 1.4426950408889634f), -a.alpha) : x;
              if (a.flags & 1u) x = clamp_mask(x, a.action_limit, b0);
              dst[j] = x;
              if (j < kDof && (a.flags & 6u)) {
                const double qd = joint_target(x, a.q0[j], a.action_scale);
                if ((a.flags & 2u) && a.qdes) a.qdes[row * kDof + j] = qd;
                if ((a.flags & 4u) && a.cmd) a.cmd[row].q_des[motor_of_isaac(j)] = qd;
              }
            }
          }
          if ((a.flags & 4u) && a.cmd) store_gains(a.cmd, row, b0, a.kp, a.kd, a.kp_deadman);
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&acc_empty[buf]);
    }
  }

  ptx::tc_fence_before();
  block_sync();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<kTmemCols>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------ host side
inline int wd_round_up(int v, int m) { return (v + m - 1) / m * m; }

// blocked image of W [N][K] for N tiles of NT rows: tile (nt, kc) = NT x 64 elements
inline void wd_pack_weights(const MlpLayer& L, int NT, int Np, int Kp, bool fp16, std::vector<uint16_t>& out) {
  out.assign((size_t)Np * Kp, 0);
  const int k_chunks = Kp / kWdChunkK;
  for (int n = 0; n < L.out; ++n)
    for (int k = 0; k < L.in; ++k) {
      const float v = L.weight[(size_t)n * L.in + k];
      const size_t tile = ((size_t)(n / NT) * k_chunks + k / kWdChunkK) * ((size_t)NT * kWdChunkK);
      const size_t idx = tile + wd_tile_offset(n % NT, k % kWdChunkK) / 2;
      uint16_t b;
      if (fp16) { const float c = v > 65504.f ? 65504.f : (v < -65504.f ? -65504.f : v); b = __half_as_ushort(__float2half_rn(c)); }
      else b = __bfloat16_as_ushort(__float2bfloat16_rn(v));
      out[idx] = b;
    }
}

// the split images of W [N][K] (wd_split_weight): tile group (nt, kc) = the hi, mid and lo NT x 64 tiles
inline void wd_pack_split(const MlpLayer& L, int NT, int Np, int Kp, std::vector<uint16_t>& out) {
  out.assign((size_t)Np * Kp * 3, 0);
  const int k_chunks = Kp / kWdChunkK;
  const size_t tile_elems = (size_t)NT * kWdChunkK;
  for (int n = 0; n < L.out; ++n)
    for (int k = 0; k < L.in; ++k) {
      uint16_t p[3];
      wd_split_weight(L.weight[(size_t)n * L.in + k], p);
      const size_t idx = ((size_t)(n / NT) * k_chunks + k / kWdChunkK) * 3 * tile_elems + wd_tile_offset(n % NT, k % kWdChunkK) / 2;
      for (int q = 0; q < 3; ++q) out[idx + q * tile_elems] = p[q];
    }
}

// returns 0 = ok, > 0 = go2p_status (CUDA failure), < 0 = this shape is not served by the wide path.
// alloc(bytes) returns device memory that the caller owns, or null.  images16: also build the bf16 / fp16 images (the
// split images of GO2P_PREC_FP32_TC are always built).
template <class Alloc>
inline int wide_prepare(const MlpModel& m, Alloc&& alloc, WideModel* wm, bool images16, std::string& err) {
  const int nl = (int)m.layers.size();
  if (nl < 2 || nl > kMaxLayers || m.layers.back().out > 16) return -1;
  for (int l = 0; l + 1 < nl; ++l) if (m.layers[l].out % 64 != 0) return -1;
  wm->n_layers = nl; wm->in_dim = m.layers.front().in; wm->out_dim = m.layers.back().out; wm->max_kp = 0;
  auto upload = [&](const void* src, size_t bytes, void** out) -> bool {
    void* p = alloc(bytes);
    if (!p) { err = "wide_prepare: cudaMalloc failed"; return false; }
    if (cudaMemcpy(p, src, bytes, cudaMemcpyHostToDevice) != cudaSuccess) { err = "wide_prepare: cudaMemcpy failed"; return false; }
    *out = p; return true;
  };
  for (int l = 0; l < nl; ++l) {
    const MlpLayer& L = m.layers[l];
    WideLayerDev& D = wm->L[l];
    const bool last = l == nl - 1;
    D.K = L.in; D.N = L.out;
    D.Kp = wd_round_up(L.in, kWdChunkK);
    D.NT = last ? 16 : (L.out % 256 == 0 ? 256 : (L.out % 128 == 0 ? 128 : 64));
    D.Np = wd_round_up(L.out, D.NT);
    // split stages hold three pieces of each operand: N tiles of at most 128 rows keep two of them (192 KB) in flight
    D.NT3 = D.NT > 128 ? 128 : D.NT;
    D.has_elu = L.has_elu ? 1 : 0; D.alpha = L.elu_alpha;
    if (l > 0 && D.Kp != wm->L[l - 1].Np) return -1;   // a hidden width that is not a multiple of 64
    wm->max_kp = std::max(wm->max_kp, D.Kp);
    std::vector<uint16_t> img;
    for (int f = 0; f < 2 && images16; ++f) {
      wd_pack_weights(L, D.NT, D.Np, D.Kp, f == 1, img);
      void* p;
      if (!upload(img.data(), img.size() * 2, &p)) return 4;
      D.w[f] = static_cast<const uint16_t*>(p);
    }
    {
      wd_pack_split(L, D.NT3, D.Np, D.Kp, img);
      void* p;
      if (!upload(img.data(), img.size() * 2, &p)) return 4;
      D.w3 = static_cast<const uint16_t*>(p);
    }
    std::vector<float> bias(D.Np, 0.f);
    for (int n = 0; n < L.out; ++n) bias[n] = L.bias[n];
    void* pb;
    if (!upload(bias.data(), bias.size() * 4, &pb)) return 4;
    D.bias = static_cast<const float*>(pb);
  }
  return 0;
}

// One persistent CTA per SM (at most one per job).  opt_in(kernel, bytes) -> cudaError_t opts the kernel in to `bytes`
// of dynamic shared memory on the current device.
template <int NT, bool kFp16, bool kSplit, class OptIn>
inline cudaError_t wd_launch(const WideGemmArgs& a, int sm_count, OptIn& opt_in, cudaStream_t st) {
  const size_t smem = (size_t)wd_stages(NT, kSplit) * (kSplit ? 3 : 1) * (kWdATileBytes + NT * kWdChunkK * 2) + 256;
  auto kernel = wide_gemm_kernel<NT, kFp16, kSplit>;
  const cudaError_t e = opt_in(reinterpret_cast<const void*>(kernel), smem);
  if (e != cudaSuccess) return e;
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;      // see griddepcontrol.wait in the kernel
  attr.val.programmaticStreamSerializationAllowed = 1;
  cfg.blockDim = dim3(kWdThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cfg.attrs = &attr; cfg.numAttrs = 1;
  const long long jobs = (long long)a.m_tiles * a.n_tiles;
  cfg.gridDim = dim3((unsigned)std::min<long long>(jobs, (long long)sm_count));
  return cudaLaunchKernelEx(&cfg, kernel, a);
}

// rows per pass: a multiple of 148 row tiles, so every layer's job count is a whole number of waves over the 148 SMs.
// Round 1 used ONE wave of row tiles (18,944 rows: the widest activation, 39 MB, stays in the 126 MB L2); measured in
// round 2 (606,208 rows, fp16 / bf16): 1 wave 1.86 / 1.85 ms, 2 waves 1.62 / 1.66 ms,
// 4 waves 1.57 / 1.51 ms, 32 waves (the whole batch) 1.54 / 1.48 ms -- the five launches per pass each end in a tail
// (layers 3 and 4 are ONE job per CTA at one wave: no overlap of epilogue and MMAs at all), and that costs more than
// reading the activations back from HBM instead of L2.  Four waves: 75,776 rows, 155 MB per activation buffer.
constexpr long long kWdChunkRows = 148 * kWdTileM * 4;

// rows of one pass of wide_launch over B rows, in whole row tiles
inline long long wide_act_rows(long long B) {
  return (std::min<long long>(B, kWdChunkRows) + kWdTileM - 1) / kWdTileM * kWdTileM;
}

// operand formats of wide_launch
enum WdOperands { kWdBf16 = 0, kWdFp16 = 1, kWdSplit = 2 };

// act: the two blocked activation buffers (ping-pong), each of wide_act_rows(B) rows x wm.max_kp 16-bit columns (three
// times that for kWdSplit).  opt_in: see wd_launch.
template <class OptIn>
inline int wide_launch(const WideModel& wm, uint16_t* const act[2], const float* d_obs, const int32_t* d_button0, float* d_act, double* d_qdes,
                       MotorCmdDev* d_cmd, long long B, WdOperands operands, uint32_t flags, const CtrlConst& cc, int sm_count,
                       OptIn&& opt_in, cudaStream_t st, int* launches, std::string& err) {
  const bool fp16 = operands == kWdFp16, split = operands == kWdSplit;
  const long long chunk = std::min<long long>(B, kWdChunkRows);
  for (long long r0 = 0; r0 < B; r0 += chunk) {
    const long long rows = std::min(chunk, B - r0);
    const int m_tiles = (int)((rows + kWdTileM - 1) / kWdTileM);
    const WideLayerDev& L0 = wm.L[0];
    {
      const long long groups = (long long)m_tiles * kWdTileM * (L0.Kp / 8);
      const int blocks = (int)std::min<long long>((groups + 255) / 256, (long long)sm_count * 8);
      cudaLaunchConfig_t lc = {};
      cudaLaunchAttribute la;
      la.id = cudaLaunchAttributeProgrammaticStreamSerialization;
      la.val.programmaticStreamSerializationAllowed = 1;
      lc.gridDim = dim3((unsigned)blocks); lc.blockDim = dim3(256); lc.stream = st; lc.attrs = &la; lc.numAttrs = 1;
      const float* src = d_obs + r0 * wm.in_dim;
      const long long m_tiles_ll = m_tiles;
      cudaError_t ec = split ? cudaLaunchKernelEx(&lc, obs_to_blocked_kernel<false, true>, src, act[0], rows, wm.in_dim, L0.Kp, m_tiles_ll)
                     : fp16  ? cudaLaunchKernelEx(&lc, obs_to_blocked_kernel<true>, src, act[0], rows, wm.in_dim, L0.Kp, m_tiles_ll)
                             : cudaLaunchKernelEx(&lc, obs_to_blocked_kernel<false>, src, act[0], rows, wm.in_dim, L0.Kp, m_tiles_ll);
      if (ec != cudaSuccess) { err = std::string("wide_launch: ") + cudaGetErrorString(ec); return 4; }
      ++*launches;
    }
    int cur = 0;
    for (int l = 0; l < wm.n_layers; ++l) {
      const WideLayerDev& L = wm.L[l];
      const bool last = l == wm.n_layers - 1;
      WideGemmArgs a{};
      const int NT = split ? L.NT3 : L.NT;
      a.a = act[cur]; a.w = split ? L.w3 : L.w[fp16 ? 1 : 0]; a.bias = L.bias;
      a.out_blocked = last ? nullptr : act[cur ^ 1];
      a.out_rows = last ? d_act + r0 * wm.out_dim : nullptr;
      a.button0 = d_button0 ? d_button0 + r0 : nullptr;
      a.qdes = d_qdes ? d_qdes + r0 * kDof : nullptr;
      a.cmd = d_cmd ? d_cmd + r0 : nullptr;
      a.kp = cc.kp; a.kd = cc.kd; a.kp_deadman = cc.kp_deadman;
      a.M = rows; a.m_tiles = m_tiles; a.n_tiles = L.Np / NT; a.k_chunks = L.Kp / kWdChunkK;
      a.N = L.N; a.out_dim = wm.out_dim; a.has_elu = L.has_elu; a.alpha = L.alpha;
      a.flags = last ? flags : 0u; a.action_limit = cc.action_limit; a.action_scale = cc.action_scale;
      for (int i = 0; i < kDof; ++i) a.q0[i] = cc.q0[i];
      cudaError_t e;
      if (split) {
        if (NT == 128) e = wd_launch<128, false, true>(a, sm_count, opt_in, st);
        else if (NT == 64) e = wd_launch<64, false, true>(a, sm_count, opt_in, st);
        else e = wd_launch<16, false, true>(a, sm_count, opt_in, st);
      } else if (L.NT == 256) e = fp16 ? wd_launch<256, true, false>(a, sm_count, opt_in, st) : wd_launch<256, false, false>(a, sm_count, opt_in, st);
      else if (L.NT == 128) e = fp16 ? wd_launch<128, true, false>(a, sm_count, opt_in, st) : wd_launch<128, false, false>(a, sm_count, opt_in, st);
      else if (L.NT == 64) e = fp16 ? wd_launch<64, true, false>(a, sm_count, opt_in, st) : wd_launch<64, false, false>(a, sm_count, opt_in, st);
      else e = fp16 ? wd_launch<16, true, false>(a, sm_count, opt_in, st) : wd_launch<16, false, false>(a, sm_count, opt_in, st);
      if (e != cudaSuccess) { err = std::string("wide_launch: ") + cudaGetErrorString(e); return 4; }
      ++*launches;
      cur ^= 1;
    }
  }
  return 0;
}

}  // namespace go2p
