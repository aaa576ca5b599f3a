// Device-side weight packer of go2p_set_weights: rebuilds, in place, every weight image a handle's kernels read from
// the caller's fp32 tensors (torch nn.Linear layout: W [N][K] row-major, b [N]).
//
//   fold_normaliser_kernel   x' = (x - mean) / std folded into layer 0 (what onnx_reader.cpp does for a Sub -> Div
//                            prefix), into a scratch copy of layer 0
//   pack_weights_kernel      per layer: the fp32 layouts of DevLayer (w_rm, w_k4, w_kn, bias), the 16-bit UMMA K-major
//                            images of the narrow tensor-core kernel (capi.cu: pack_umma_kmajor) and the blocked tiles +
//                            padded bias of the wide GEMMs (kernels_wide.cuh: wd_pack_weights), and with kSplit the
//                            three-piece bf16 images of GO2P_PREC_FP32_TC (wd_pack_split)
//
// The images must be byte-identical to what the host packers produce for the same tensors.  The host code is built
// without -march, so it has no FMA; the device compiler contracts a*b+c into FMA by default.  Every rounding step is
// therefore spelled as an explicitly rounded operation (__dmul_rn, __dadd_rn, __ddiv_rn, __fsub_rn, __double2float_rn),
// in the same order as the host code.  Only elements that carry a value are written: the zero padding of every image
// was written at go2p_create and no tensor of the same topology changes it.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <cstdint>

#include "kernels_wide.cuh"
#include "policy_dev.cuh"

namespace go2p {

struct PackLayer {
  const float* w;          // [N][K] fp32, row-major
  const float* b;          // [N] fp32, or null = zeros
  int K, N;
  // DevLayer
  float* w_rm; float* w_k4; float* w_kn; float* bias;
  int Kp, Np;
  // narrow tensor-core images (null when the handle has none): [0] bf16, [1] fp16, this layer's part of d_wpack
  uint16_t* tc[2];
  int tc_Kp;
  double wscale, bscale;   // base-2 scaling of the layer (capi.cu: upload_model)
  // wide GEMM images (null when the handle has none)
  uint16_t* wd[2];
  float* wd_bias;
  int wd_NT, wd_Kp;
};

// the split images of GO2P_PREC_FP32_TC (kernels_wide.cuh: wd_pack_split)
struct PackSplitLayer {
  uint16_t* w3;
  float* bias;             // the wide GEMMs' padded bias
  int NT, Kp;
};

struct PackArgs {
  PackLayer L[kMaxLayers];
  int n_layers;
  PackSplitLayer S[kMaxLayers];   // read by pack_weights_kernel<true> only; after n_layers, so L keeps its offsets
};

// capi.cu: to_bf16 / to_f16 / from_bf16 / from_f16.  std::max(-65504.f, f) is (-65504 < f ? f : -65504) and
// std::min(65504.f, t) is (t < 65504 ? t : 65504): spelled the same way so that NaN maps to the same code as on the host.
__device__ __forceinline__ uint16_t pk_enc(float f, bool fp16) {
  if (fp16) {
    f = (-65504.f < f) ? f : -65504.f;
    f = (f < 65504.f) ? f : 65504.f;
    return __half_as_ushort(__float2half_rn(f));
  }
  return __bfloat16_as_ushort(__float2bfloat16_rn(f));
}
__device__ __forceinline__ float pk_dec(uint16_t b, bool fp16) {
  return fp16 ? __half2float(__ushort_as_half(b)) : __bfloat162float(__ushort_as_bfloat16(b));
}

// onnx_reader.cpp, the normaliser fold of the first Gemm: one thread per output row, k in the reader's order.
// The reader builds pre_shift = (0 - mean) / std and pre_scale = 1 / std (a Sub node, then a Div node) in double.
__global__ void fold_normaliser_kernel(const float* __restrict__ w, const float* __restrict__ b, const float* __restrict__ mean,
                                       const float* __restrict__ stdv, int K, int N, float* __restrict__ w_out,
                                       float* __restrict__ b_out) {
  const int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= N) return;
  double acc = b ? (double)b[o] : 0.0;
  for (int k = 0; k < K; ++k) {
    const double s = (double)stdv[k];
    const double scale = __ddiv_rn(1.0, s);
    const double shift = __ddiv_rn(__dsub_rn(0.0, (double)mean[k]), s);
    const double v = (double)w[(size_t)o * K + k];
    acc = __dadd_rn(acc, __dmul_rn(v, shift));
    w_out[(size_t)o * K + k] = __double2float_rn(__dmul_rn(v, scale));
  }
  b_out[o] = __double2float_rn(acc);
}

// blockIdx.y = layer; a grid-stride walk over its N x (K + 1) elements, column K standing for the bias.  kSplit: also the
// split images (a.S) of a handle that serves GO2P_PREC_FP32_TC
template <bool kSplit>
__global__ void pack_weights_kernel(const __grid_constant__ PackArgs a) {
  const PackLayer& L = a.L[blockIdx.y];
  const long long total = (long long)L.N * (L.K + 1);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(i / (L.K + 1)), k = (int)(i % (L.K + 1));
    if (k < L.K) {
      const float v = L.w[(size_t)n * L.K + k];
      L.w_rm[(size_t)n * L.Kp + k] = v;
      L.w_k4[((size_t)(k / 4) * L.N + n) * 4 + (k % 4)] = v;
      L.w_kn[(size_t)k * L.Np + n] = v;
      if (L.tc[0]) {
        const float s = __double2float_rn(__dmul_rn((double)v, L.wscale));
        const size_t idx = ((size_t)(n / 8) * (L.tc_Kp / 8) + (k / 8)) * 64 + (n % 8) * 8 + (k % 8);
        L.tc[0][idx] = pk_enc(s, false);
        L.tc[1][idx] = pk_enc(s, true);
      }
      if (L.wd[0]) {
        const int k_chunks = L.wd_Kp / kWdChunkK;
        const size_t tile = ((size_t)(n / L.wd_NT) * k_chunks + k / kWdChunkK) * ((size_t)L.wd_NT * kWdChunkK);
        const size_t idx = tile + wd_tile_offset(n % L.wd_NT, k % kWdChunkK) / 2;
        const float c = v > 65504.f ? 65504.f : (v < -65504.f ? -65504.f : v);   // wd_pack_weights
        L.wd[0][idx] = __bfloat16_as_ushort(__float2bfloat16_rn(v));
        L.wd[1][idx] = __half_as_ushort(__float2half_rn(c));
      }
      if constexpr (kSplit) {
        const PackSplitLayer& S = a.S[blockIdx.y];
        const size_t tile_elems = (size_t)S.NT * kWdChunkK;
        const size_t idx = ((size_t)(n / S.NT) * (S.Kp / kWdChunkK) + k / kWdChunkK) * 3 * tile_elems + wd_tile_offset(n % S.NT, k % kWdChunkK) / 2;
        uint16_t p[3];
        wd_split_weight(v, p);
#pragma unroll
        for (int q = 0; q < 3; ++q) S.w3[idx + q * tile_elems] = p[q];
      }
    } else {
      const float v = L.b ? L.b[n] : 0.f;
      L.bias[n] = v;
      if (L.tc[0]) {
        // the bias rides in K rows in and in+1 as hi / lo 16-bit halves of bias * bscale
        const float s = __double2float_rn(__dmul_rn((double)v, L.bscale));
#pragma unroll
        for (int f = 0; f < 2; ++f) {
          const uint16_t hi = pk_enc(s, f == 1);
          const uint16_t lo = pk_enc(__fsub_rn(s, pk_dec(hi, f == 1)), f == 1);
          const size_t base = (size_t)(n / 8) * (L.tc_Kp / 8) * 64 + (n % 8) * 8;
          L.tc[f][base + (size_t)(L.K / 8) * 64 + (L.K % 8)] = hi;
          L.tc[f][base + (size_t)((L.K + 1) / 8) * 64 + ((L.K + 1) % 8)] = lo;
        }
      }
      if (L.wd[0]) L.wd_bias[n] = v;
      if constexpr (kSplit) a.S[blockIdx.y].bias[n] = v;
    }
  }
}

}  // namespace go2p
