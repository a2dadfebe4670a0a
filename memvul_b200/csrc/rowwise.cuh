// Row-wise HBM-bound kernels: embedding gather + LayerNorm (SURVEY.md 2.2 row K1) and the
// LayerNorm that follows the two residual GEMMs (second half of rows K4 / K6).
// One warp per token row; every lane owns NV float4 (NV = H / 128), loads are 128-bit and
// fully coalesced, statistics are two-pass in registers (mean, then centred variance) exactly
// like the reference's fp32 LayerNorm (eps 1e-12, HF BertEmbeddings / BertSelfOutput / BertOutput).
// Each kernel writes the fp32 residual stream AND the fp16 copy the next tcgen05 GEMM reads.
#pragma once
#include "ptx.cuh"

namespace mv {

template <int NV>
__device__ __forceinline__ void ln_store(float4 (&v)[NV], const float* __restrict__ gamma,
                                         const float* __restrict__ beta, float eps, float* __restrict__ out32,
                                         __half* __restrict__ out16, int lane) {
  constexpr int H = NV * 128;
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  const float mean = warp_sum(s) * (1.0f / H);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    v[i].x -= mean; v[i].y -= mean; v[i].z -= mean; v[i].w -= mean;
    q += (v[i].x * v[i].x + v[i].y * v[i].y) + (v[i].z * v[i].z + v[i].w * v[i].w);
  }
  const float rstd = 1.0f / sqrtf(warp_sum(q) * (1.0f / H) + eps);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int col = i * 128 + lane * 4;
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + col));
    const float4 b = __ldg(reinterpret_cast<const float4*>(beta + col));
    float4 o;
    o.x = v[i].x * rstd * g.x + b.x;
    o.y = v[i].y * rstd * g.y + b.y;
    o.z = v[i].z * rstd * g.z + b.z;
    o.w = v[i].w * rstd * g.w + b.w;
    if (out32) *reinterpret_cast<float4*>(out32 + col) = o;
    if (out16) {
      uint2 pk;
      pk.x = pack_half2(o.x, o.y);
      pk.y = pack_half2(o.z, o.w);
      *reinterpret_cast<uint2*>(out16 + col) = pk;
    }
  }
}

// y [M,H] fp32 (pre-LN residual sum)  ->  x32 [M,H] fp32, x16 [M,H] fp16.   In-place (x32 == y) is fine.
// x32_stride: elements between consecutive output rows of x32 (H for a dense matrix; S*H scatters row b to the
// [CLS] slot of sequence b in a [B,S,H] tensor).
template <int NV>
__global__ void __launch_bounds__(256) layernorm_rows_kernel(const float* y, const float* __restrict__ gamma,
                                                             const float* __restrict__ beta, float eps, float* x32,
                                                             long long x32_stride, __half* __restrict__ x16, int M) {
  constexpr int H = NV * 128;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= M) return;
  const float* src = y + static_cast<size_t>(row) * H;
  float4 v[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = *reinterpret_cast<const float4*>(src + i * 128 + lane * 4);
  ln_store<NV>(v, gamma, beta, eps, x32 ? x32 + static_cast<size_t>(row) * x32_stride : nullptr,
               x16 ? x16 + static_cast<size_t>(row) * H : nullptr, lane);
}

// Gather one row per sequence (row b*S -- or row_start[b] in the packed layout -- of a token-major matrix) into dense
// [B, H] matrices: the [CLS] rows that the last encoder layer's output projection / FFN actually need (BertPooler
// reads hidden[:,0] only, model_memory.py:99).
__global__ void __launch_bounds__(256) gather_cls_rows_kernel(const float* __restrict__ x32, const __half* __restrict__ c16,
                                                              float* __restrict__ x32_cls, __half* __restrict__ c16_cls,
                                                              const int* __restrict__ row_start, int B, int S, int H) {
  const int b = blockIdx.x;
  const size_t src = (row_start ? static_cast<size_t>(row_start[b]) : static_cast<size_t>(b) * S) * H;
  const size_t dst = static_cast<size_t>(b) * H;
  for (int i = threadIdx.x * 4; i < H; i += blockDim.x * 4) {
    *reinterpret_cast<float4*>(x32_cls + dst + i) = *reinterpret_cast<const float4*>(x32 + src + i);
    *reinterpret_cast<uint2*>(c16_cls + dst + i) = *reinterpret_cast<const uint2*>(c16 + src + i);
  }
}

// Packed (token-major) residual stream -> the padded [B,S,H] tensor the embedder interface returns
// (custom_PTM_embedder.py:235); padded positions are zero-filled.  One warp per output row.
__global__ void __launch_bounds__(256) unpack_rows_kernel(const float* __restrict__ xp, const int* __restrict__ row_start,
                                                          const int* __restrict__ lens, float* __restrict__ out, int B,
                                                          int S, int H) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= B * S) return;
  const int b = row / S, s = row - b * S;
  float4* dst = reinterpret_cast<float4*>(out + static_cast<size_t>(row) * H);
  if (s < lens[b]) {
    const float4* src = reinterpret_cast<const float4*>(xp + (static_cast<size_t>(row_start[b]) + s) * H);
    for (int i = lane; i < H / 4; i += 32) dst[i] = src[i];
  } else {
    for (int i = lane; i < H / 4; i += 32) dst[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

// K1: LN(word[ids] + pos[s] + type[tt]).  ids / type_ids are int64 [B,S] (padded) as AllenNLP's
// PretrainedTransformerIndexer produces them (SURVEY.md 8b); type_ids == nullptr means all-zero
// (custom_PTM_embedder.py:199-202).  Out-of-range ids are clamped AND reported: bit 1 of *bad is set, which the host
// turns into the error the reference raises (torch.embedding index error; custom_PTM_embedder.py:205 for type ids).
// Padded layout (row_start == nullptr): output row b*S + s for every s < S.
// Packed layout: only s < lens[b] is computed and lands at row row_start[b] + s.  The encoder's kernels also read rows
// past the last token T that none of them writes: whole 256-row GEMM tiles, and the last sequence's ragged key block
// (up to 63 rows past T, which P = 0 multiplies: a NaN there would still poison the sequence).  So the tail blocks
// zero-fill rows [T, round_up(T, 256) + 64) (clipped to the B*S-row buffers) of x32, x16 and of the encoder's scratch
// matrices qkv [*, 3H], ctx [*, H], ffn [*, inter] (each nullable), whatever the memory held before.
constexpr int kEmbedTailBlocks = (256 + 64) / 8;
template <int NV>
__global__ void __launch_bounds__(256) embed_layernorm_kernel(
    const long long* __restrict__ ids, const long long* __restrict__ type_ids, const float* __restrict__ word,
    const float* __restrict__ pos, const float* __restrict__ type, const float* __restrict__ gamma,
    const float* __restrict__ beta, float eps, float* __restrict__ x32, __half* __restrict__ x16, int B, int S,
    int vocab, int type_vocab, const int* __restrict__ lens, const int* __restrict__ row_start, int* __restrict__ bad,
    __half* __restrict__ qkv, __half* __restrict__ ctx, __half* __restrict__ ffn, int inter) {
  constexpr int H = NV * 128;
  const int lane = threadIdx.x & 31;
  const int chunks = (S + 7) >> 3;                          // 8 rows (warps) per block, blocks never straddle sequences
  const int b = blockIdx.x / chunks;
  const int s = (blockIdx.x - b * chunks) * 8 + (threadIdx.x >> 5);
  if (b >= B) {
    // packed layout only: tail blocks, one row per warp
    const int T = row_start[B];
    const size_t r = static_cast<size_t>(T + (blockIdx.x - B * chunks) * 8 + (threadIdx.x >> 5));
    const int end = min((((T + 255) >> 8) << 8) + 64, B * S);
    if (r < static_cast<size_t>(end)) {
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const int col = i * 128 + lane * 4;
        *reinterpret_cast<float4*>(x32 + r * H + col) = make_float4(0.f, 0.f, 0.f, 0.f);
        *reinterpret_cast<uint2*>(x16 + r * H + col) = make_uint2(0u, 0u);
      }
      auto zero_row = [&](__half* m, int cols) {           // 16-byte stores: cols is a multiple of 128
        if (m)
          for (int c = lane * 8; c < cols; c += 256) *reinterpret_cast<uint4*>(m + r * cols + c) = make_uint4(0u, 0u, 0u, 0u);
      };
      zero_row(qkv, 3 * H);
      zero_row(ctx, H);
      zero_row(ffn, inter);
    }
    return;
  }
  if (s >= S || (row_start && s >= lens[b])) return;
  const size_t in_row = static_cast<size_t>(b) * S + s;
  const size_t out_row = row_start ? static_cast<size_t>(row_start[b]) + s : in_row;
  long long id = ids[in_row];
  long long tt = type_ids ? type_ids[in_row] : 0;
  if (id < 0 || id >= vocab || tt < 0 || tt >= type_vocab) {
    if (lane == 0 && bad) atomicOr(bad, 2);
    id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
    tt = tt < 0 ? 0 : (tt >= type_vocab ? type_vocab - 1 : tt);
  }
  const float* w = word + static_cast<size_t>(id) * H;
  const float* p = pos + static_cast<size_t>(s) * H;
  const float* t = type + static_cast<size_t>(tt) * H;
  float4 v[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int col = i * 128 + lane * 4;
    const float4 a = __ldg(reinterpret_cast<const float4*>(w + col));
    const float4 bb = __ldg(reinterpret_cast<const float4*>(p + col));
    const float4 c = __ldg(reinterpret_cast<const float4*>(t + col));
    v[i] = make_float4((a.x + bb.x) + c.x, (a.y + bb.y) + c.y, (a.z + bb.z) + c.z, (a.w + bb.w) + c.w);
  }
  ln_store<NV>(v, gamma, beta, eps, x32 + out_row * H, x16 + out_row * H, lane);
}

}  // namespace mv
