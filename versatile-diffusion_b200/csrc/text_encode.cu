// vdb200 — the embedding layer of the Optimus BERT text encoder (sm_100a).  Replaces BertEmbeddings.forward (reference
// lib/model_zoo/optimus_models/optimus_bert.py:144-175) as optimus_vae_next.encode calls it (optimus.py:729-743: no position
// or token-type ids, so positions 0.. and token type 0): LayerNorm(word[id] + position[j] + token_type[0]) in fp32, one bf16
// row per token.  The encoder layers after it run on vdb_gemm_bf16 / vdb_attention_keylen_bf16 / vdb_layernorm.
#include "common.cuh"
#include "host_util.h"

namespace vdb {

constexpr int kEmbedMaxVec = 8;   // float4 columns per lane: C <= 32 * 4 * 8 = 1024

// One warp per token row.  Lane l owns the float4 columns l, l + 32, ... of the row, so the three fp32 table rows are read
// in place (coalesced 512-byte warp loads) and the sum stays in registers for both LayerNorm passes.
__global__ void __launch_bounds__(256) bert_embed_ln_kernel(
    const int* __restrict__ ids, long long rows, int L, int vocab, const float* __restrict__ word,
    const float* __restrict__ pos, const float* __restrict__ type0, const float* __restrict__ gamma,
    const float* __restrict__ beta, float eps, int C, __nv_bfloat16* __restrict__ y) {
  const long long row = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const int j = static_cast<int>(row % L);
  const int id = min(max(__ldg(ids + row), 0), vocab - 1);   // an id outside the table reads a valid row, never a stray one
  const int nv = C >> 7;                                     // float4 columns per lane
  const float4* w4 = reinterpret_cast<const float4*>(word + static_cast<long long>(id) * C);
  const float4* p4 = reinterpret_cast<const float4*>(pos + static_cast<long long>(j) * C);
  const float4* t4 = reinterpret_cast<const float4*>(type0);
  float4 e[kEmbedMaxVec];
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < kEmbedMaxVec; ++k) {
    if (k < nv) {
      const int c = lane + 32 * k;
      const float4 a = __ldg(w4 + c), b = __ldg(p4 + c), t = __ldg(t4 + c);
      e[k] = make_float4((a.x + b.x) + t.x, (a.y + b.y) + t.y, (a.z + b.z) + t.z, (a.w + b.w) + t.w);
      s += (e[k].x + e[k].y) + (e[k].z + e[k].w);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float inv_c = 1.0f / static_cast<float>(C);
  const float mean = s * inv_c;
  float q = 0.f;
#pragma unroll
  for (int k = 0; k < kEmbedMaxVec; ++k) {
    if (k < nv) {
      const float dx = e[k].x - mean, dy = e[k].y - mean, dz = e[k].z - mean, dw = e[k].w - mean;
      q += (dx * dx + dy * dy) + (dz * dz + dw * dw);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  const float rstd = rsqrtf(q * inv_c + eps);
  const float4* g4 = reinterpret_cast<const float4*>(gamma);
  const float4* b4 = reinterpret_cast<const float4*>(beta);
  uint2* yrow = reinterpret_cast<uint2*>(y + row * C);
#pragma unroll
  for (int k = 0; k < kEmbedMaxVec; ++k) {
    if (k < nv) {
      const int c = lane + 32 * k;
      const float4 g = __ldg(g4 + c), b = __ldg(b4 + c);
      yrow[c] = make_uint2(pack_bf16x2((e[k].x - mean) * rstd * g.x + b.x, (e[k].y - mean) * rstd * g.y + b.y),
                           pack_bf16x2((e[k].z - mean) * rstd * g.z + b.z, (e[k].w - mean) * rstd * g.w + b.w));
    }
  }
}

}  // namespace vdb

using namespace vdb;

extern "C" {

int vdb_bert_embed_ln(const int* ids, int n, int L, const float* word_emb, int vocab, const float* pos_emb, int max_pos,
                      const float* type_emb, const float* gamma, const float* beta, float eps, int C, void* y, void* stream) {
  if (!ids || !word_emb || !pos_emb || !type_emb || !gamma || !beta || !y || n <= 0 || L <= 0 || vocab <= 0)
    return set_error(VDB_ERR_INVALID, "bert_embed_ln: null/empty argument");
  if (C <= 0 || (C % 128) || C > 32 * 4 * kEmbedMaxVec)
    return set_error(VDB_ERR_INVALID, "bert_embed_ln: width %d must be a multiple of 128 and <= %d", C, 32 * 4 * kEmbedMaxVec);
  if (L > max_pos)
    return set_error(VDB_ERR_INVALID, "bert_embed_ln: %d positions but the position table has %d rows", L, max_pos);
  if ((reinterpret_cast<uintptr_t>(word_emb) | reinterpret_cast<uintptr_t>(pos_emb) | reinterpret_cast<uintptr_t>(type_emb) |
       reinterpret_cast<uintptr_t>(gamma) | reinterpret_cast<uintptr_t>(beta) | reinterpret_cast<uintptr_t>(y)) & 15)
    return set_error(VDB_ERR_INVALID, "bert_embed_ln: tables, gamma, beta and y must be 16-byte aligned");
  const long long rows = static_cast<long long>(n) * L;
  const long long blocks = (rows + 7) / 8;   // 8 warps (rows) per 256-thread block
  bert_embed_ln_kernel<<<static_cast<unsigned>(blocks), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      ids, rows, L, vocab, word_emb, pos_emb, type_emb, gamma, beta, eps, C, reinterpret_cast<__nv_bfloat16*>(y));
  VDB_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return VDB_OK;
}

}  // extern "C"
