// vdb200 — autoregressive Optimus GPT-2 decode (sm_100a): single-query attention over a per-layer KV cache and on-device
// token sampling.  Replaces the per-token loop of sample_single_sequence_conditional (reference lib/model_zoo/optimus.py:662-688),
// which re-runs the whole prefix through GPT2ForLatentConnector_XX (optimus_models/optimus_gpt2.py:813-1112) for every new
// token and samples on the host side of torch.multinomial.  Every kernel reads its position from a device step counter, so one
// captured CUDA graph of the token step serves all steps of a decode.
#include "common.cuh"
#include "host_util.h"

namespace vdb {

constexpr int kDecHead = 64;     // d_head of every Optimus GPT-2 size
constexpr int kDecSlots = 32;    // KV-cache slots per (row, head): max_length 30 tokens fit with room to spare

// ---------------------------------------------------------------------------------------------
// Attention of the newest token (Attention.forward + _attn, optimus_gpt2.py:151-209): one warp per (row, head).
// The latent memory slot (past key == past value == linear(z) slice of this layer, :887-893) is key 0; the cached
// tokens 0..t are keys 1..t+1, so at most 31 keys and one key per lane.  The causal mask of the reference allows exactly
// these keys for the newest query, so no mask is applied.  fp32 scores and softmax; bf16 in and out.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) kv_decode_attention_kernel(
    const __nv_bfloat16* __restrict__ qkv, long long ldqkv, const __nv_bfloat16* __restrict__ mem, long long ldmem,
    __nv_bfloat16* __restrict__ kcache, __nv_bfloat16* __restrict__ vcache, const int* __restrict__ step, int n, int H,
    float scale, __nv_bfloat16* __restrict__ out, long long ldo) {
  const int lane = threadIdx.x & 31;
  const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (w >= n * H) return;
  const int row = w / H, h = w % H;
  const int t = *step;
  if (t < 0 || t > kDecSlots - 2) return;   // a counter past the cache (or the 32 keys a warp holds) is a no-op, never a stray write
  const int C = H * kDecHead;
  const __nv_bfloat16* q = qkv + row * ldqkv + h * kDecHead;
  const __nv_bfloat16* m = mem + row * ldmem + h * kDecHead;
  __nv_bfloat16* kc = kcache + static_cast<long long>(w) * kDecSlots * kDecHead;
  __nv_bfloat16* vc = vcache + static_cast<long long>(w) * kDecSlots * kDecHead;

  // append this token's k / v (2 dims per lane) at slot t
  const int d = 2 * lane;
  *reinterpret_cast<__nv_bfloat162*>(kc + t * kDecHead + d) = *reinterpret_cast<const __nv_bfloat162*>(q + C + d);
  *reinterpret_cast<__nv_bfloat162*>(vc + t * kDecHead + d) = *reinterpret_cast<const __nv_bfloat162*>(q + 2 * C + d);
  __syncwarp();   // orders the appends before the other lanes read them back

  const int nkeys = t + 2;
  float s = -INFINITY;
  if (lane < nkeys) {
    const __nv_bfloat16* kp = lane == 0 ? m : kc + (lane - 1) * kDecHead;
    float acc = 0.f;
#pragma unroll
    for (int c = 0; c < kDecHead; c += 8) {
      const uint4 qa = *reinterpret_cast<const uint4*>(q + c);
      const uint4 ka = *reinterpret_cast<const uint4*>(kp + c);
      const __nv_bfloat162* q2 = reinterpret_cast<const __nv_bfloat162*>(&qa);
      const __nv_bfloat162* k2 = reinterpret_cast<const __nv_bfloat162*>(&ka);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 qf = __bfloat1622float2(q2[j]), kf = __bfloat1622float2(k2[j]);
        acc = fmaf(qf.x, kf.x, acc);
        acc = fmaf(qf.y, kf.y, acc);
      }
    }
    s = acc * scale;
  }
  float mx = s;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  const float e = lane < nkeys ? expf(s - mx) : 0.f;
  float sum = e;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float pr = e / sum;

  float o0 = 0.f, o1 = 0.f;
  for (int j = 0; j < nkeys; ++j) {
    const float pj = __shfl_sync(0xffffffffu, pr, j);
    const __nv_bfloat16* vp = j == 0 ? m : vc + (j - 1) * kDecHead;
    const float2 vf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(vp + d));
    o0 = fmaf(pj, vf.x, o0);
    o1 = fmaf(pj, vf.y, o1);
  }
  *reinterpret_cast<__nv_bfloat162*>(out + row * ldo + h * kDecHead + d) = __floats2bfloat162_rn(o0, o1);
}

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC 2011): counter (row, step, 0, 0), key = seed.
// ---------------------------------------------------------------------------------------------
VDB_DEVINL float philox_uniform(unsigned long long seed, unsigned row, unsigned step) {
  unsigned c0 = row, c1 = step, c2 = 0u, c3 = 0u;
  unsigned k0 = static_cast<unsigned>(seed), k1 = static_cast<unsigned>(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const unsigned hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const unsigned hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const unsigned n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return (static_cast<float>(c0 >> 8) + 0.5f) * (1.0f / 16777216.0f);   // in (0, 1)
}

constexpr int kSampleThreads = 1024;

// next-step input: wte[tok] + wpe[pos] + emb_add[row] (GPT2Model_XX.forward, optimus_gpt2.py:941-951), fp32 sum rounded to bf16
VDB_DEVINL void embed_row(const __nv_bfloat16* __restrict__ wte, const float* __restrict__ wpe, const float* __restrict__ emb_add,
                          long long ld_emb, int row, int tok, int pos, int C, __nv_bfloat16* __restrict__ x, long long ldx) {
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const float v = __bfloat162float(wte[static_cast<long long>(tok) * C + c]) + wpe[static_cast<long long>(pos) * C + c] +
                    emb_add[row * ld_emb + c];
    x[row * ldx + c] = __float2bfloat16_rn(v);
  }
}

// ---------------------------------------------------------------------------------------------
// One CTA per row: softmax(logits / T) and an inverse-CDF draw in vocabulary order (torch.multinomial of optimus.py:678),
// then the EOS / max-length bookkeeping of :680-685 and the embedding of the drawn token for the next step.
// Each thread owns a contiguous vocabulary chunk; the chunk sums are combined in a fixed order, so results are deterministic.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kSampleThreads) sample_tokens_kernel(
    const float* __restrict__ logits, long long ldl, int V, const float* __restrict__ temperature, const int* __restrict__ step,
    const unsigned long long* __restrict__ seed, const float* __restrict__ uniforms, int ldu, const int* __restrict__ forced,
    int eos, int max_len, int* __restrict__ tokens, int ldt, const __nv_bfloat16* __restrict__ wte, const float* __restrict__ wpe,
    const float* __restrict__ emb_add, long long ld_emb, int C, __nv_bfloat16* __restrict__ x_next, long long ldx) {
  __shared__ float red[32];
  __shared__ float scan[kSampleThreads];
  __shared__ int pick, last_nz;
  const int row = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int t = *step;
  if (t < 0 || t + 1 >= ldt) return;        // block-uniform: a counter past the token rows writes nothing
  int tok;
  if (forced) {
    tok = forced[row * ldt + t + 1];
  } else if (tokens[row * ldt + t] == eos) {
    tok = eos;                                      // row already finished: keep it finished
  } else {
    const float T = *temperature;
    const float* lr = logits + row * ldl;
    const int chunk = (V + kSampleThreads - 1) / kSampleThreads;
    const int i0 = min(V, tid * chunk), i1 = min(V, i0 + chunk);
    float mx = -INFINITY;
    for (int i = i0; i < i1; ++i) mx = fmaxf(mx, lr[i] / T);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if (lane == 0) red[wid] = mx;
    if (tid == 0) { pick = 0x7fffffff; last_nz = -1; }
    __syncthreads();
    mx = red[0];
    for (int k = 1; k < kSampleThreads / 32; ++k) mx = fmaxf(mx, red[k]);
    float part = 0.f;
    int my_last = -1;
    for (int i = i0; i < i1; ++i) {
      const float e = expf(lr[i] / T - mx);
      part += e;
      if (e > 0.f) my_last = i;
    }
    scan[tid] = part;
    if (my_last >= 0) atomicMax(&last_nz, my_last);
    __syncthreads();
    // fixed-order inclusive scan of the chunk sums (Hillis-Steele over shared memory)
    for (int o = 1; o < kSampleThreads; o <<= 1) {
      const float v = tid >= o ? scan[tid - o] : 0.f;
      __syncthreads();
      scan[tid] += v;
      __syncthreads();
    }
    const float total = scan[kSampleThreads - 1];
    const float u = uniforms ? uniforms[row * ldu + t] : philox_uniform(*seed, static_cast<unsigned>(row), static_cast<unsigned>(t));
    const float target = u * total;
    // the inclusive scan values partition [0, total) between the threads, so exactly one thread owns the target
    const float lo = tid ? scan[tid - 1] : 0.f;
    if (lo <= target && target < scan[tid]) {
      const float local = target - lo;
      float run = 0.f;
      int sel = my_last;                            // the chunk's last non-zero entry if rounding leaves the crossing unmet
      for (int i = i0; i < i1; ++i) {
        run += expf(lr[i] / T - mx);
        if (run > local) { sel = i; break; }
      }
      atomicMin(&pick, sel);
    }
    __syncthreads();
    tok = pick >= 0 && pick != 0x7fffffff ? pick : last_nz;   // rounding can leave the target at the very top of the CDF
    if (t + 2 >= max_len) tok = eos;                // the last slot of a full-length sequence is overwritten with EOS
  }
  if (tid == 0) tokens[row * ldt + t + 1] = tok;
  if (x_next) embed_row(wte, wpe, emb_add, ld_emb, row, tok, t + 2, C, x_next, ldx);
}

__global__ void token_embed_kernel(const int* __restrict__ tokens, int ldt, const int* __restrict__ step, int pos_offset,
                                   const __nv_bfloat16* __restrict__ wte, const float* __restrict__ wpe,
                                   const float* __restrict__ emb_add, long long ld_emb, int C, __nv_bfloat16* __restrict__ x,
                                   long long ldx) {
  const int row = blockIdx.x;
  const int t = step ? *step : 0;
  embed_row(wte, wpe, emb_add, ld_emb, row, tokens[row * ldt + t], t + pos_offset, C, x, ldx);
}

}  // namespace vdb

using namespace vdb;

extern "C" {

int vdb_kv_decode_attention(const void* qkv, long long ldqkv, const void* mem, long long ldmem, void* kcache, void* vcache,
                            const int* step, int n, int H, float scale, void* out, long long ldo, void* stream) {
  if (!qkv || !mem || !kcache || !vcache || !step || !out || n <= 0 || H <= 0)
    return set_error(VDB_ERR_INVALID, "kv_decode_attention: null/empty argument");
  if ((ldqkv % 8) || (ldmem % 8) || (ldo % 2) || ldqkv < 3LL * H * kDecHead || ldo < 1LL * H * kDecHead)
    return set_error(VDB_ERR_INVALID, "kv_decode_attention: ldqkv / ldmem must be multiples of 8, ldqkv >= 3*H*64, ldo >= H*64");
  if ((reinterpret_cast<uintptr_t>(qkv) | reinterpret_cast<uintptr_t>(mem)) & 15)
    return set_error(VDB_ERR_INVALID, "kv_decode_attention: qkv / mem must be 16-byte aligned");
  const int warps = n * H;
  kv_decode_attention_kernel<<<(warps + 3) / 4, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const __nv_bfloat16*>(qkv), ldqkv, reinterpret_cast<const __nv_bfloat16*>(mem), ldmem,
      reinterpret_cast<__nv_bfloat16*>(kcache), reinterpret_cast<__nv_bfloat16*>(vcache), step, n, H, scale,
      reinterpret_cast<__nv_bfloat16*>(out), ldo);
  VDB_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return VDB_OK;
}

int vdb_sample_tokens(const float* logits, long long ldl, int V, int n, const float* temperature, const int* step,
                      const unsigned long long* seed, const float* uniforms, int ldu, const int* forced, int eos, int max_len,
                      int* tokens, int ldt, const void* wte, const float* wpe, const float* emb_add, long long ld_emb, int C,
                      void* x_next, long long ldx, void* stream) {
  if (!step || !tokens || n <= 0 || max_len < 2 || ldt < max_len)
    return set_error(VDB_ERR_INVALID, "sample_tokens: null/empty argument or ldt < max_len");
  if (!forced && (!logits || V <= 0 || ldl < V || !temperature || (!uniforms && !seed)))
    return set_error(VDB_ERR_INVALID, "sample_tokens: sampling needs logits (ldl >= V), temperature and a seed or uniforms");
  if (x_next && (!wte || !wpe || !emb_add || C <= 0))
    return set_error(VDB_ERR_INVALID, "sample_tokens: the next-step embedding needs wte, wpe and emb_add");
  sample_tokens_kernel<<<n, kSampleThreads, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      logits, ldl, V, temperature, step, seed, uniforms, ldu, forced, eos, max_len, tokens, ldt,
      reinterpret_cast<const __nv_bfloat16*>(wte), wpe, emb_add, ld_emb, C, reinterpret_cast<__nv_bfloat16*>(x_next), ldx);
  VDB_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return VDB_OK;
}

int vdb_token_embed(const int* tokens, int ldt, const int* step, int pos_offset, const void* wte, const float* wpe,
                    const float* emb_add, long long ld_emb, int n, int C, void* x, long long ldx, void* stream) {
  if (!tokens || !wte || !wpe || !emb_add || !x || n <= 0 || C <= 0)
    return set_error(VDB_ERR_INVALID, "token_embed: null/empty argument");
  token_embed_kernel<<<n, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      tokens, ldt, step, pos_offset, reinterpret_cast<const __nv_bfloat16*>(wte), wpe, emb_add, ld_emb, C,
      reinterpret_cast<__nv_bfloat16*>(x), ldx);
  VDB_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return VDB_OK;
}

}  // extern "C"
