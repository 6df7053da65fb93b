// Token sampling on the device: temperature -> top-k -> softmax -> multinomial, the order of HF's
// TemperatureLogitsWarper / TopKLogitsWarper, over the fp32 logits the logits kernels write. The contract
// (kept set with ties, fp64 weights, Philox4x64-10 stream keyed by the token's position) is stated in
// include/vcl.h above vcl_sampling; tests/_sampling_oracle.py restates it on the host.
//
// One 1024-thread CTA per row:
//   1. max + arg-max (coalesced; NaN counts as -inf). temperature <= 0 stops here: the arg-max with the
//      lowest index winning, the same comparisons as argmax_kernel (elementwise.cu).
//   2. tau = the k-th largest logit: radix select over the order-preserving uint32 image of the floats,
//      4 passes of 8 bits with a shared-memory histogram (k = 1: tau = max; no filter: every id is kept).
//   3. each thread owns a contiguous run of ids, sums exp((l - max) / T) in fp64 over the kept ones in
//      ascending order; a block-wide exclusive scan of those sums gives every run its running-sum start.
//   4. t = u * Z; the thread whose run holds the crossing walks it again and reports the first id whose
//      running sum exceeds t (smallest over threads). No crossing (rounding): the largest kept id.
#include <math.h>

#include "common.cuh"
#include "kernels.h"

namespace vcl {

namespace {

constexpr int SAMPLE_THREADS = 1024;

__device__ __forceinline__ float nan_to_ninf(float x) { return x != x ? -INFINITY : x; }

// order-preserving image: a < b (floats, no NaN)  <=>  fkey(a) < fkey(b)
__device__ __forceinline__ uint32_t fkey(float x) {
  const uint32_t u = __float_as_uint(x);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// Philox4x64-10 (Salmon et al., SC'11), word 0 of the block at counter (c0, c1, 0, 0), key (k0, 0)
__device__ __forceinline__ uint64_t philox4x64_w0(uint64_t k0, uint64_t c0, uint64_t c1) {
  uint64_t x0 = c0, x1 = c1, x2 = 0, x3 = 0, k1 = 0;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r > 0) { k0 += 0x9E3779B97F4A7C15ull; k1 += 0xBB67AE8584CAA73Bull; }
    const uint64_t hi0 = __umul64hi(0xD2E7470EE14C6C93ull, x0), lo0 = 0xD2E7470EE14C6C93ull * x0;
    const uint64_t hi1 = __umul64hi(0xCA5A826395121157ull, x2), lo1 = 0xCA5A826395121157ull * x2;
    x0 = hi1 ^ x1 ^ k0; x1 = lo1; x2 = hi0 ^ x3 ^ k1; x3 = lo0;
  }
  return x0;
}

__global__ void __launch_bounds__(SAMPLE_THREADS)
sample_kernel(const float* __restrict__ logits, long long ld, int V, const SampleParams* __restrict__ params_dev,
              SampleParams params, int pos, const int* __restrict__ pos_dev, int* __restrict__ out,
              long long out_stride) {
  __shared__ float sv[32];
  __shared__ int si[32];
  __shared__ uint32_t hist[256];
  __shared__ uint32_t s_sel[2];          // selected digit, count still to skip below it
  __shared__ double s_wsum[32];
  __shared__ int s_tok, s_last;
  const SampleParams p = params_dev != nullptr ? *params_dev : params;
  const int row = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const float* l = logits + (long long)row * ld;

  // ---- 1. max and arg-max -----------------------------------------------------------------------
  float best = -INFINITY;
  int bi = 0x7fffffff;
  for (int i = tid; i < V; i += SAMPLE_THREADS) {
    const float x = l[i];
    if (x > best) { best = x; bi = i; }            // increasing index: ties keep the lowest
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
  }
  if (lane == 0) { sv[warp] = best; si[warp] = bi; }
  __syncthreads();
  best = sv[lane]; bi = si[lane];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
  }
  const float mx = best;                            // every thread holds the row's max and its lowest index
  if (p.temperature <= 0.f || !(mx > -INFINITY && mx < INFINITY)) {
    // greedy; also a row without a finite maximum (all -inf / NaN: id 0; +inf present: its lowest id)
    if (tid == 0) {
      const int tok = (p.temperature <= 0.f || bi != 0x7fffffff) ? bi : 0;
      out[(long long)row * out_stride] = tok;
    }
    return;
  }

  // ---- 2. tau = k-th largest (counting multiplicity) -------------------------------------------------
  const int k = (p.top_k >= 1 && p.top_k < V) ? p.top_k : V;
  uint32_t tau_key = 0;                            // kept: fkey(l) >= tau_key
  if (k == 1) {
    tau_key = fkey(mx);
  } else if (k < V) {
    uint32_t prefix = 0, pmask = 0, krem = (uint32_t)k;
    for (int shift = 24; shift >= 0; shift -= 8) {
      if (tid < 256) hist[tid] = 0;
      __syncthreads();
      for (int i0 = 0; i0 < V; i0 += SAMPLE_THREADS) {
        const int i = i0 + tid;
        const uint32_t key = i < V ? fkey(nan_to_ninf(l[i])) : 0u;
        const bool take = i < V && (key & pmask) == prefix;
        const uint32_t d = take ? (key >> shift) & 255u : 0x100u;
        const uint32_t peers = __match_any_sync(0xffffffffu, d);
        if (take && lane == __ffs(peers) - 1) atomicAdd(&hist[d], (uint32_t)__popc(peers));
      }
      __syncthreads();
      if (tid < 256) {
        // inclusive scan over the digits in DESCENDING order: thread t holds digit 255 - t
        const uint32_t h = hist[255 - tid];
        uint32_t inc = h;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o);
          if (lane >= o) inc += v;
        }
        if (lane == 31) si[warp] = (int)inc;
        __syncwarp();
        asm volatile("bar.sync 1, 256;" ::: "memory");
        uint32_t base = 0;
        for (int w = 0; w < warp; ++w) base += (uint32_t)si[w];
        inc += base;
        if (inc >= krem && inc - h < krem) { s_sel[0] = 255 - tid; s_sel[1] = krem - (inc - h); }
      }
      __syncthreads();
      prefix |= s_sel[0] << shift;
      pmask |= 255u << shift;
      krem = s_sel[1];
      __syncthreads();                             // s_sel / si / hist are rewritten by the next pass
    }
    tau_key = prefix;
  }

  // ---- 3. fp64 weights over contiguous runs of ids, block exclusive scan ---------------------------------
  const int run = (V + SAMPLE_THREADS - 1) / SAMPLE_THREADS;
  const int i_lo = tid * run, i_hi = min(i_lo + run, V);
  const double mxd = (double)mx, Td = (double)p.temperature;
  double s = 0.0;
  int last = -1;
  for (int i = i_lo; i < i_hi; ++i) {
    const float x = nan_to_ninf(l[i]);
    if (fkey(x) >= tau_key) { s += exp(((double)x - mxd) / Td); last = i; }
  }
  if (tid == 0) { s_tok = 0x7fffffff; s_last = -1; }
  double inc = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const double v = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += v;
  }
  if (lane == 31) s_wsum[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    double w = s_wsum[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double v = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += v;
    }
    s_wsum[lane] = w;                              // inclusive over warps
  }
  __syncthreads();
  const double pre = inc - s + (warp > 0 ? s_wsum[warp - 1] : 0.0);
  const double Z = s_wsum[31];

  // ---- 4. draw and pick ---------------------------------------------------------------------------
  const int tok_pos = pos + (pos_dev != nullptr ? __ldg(pos_dev) : 0);
  const uint64_t r = philox4x64_w0(p.seed, (uint64_t)(long long)tok_pos, (uint64_t)row);
  const double t = (double)(r >> 11) * 0x1.0p-53 * Z;
  if (last >= 0) atomicMax(&s_last, last);
  if (last >= 0 && pre + s > t) {
    double acc = pre;
    for (int i = i_lo; i < i_hi; ++i) {
      const float x = nan_to_ninf(l[i]);
      if (fkey(x) < tau_key) continue;
      acc += exp(((double)x - mxd) / Td);
      if (acc > t) { atomicMin(&s_tok, i); break; }
    }
  }
  __syncthreads();
  if (tid == 0) out[(long long)row * out_stride] = s_tok != 0x7fffffff ? s_tok : s_last;
}

__global__ void set_sample_params_kernel(SampleParams* dst, SampleParams p) { *dst = p; }

}  // namespace

int launch_sample(const float* logits, long long ld, int B, int V, const SampleParams* params_dev,
                  const SampleParams& params, int pos, const int* pos_dev, int* out, long long out_stride,
                  cudaStream_t stream) {
  VCL_REQUIRE(V > 0 && ld >= V, "sample: V=%d ld=%lld", V, ld);
  if (B <= 0) return 0;
  sample_kernel<<<B, SAMPLE_THREADS, 0, stream>>>(logits, ld, V, params_dev, params, pos, pos_dev, out, out_stride);
  VCL_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return 0;
}

int launch_set_sample_params(SampleParams* dst, const SampleParams& p, cudaStream_t stream) {
  set_sample_params_kernel<<<1, 1, 0, stream>>>(dst, p);
  VCL_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return 0;
}

}  // namespace vcl
