// Device-side token sampler and the per-step bookkeeping of the on-device generation loop.
//
// Replaces stripedhyena.sample.sample (call site evo/generation.py:162-167) and the host half of the token loop
// (evo/generation.py:131-189: pick token, store logits/token, feed the token back): greedy when top_k == 1, else
// top-k -> / temperature -> top-p tail mask -> multinomial, 512-way per row.  The reference draws from torch's
// global RNG, so only the greedy path can be bit-identical; the sampling path reproduces the DISTRIBUTION
// (tests/test_gpu_parity.py checks the kept set and a chi-square of the draws against the host implementation) with
// a counter-based Philox4x32-10 stream keyed by (seed, step, row), which makes a generation reproducible under
// CUDA-graph replay (no host RNG state inside the loop).
//
// One CTA per row, one thread per vocabulary entry (V <= 1024):
//   rank of every entry by counting (V^2 broadcast compares from shared memory; stable: ties -> lower index first),
//   top-k = ranks < k, bf16-rounded temperature division like the reference's bf16 tensor op, softmax over the kept
//   set, suffix sums (Hillis-Steele) for the "cumulative mass from the smallest up" top-p mask, inverse-CDF draw.
#include "common.cuh"
#include "../../include/evo_b200.h"

using namespace evo;

namespace {

constexpr int MAXV = 1024;

__device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
  const uint32_t hi0 = __umulhi(M0, c[0]), lo0 = M0 * c[0];
  const uint32_t hi1 = __umulhi(M1, c[2]), lo1 = M1 * c[2];
  const uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
  c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
}
// uniform in [0, 1) from Philox4x32-10 keyed by seed, counter (step, row)
__device__ __forceinline__ float philox_uniform(uint64_t seed, uint64_t step, uint32_t row) {
  uint32_t c[4] = {(uint32_t)step, (uint32_t)(step >> 32), row, 0x45564f32u};
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) { philox_round(c, k0, k1); k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
  return (float)(c[0] >> 8) * (1.0f / 16777216.0f);
}

struct SampleCfg { int top_k; float top_p; float temperature; unsigned long long seed; };

// returns the chosen vocabulary index (valid in every thread)
__device__ int sample_row(const bf16* __restrict__ logits, int V, const SampleCfg cfg, uint64_t step, uint32_t row) {
  __shared__ float s_val[MAXV];        // logits by index, later: by rank
  __shared__ int s_idx[MAXV];          // index by rank
  __shared__ float s_scan[2][MAXV];
  __shared__ float s_red[33];
  __shared__ int s_pick;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5, nwarp = blockDim.x >> 5;
  const float mine = t < V ? __bfloat162float(logits[t]) : -INFINITY;
  s_val[t] = mine;
  __syncthreads();
  // stable descending rank: entries strictly greater, or equal with a lower index, come first (argmax = rank 0 = first maximum)
  int rank = 0;
  if (t < V) {
    for (int j = 0; j < V; ++j) {
      const float o = s_val[j];
      rank += (o > mine) || (o == mine && j < t);
    }
    if (mine != mine) rank = V - 1;    // NaN logits sort last (never picked unless everything is NaN)
  }
  __syncthreads();
  if (cfg.top_k == 1) {
    if (t < V && rank == 0) s_pick = t;
    __syncthreads();
    return s_pick;
  }
  const int k = cfg.top_k > 0 ? min(cfg.top_k, V) : V;
  // by rank; the temperature division is a bf16 tensor op in the reference (kept / temperature on bf16 logits)
  float scaled = mine;
  if (cfg.temperature != 1.0f) scaled = rbf(mine / cfg.temperature);
  if (t < V) { s_idx[rank] = t; s_scan[0][rank] = scaled; }
  __syncthreads();
  const bool kept = t < k;
  const float v = kept ? s_scan[0][t] : -INFINITY;       // thread t now owns RANK t
  const float vmax = s_scan[0][0];
  __syncthreads();
  // softmax over the kept set
  float e = kept ? __expf(v - vmax) : 0.f;
  float sum = e;
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
  if (lane == 0) s_red[warp] = sum;
  __syncthreads();
  if (warp == 0) {
    float w = lane < nwarp ? s_red[lane] : 0.f;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) w += __shfl_xor_sync(0xffffffffu, w, off);
    if (lane == 0) s_red[32] = w;
  }
  __syncthreads();
  const float total = s_red[32];
  float p = e / total;
  bool alive = kept;
  if (cfg.top_p > 0.f && cfg.top_p < 1.f) {
    // mass of this entry and of everything smaller (ranks >= t): suffix sum; dropped when <= 1 - top_p
    int cur = 0;
    s_scan[0][t] = p;
    __syncthreads();
    for (int off = 1; off < (int)blockDim.x; off <<= 1) {
      const float add = (t + off < (int)blockDim.x) ? s_scan[cur][t + off] : 0.f;
      s_scan[cur ^ 1][t] = s_scan[cur][t] + add;
      cur ^= 1;
      __syncthreads();
    }
    alive = kept && !(s_scan[cur][t] <= 1.0f - cfg.top_p);
    __syncthreads();
  }
  // renormalised inverse CDF over the surviving entries in rank order (prefix sums)
  {
    int cur = 0;
    s_scan[0][t] = alive ? e : 0.f;
    __syncthreads();
    for (int off = 1; off < (int)blockDim.x; off <<= 1) {
      const float add = (t >= off) ? s_scan[cur][t - off] : 0.f;
      s_scan[cur ^ 1][t] = s_scan[cur][t] + add;
      cur ^= 1;
      __syncthreads();
    }
    const float incl = s_scan[cur][t];
    const float mass = s_scan[cur][blockDim.x - 1];
    const float u = philox_uniform(cfg.seed, step, row) * mass;
    if (t == 0) s_pick = s_idx[0];                        // fallback (u == mass by rounding)
    __syncthreads();
    const float excl = incl - (alive ? e : 0.f);
    if (alive && u >= excl && u < incl) s_pick = s_idx[t];
    __syncthreads();
  }
  return s_pick;
}

__global__ void __launch_bounds__(MAXV) sample_kernel(const bf16* __restrict__ logits, long long* __restrict__ out, int V, SampleCfg cfg, unsigned long long step) {
  const int row = blockIdx.x;
  const int pick = sample_row(logits + (long long)row * V, V, cfg, step, row);
  if (threadIdx.x == 0) out[row] = pick;
}

// one step of the on-device loop: token = forced[:, i] while i < n_forced, else sampled; logits / token recorded for
// generated positions; the token is written back into the step's input buffer.  i = *step_dev.
__global__ void __launch_bounds__(MAXV) sample_step_kernel(const bf16* __restrict__ logits, long long* __restrict__ x, int V,
                                                          const evo_loop_params* __restrict__ lp, const long long* __restrict__ step_dev) {
  pdl_launch_dependents(); pdl_wait();
  const int row = blockIdx.x;
  const long long i = *step_dev;
  const evo_loop_params P = *lp;
  long long tok;
  if (i < P.n_forced) {
    tok = P.forced[(long long)row * P.forced_stride + i];
  } else {
    const SampleCfg cfg = {P.top_k, P.top_p, P.temperature, (unsigned long long)P.seed};
    tok = sample_row(logits + (long long)row * V, V, cfg, (uint64_t)(P.step0 + i), row);
    const long long k = i - P.n_forced;
    if (k < P.n_out) {
      if (threadIdx.x == 0 && P.picked) P.picked[(long long)row * P.picked_stride + k] = tok;
      if (P.kept_logits && threadIdx.x < V)
        P.kept_logits[((long long)row * P.n_out + k) * V + threadIdx.x] = __bfloat162float(logits[(long long)row * V + threadIdx.x]);
    }
  }
  if (threadIdx.x == 0) x[row] = tok;
}

// one step of the ragged loop: row b has its own forced prefix and its own number of recorded tokens.  A row whose
// steps are done (i >= n_forced[b] + n_out[b]) neither samples nor records, and keeps its input token.
__global__ void __launch_bounds__(MAXV) sample_step_rows_kernel(const bf16* __restrict__ logits, long long* __restrict__ x, int V,
                                                               const evo_ragged_loop_params* __restrict__ lp, const long long* __restrict__ step_dev) {
  pdl_launch_dependents(); pdl_wait();
  const int row = blockIdx.x;
  const long long i = *step_dev;
  const evo_ragged_loop_params P = *lp;
  const long long nf = P.n_forced[row], no = P.n_out[row];
  long long tok;
  if (i < nf) {
    tok = P.forced[(long long)row * P.forced_stride + i];
  } else {
    const long long k = i - nf;
    if (k >= no) return;                                             // uniform per CTA
    const SampleCfg cfg = {P.top_k, P.top_p, P.temperature, (unsigned long long)P.seed};
    tok = sample_row(logits + (long long)row * V, V, cfg, (uint64_t)i, row);
    const long long col = P.out_cols - no + k;                        // the row's tokens fill its last n_out columns
    if (threadIdx.x == 0 && P.picked) P.picked[(long long)row * P.out_cols + col] = tok;
    if (P.kept_logits && threadIdx.x < V)
      P.kept_logits[((long long)row * P.out_cols + col) * V + threadIdx.x] = __bfloat162float(logits[(long long)row * V + threadIdx.x]);
  }
  if (threadIdx.x == 0) x[row] = tok;
}

// step += 1; pos[b] = start[b] + min(step, steps_b - 1): a finished row stays at the position of its last step
__global__ void ragged_advance_kernel(long long* __restrict__ pos, long long* __restrict__ step, const evo_ragged_loop_params* __restrict__ lp, int B) {
  pdl_launch_dependents(); pdl_wait();
  const long long s = *step + 1;
  __syncthreads();                                                    // every thread has read the old step
  const int b = threadIdx.x;
  if (b < B) {
    const long long steps = lp->n_forced[b] + lp->n_out[b];
    pos[b] = lp->start[b] + max(0LL, min(s, steps - 1));
  }
  if (b == 0) *step = s;
}

__global__ void advance2_kernel(long long* a, long long* b, long long delta) {
  pdl_launch_dependents(); pdl_wait();
  if (threadIdx.x == 0) { if (a) *a += delta; if (b) *b += delta; }
}

}  // namespace

extern "C" int evo_sample(const void* logits, int64_t* out, int B, int V, int top_k, float top_p, float temperature,
                          uint64_t seed, uint64_t step, void* stream) {
  EVO_REQUIRE(V > 0 && V <= MAXV, "evo_sample: vocabulary %d unsupported (<= %d)", V, MAXV);
  EVO_REQUIRE(!(top_p > 1.0f), "evo_sample: top-p should be in (0, 1]");
  EVO_REQUIRE(temperature > 0.f || top_k == 1, "evo_sample: temperature must be positive");
  if (B == 0) return 0;
  const SampleCfg cfg = {top_k, top_p, temperature, (unsigned long long)seed};
  sample_kernel<<<B, (V + 31) / 32 * 32, 0, (cudaStream_t)stream>>>((const bf16*)logits, (long long*)out, V, cfg, (unsigned long long)step);
  return check_launch("evo_sample");
}

extern "C" int evo_sample_step(const void* logits, int64_t* x, int B, int V, const evo_loop_params* loop_params_dev,
                               const int64_t* step_dev, void* stream) {
  EVO_REQUIRE(V > 0 && V <= MAXV, "evo_sample_step: vocabulary %d unsupported (<= %d)", V, MAXV);
  if (B == 0) return 0;
  EVO_CUDA(launch_pdl(sample_step_kernel, dim3(B), dim3((V + 31) / 32 * 32), 0, (cudaStream_t)stream, (const bf16*)logits, (long long*)x, V,
                      loop_params_dev, (const long long*)step_dev));
  return check_launch("evo_sample_step");
}

extern "C" int evo_sample_step_rows(const void* logits, int64_t* x, int B, int V, const evo_ragged_loop_params* loop_params_dev,
                                    const int64_t* step_dev, void* stream) {
  EVO_REQUIRE(V > 0 && V <= MAXV, "evo_sample_step_rows: vocabulary %d unsupported (<= %d)", V, MAXV);
  EVO_REQUIRE(B >= 0 && B <= 65535, "evo_sample_step_rows: bad batch %d", B);
  if (B == 0) return 0;
  EVO_CUDA(launch_pdl(sample_step_rows_kernel, dim3(B), dim3((V + 31) / 32 * 32), 0, (cudaStream_t)stream, (const bf16*)logits, (long long*)x, V,
                      loop_params_dev, (const long long*)step_dev));
  return check_launch("evo_sample_step_rows");
}

extern "C" int evo_ragged_advance(int64_t* pos, int64_t* step, const evo_ragged_loop_params* loop_params_dev, int B, void* stream) {
  EVO_REQUIRE(B >= 1 && B <= 1024, "evo_ragged_advance: batch %d unsupported (1..1024)", B);
  EVO_CUDA(launch_pdl(ragged_advance_kernel, dim3(1), dim3((B + 31) / 32 * 32), 0, (cudaStream_t)stream, (long long*)pos, (long long*)step,
                      loop_params_dev, B));
  return check_launch("evo_ragged_advance");
}

extern "C" int evo_advance_counters(int64_t* a, int64_t* b, int64_t delta, void* stream) {
  EVO_CUDA(launch_pdl(advance2_kernel, dim3(1), dim3(32), 0, (cudaStream_t)stream, (long long*)a, (long long*)b, (long long)delta));
  return check_launch("evo_advance_counters");
}
