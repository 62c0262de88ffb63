// Decode-step kernels (one new token per sequence): everything a CUDA-graph replay of the
// step needs, with the sequence position read from DEVICE memory so the same captured graph
// serves every step (the reference re-launches ~20 tiny kernels per layer per token from
// Python, SURVEY.md 8a row a9/a12).
#include "common.cuh"
#include "../../include/evo_b200.h"
#include <cstdlib>

using namespace evo;

namespace {

constexpr int HD = 128;

__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }

// out[m, g*128 + c] = bf16(gelu(t[m, g*256 + c])) * t[m, g*256 + 128 + c]   (t = [l1 | l2] interleaved GEMM output)
__global__ void gelu_gate_kernel(const bf16* __restrict__ t, bf16* __restrict__ out, long long M, int ipad) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;      // (m, pair of columns)
  long long total = M * (ipad / 2);
  if (idx >= total) return;
  int c2 = (int)(idx % (ipad / 2)) * 2;
  long long m = idx / (ipad / 2);
  int g = c2 / 128, c = c2 % 128;
  const uint32_t a = *reinterpret_cast<const uint32_t*>(t + m * 2 * ipad + g * 256 + c);
  const uint32_t b = *reinterpret_cast<const uint32_t*>(t + m * 2 * ipad + g * 256 + 128 + c);
  float o0 = rbf(gelu_erf(bf_lo(a))) * bf_lo(b), o1 = rbf(gelu_erf(bf_hi(a))) * bf_hi(b);
  *reinterpret_cast<uint32_t*>(out + m * ipad + c2) = pack_bf16(o0, o1);
}

// L == 1: rotary on q,k at position *pos, k,v appended to the cache at row *pos.
// qkv (B, 3, H, 128) in place; cos/sin tables indexed by absolute position.
// ROWS: pos_ptr is a (B) vector and row b uses pos_ptr[b] (ragged batches); otherwise one position for the batch.
template <bool ROWS>
__global__ void decode_qkv_prep_kernel(bf16* __restrict__ qkv, bf16* __restrict__ cache, const bf16* __restrict__ cos, const bf16* __restrict__ sin,
                                       const long long* __restrict__ pos_ptr, int B, int H, long long max_seqlen) {
  pdl_launch_dependents(); pdl_wait();
  int idx = blockIdx.x * blockDim.x + threadIdx.x;       // (b, h, i) i in [0, 64)
  if (idx >= B * H * 64) return;
  int i = idx % 64, h = (idx / 64) % H, b = idx / (64 * H);
  const long long pos = pos_ptr[ROWS ? b : 0];
  if (pos < 0 || pos >= max_seqlen) return;
  const float c = __bfloat162float(cos[pos * 64 + i]), s = __bfloat162float(sin[pos * 64 + i]);
  bf16* q = qkv + ((long long)(b * 3 + 0) * H + h) * HD;
  bf16* k = qkv + ((long long)(b * 3 + 1) * H + h) * HD;
  const bf16* v = qkv + ((long long)(b * 3 + 2) * H + h) * HD;
  float q0 = __bfloat162float(q[i]), q1 = __bfloat162float(q[i + 64]);
  float k0 = __bfloat162float(k[i]), k1 = __bfloat162float(k[i + 64]);
  bf16 kr0 = __float2bfloat16_rn(k0 * c - k1 * s), kr1 = __float2bfloat16_rn(k0 * s + k1 * c);
  q[i] = __float2bfloat16_rn(q0 * c - q1 * s);
  q[i + 64] = __float2bfloat16_rn(q0 * s + q1 * c);
  k[i] = kr0; k[i + 64] = kr1;
  bf16* ck = cache + (((long long)b * max_seqlen + pos) * 2 + 0) * H * HD + (long long)h * HD;
  bf16* cv = ck + (long long)H * HD;
  ck[i] = kr0; ck[i + 64] = kr1;
  cv[i] = v[i]; cv[i + 64] = v[i + 64];
}

// Single-query attention over the KV cache, keys [0, *pos].  grid (H, B, nsplit); each CTA scans a
// contiguous key range: thread t owns keys t, t+128, ... of the range (one 256-byte K row and one
// V row per key), keeps an online-softmax state and a 128-wide fp32 accumulator in registers, and the
// 128 partial states are merged through shared memory; splits are merged by the last kernel.
constexpr int DT = 128;
template <bool ROWS>
__global__ void __launch_bounds__(DT) decode_attn_kernel(const bf16* __restrict__ qkv, const bf16* __restrict__ cache, float* __restrict__ part_o,
                                                         float* __restrict__ part_ml, const long long* __restrict__ pos_ptr,
                                                         int H, long long max_seqlen, int nsplit, float scale) {
  pdl_launch_dependents(); pdl_wait();
  const int h = blockIdx.x, b = blockIdx.y, sp = blockIdx.z, tid = threadIdx.x;
  const long long nk = min(pos_ptr[ROWS ? b : 0] + 1, max_seqlen);
  const long long per = (nk + nsplit - 1) / nsplit;
  const long long k0 = (long long)sp * per, k1 = min(nk, k0 + per);
  __shared__ float qs[HD];
  __shared__ float red_m[DT], red_l[DT];
  __shared__ float red_o[32][HD + 1];
  qs[tid] = __bfloat162float(qkv[((long long)(b * 3) * H + h) * HD + tid]) * scale;
  __syncthreads();
  float m = -INFINITY, l = 0.f, o[HD];
#pragma unroll
  for (int d = 0; d < HD; ++d) o[d] = 0.f;
  const long long row_stride = 2LL * H * HD;
  const bf16* kb = cache + ((long long)b * max_seqlen) * row_stride + (long long)h * HD;
  for (long long j = k0 + tid; j < k1; j += DT) {
    const uint4* kr = reinterpret_cast<const uint4*>(kb + j * row_stride);
    const uint4* vr = reinterpret_cast<const uint4*>(kb + j * row_stride + (long long)H * HD);
    float sdot = 0.f;
#pragma unroll
    for (int c = 0; c < HD / 8; ++c) {
      uint4 kv = __ldg(kr + c);
      const uint32_t* w = reinterpret_cast<const uint32_t*>(&kv);
#pragma unroll
      for (int e = 0; e < 4; ++e) { sdot = fmaf(qs[c * 8 + 2 * e], bf_lo(w[e]), sdot); sdot = fmaf(qs[c * 8 + 2 * e + 1], bf_hi(w[e]), sdot); }
    }
    const float mn = fmaxf(m, sdot);
    const float alpha = __expf(m - mn), p = __expf(sdot - mn);
    const float pb = rbf(p);                      // P rounded to bf16 before the PV product, like the prefill kernel
    l = l * alpha + p;
#pragma unroll
    for (int c = 0; c < HD / 8; ++c) {
      uint4 vv = __ldg(vr + c);
      const uint32_t* w = reinterpret_cast<const uint32_t*>(&vv);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        o[c * 8 + 2 * e] = fmaf(pb, bf_lo(w[e]), o[c * 8 + 2 * e] * alpha);
        o[c * 8 + 2 * e + 1] = fmaf(pb, bf_hi(w[e]), o[c * 8 + 2 * e + 1] * alpha);
      }
    }
    m = mn;
  }
  // merge the 128 per-thread states: common max, rescale, then reduce 32 threads at a time through smem
  red_m[tid] = m;
  __syncthreads();
  float M = -INFINITY;
  for (int i = 0; i < DT; ++i) M = fmaxf(M, red_m[i]);
  const float sc = (m == -INFINITY) ? 0.f : __expf(m - M);
  red_l[tid] = l * sc;
  __syncthreads();
  float acc = 0.f;                                 // thread tid owns output dim tid
  for (int round = 0; round < DT / 32; ++round) {
    if (tid / 32 == round) {
#pragma unroll
      for (int d = 0; d < HD; ++d) red_o[tid % 32][d] = o[d] * sc;
    }
    __syncthreads();
    for (int i = 0; i < 32; ++i) acc += red_o[i][tid];
    __syncthreads();
  }
  float L = 0.f;
  for (int i = 0; i < DT; ++i) L += red_l[i];
  const long long pidx = ((long long)b * H + h) * nsplit + sp;
  part_o[pidx * HD + tid] = acc;
  if (tid == 0) { part_ml[pidx * 2] = M; part_ml[pidx * 2 + 1] = L; }
}

// ---- decode attention, TMA-fed (default when max_seqlen % 64 == 0) ----
// The per-thread-row kernel above issues 16-byte loads whose 32 lanes touch 32 different 128-byte lines (K rows of
// one head are 16 KB apart): the L1 tag stage caps it near 3 TB/s.  Here a producer warp streams 64-key K and V tiles
// of one (b, h) into a 3-stage shared-memory ring with TMA (box {128, 1, 64} of the cache viewed as
// (hd, 2H, B*S)), and four independent compute warps each own 16 keys of every tile: QK with lane = (key, half
// row) reading rotated 16-byte chunks (conflict-free), a warp-local online softmax, PV with lane = 4 output dims.
// The warps' (m, l, o) states are merged once at the end; splits are merged by decode_attn_merge_kernel.
constexpr int TK = 64;                 // keys per tile
constexpr int AST = 3;                 // ring stages
constexpr int TILE_BYTES = TK * HD * 2;          // 16 KB (K) + 16 KB (V) per stage
constexpr int ATT2_SMEM = AST * 2 * TILE_BYTES + 1024;
template <bool ROWS>
__global__ void __launch_bounds__(160, 2) decode_attn_tma_kernel(const __grid_constant__ CUtensorMap tm, const bf16* __restrict__ qkv,
                                                                 float* __restrict__ part_o, float* __restrict__ part_ml,
                                                                 const long long* __restrict__ pos_ptr, int H, long long S, int nsplit, float scale) {
  pdl_launch_dependents(); pdl_wait();
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + AST * 2 * TILE_BYTES);
  uint64_t* empty = full + AST;
  bf16* qb = reinterpret_cast<bf16*>(empty + AST);                   // 256 B
  float* red = reinterpret_cast<float*>(qb + HD);                      // [4][2] (m, l) then [4][128] o, overlaid on stage 0 after the loop
  const int h = blockIdx.x, b = blockIdx.y, sp = blockIdx.z, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long long nk = min(pos_ptr[ROWS ? b : 0] + 1, S);
  long long per = (nk + nsplit - 1) / nsplit;
  per = (per + TK - 1) / TK * TK;                                      // splits start on tile boundaries
  const long long k0 = (long long)sp * per, k1 = min(nk, k0 + per);
  const int ntiles = k1 > k0 ? (int)((k1 - k0 + TK - 1) / TK) : 0;
  if (tid == 0) {
    for (int i = 0; i < AST; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 4); }
    fence_barrier_init();
  }
  if (tid < HD) qb[tid] = qkv[((long long)(b * 3) * H + h) * HD + tid];
  __syncthreads();

  float m = -INFINITY, l = 0.f, o0 = 0.f, o1 = 0.f, o2 = 0.f, o3 = 0.f;
  if (warp == 4) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int t = 0; t < ntiles; ++t) {
        mbar_wait(&empty[stage], phase ^ 1);
        mbar_arrive_expect_tx(&full[stage], 2 * TILE_BYTES);
        const int row = (int)((long long)b * S + k0 + (long long)t * TK);
        tma_load_3d(smem + stage * 2 * TILE_BYTES, &tm, &full[stage], 0, h, row);
        tma_load_3d(smem + stage * 2 * TILE_BYTES + TILE_BYTES, &tm, &full[stage], 0, H + h, row);
        if (++stage == AST) { stage = 0; phase ^= 1; }
      }
    }
  } else {
    const int key = lane & 15, half = lane >> 4;
    int stage = 0; uint32_t phase = 0;
    for (int t = 0; t < ntiles; ++t) {
      mbar_wait(&full[stage], phase);
      const uint8_t* Ks = smem + stage * 2 * TILE_BYTES;
      const uint8_t* Vs = Ks + TILE_BYTES;
      const long long jg = k0 + (long long)t * TK + warp * 16 + key;
      float sd = 0.f;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const int cc = (c + lane) & 7;                                 // rotated: a quarter-warp covers all 32 banks
        const uint4 kv = *reinterpret_cast<const uint4*>(Ks + (warp * 16 + key) * (HD * 2) + half * 128 + cc * 16);
        const uint4 qv = *reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(qb) + half * 128 + cc * 16);
        const uint32_t* kw = reinterpret_cast<const uint32_t*>(&kv);
        const uint32_t* qw = reinterpret_cast<const uint32_t*>(&qv);
#pragma unroll
        for (int e = 0; e < 4; ++e) { sd = fmaf(bf_lo(qw[e]), bf_lo(kw[e]), sd); sd = fmaf(bf_hi(qw[e]), bf_hi(kw[e]), sd); }
      }
      sd += __shfl_xor_sync(0xffffffffu, sd, 16);
      sd = jg < k1 ? sd * scale : -INFINITY;
      float mx = sd;
#pragma unroll
      for (int x = 8; x > 0; x >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, x));
      const float mn = fmaxf(m, mx);
      if (mn != -INFINITY) {                                           // warp-uniform
        const float alpha = __expf(m - mn), pe = __expf(sd - mn);
        l = l * alpha + (half == 0 ? pe : 0.f);
        const float pb = rbf(pe);                                      // P rounded to bf16 before the PV product, like the prefill kernel
        o0 *= alpha; o1 *= alpha; o2 *= alpha; o3 *= alpha;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float pj = __shfl_sync(0xffffffffu, pb, j);
          if (pj != 0.f) {                                             // masked keys (and underflowed ones) contribute nothing; garbage rows never reach the FMA
            const uint2 vv = *reinterpret_cast<const uint2*>(Vs + (warp * 16 + j) * (HD * 2) + lane * 8);
            o0 = fmaf(pj, bf_lo(vv.x), o0); o1 = fmaf(pj, bf_hi(vv.x), o1);
            o2 = fmaf(pj, bf_lo(vv.y), o2); o3 = fmaf(pj, bf_hi(vv.y), o3);
          }
        }
        m = mn;
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[stage]);
      if (++stage == AST) { stage = 0; phase ^= 1; }
    }
#pragma unroll
    for (int x = 16; x > 0; x >>= 1) l += __shfl_xor_sync(0xffffffffu, l, x);
  }
  __syncthreads();                                                      // every tile consumed: stage 0 is free for the merge
  float* red_o = reinterpret_cast<float*>(smem);                       // [4][128]
  if (warp < 4) {
    if (lane == 0) { red[warp * 2] = m; red[warp * 2 + 1] = l; }
    *reinterpret_cast<float4*>(red_o + warp * HD + lane * 4) = make_float4(o0, o1, o2, o3);
  }
  __syncthreads();
  if (tid < HD) {
    float M = -INFINITY;
#pragma unroll
    for (int w = 0; w < 4; ++w) M = fmaxf(M, red[w * 2]);
    float acc = 0.f, L = 0.f;
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      const float sc = red[w * 2] == -INFINITY ? 0.f : __expf(red[w * 2] - M);
      acc += red_o[w * HD + tid] * sc;
      L += red[w * 2 + 1] * sc;
    }
    const long long pidx = ((long long)b * H + h) * nsplit + sp;
    part_o[pidx * HD + tid] = acc;
    if (tid == 0) { part_ml[pidx * 2] = M; part_ml[pidx * 2 + 1] = L; }
  }
}

__global__ void decode_attn_merge_kernel(const float* __restrict__ part_o, const float* __restrict__ part_ml, bf16* __restrict__ out,
                                         int H, int nsplit) {
  pdl_launch_dependents(); pdl_wait();
  const int h = blockIdx.x, b = blockIdx.y, d = threadIdx.x;
  const long long base = ((long long)b * H + h) * nsplit;
  float M = -INFINITY;
  for (int s = 0; s < nsplit; ++s) M = fmaxf(M, part_ml[(base + s) * 2]);
  float L = 0.f, acc = 0.f;
  for (int s = 0; s < nsplit; ++s) {
    const float ms = part_ml[(base + s) * 2];
    const float w = (ms == -INFINITY) ? 0.f : __expf(ms - M);
    L += part_ml[(base + s) * 2 + 1] * w;
    acc += part_o[(base + s) * HD + d] * w;
  }
  out[((long long)b * H + h) * HD + d] = __float2bfloat16_rn(acc / L);
}

__global__ void add_i64_kernel(long long* p, long long v) { *p += v; }

}  // namespace

extern "C" int evo_gelu_gate_interleaved(const void* t, void* out, int64_t M, int ipad, void* stream) {
  EVO_REQUIRE(ipad % 128 == 0, "evo_gelu_gate_interleaved: ipad must be a multiple of 128");
  long long total = M * (ipad / 2);
  if (total == 0) return 0;
  gelu_gate_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>((const bf16*)t, (bf16*)out, M, ipad);
  return check_launch("evo_gelu_gate_interleaved");
}

template <bool ROWS>
static int decode_qkv_prep(const char* name, void* qkv, void* cache, const void* cos, const void* sin, const int64_t* pos,
                           int B, int H, int hd, int64_t max_seqlen, void* stream) {
  EVO_REQUIRE(hd == HD, "%s: head_dim %d unsupported", name, hd);
  int n = B * H * 64;
  EVO_CUDA(launch_pdl(decode_qkv_prep_kernel<ROWS>, dim3((n + 127) / 128), dim3(128), 0, (cudaStream_t)stream, (bf16*)qkv, (bf16*)cache, (const bf16*)cos, (const bf16*)sin,
                      (const long long*)pos, B, H, max_seqlen));
  return check_launch(name);
}

extern "C" int evo_decode_qkv_prep(void* qkv, void* cache, const void* cos, const void* sin, const int64_t* pos,
                                   int B, int H, int hd, int64_t max_seqlen, void* stream) {
  return decode_qkv_prep<false>("evo_decode_qkv_prep", qkv, cache, cos, sin, pos, B, H, hd, max_seqlen, stream);
}

extern "C" int evo_decode_qkv_prep_rows(void* qkv, void* cache, const void* cos, const void* sin, const int64_t* pos,
                                        int B, int H, int hd, int64_t max_seqlen, void* stream) {
  return decode_qkv_prep<true>("evo_decode_qkv_prep_rows", qkv, cache, cos, sin, pos, B, H, hd, max_seqlen, stream);
}

extern "C" size_t evo_decode_attn_workspace(int B, int H, int nsplit) { return (size_t)B * H * nsplit * (HD + 2) * sizeof(float); }

template <bool ROWS>
static int decode_attn(const char* name, const void* qkv, const void* cache, void* out, const int64_t* pos, int B, int H, int hd,
                       int64_t max_seqlen, int nsplit, float softmax_scale, void* workspace, size_t workspace_bytes, void* stream) {
  EVO_REQUIRE(hd == HD, "%s: head_dim %d unsupported", name, hd);
  EVO_REQUIRE(nsplit >= 1 && nsplit <= 64, "%s: bad nsplit %d", name, nsplit);
  EVO_REQUIRE(workspace && workspace_bytes >= evo_decode_attn_workspace(B, H, nsplit), "%s: workspace too small", name);
  float* part_o = (float*)workspace;
  float* part_ml = part_o + (size_t)B * H * nsplit * HD;
  static const bool force_v1 = getenv("EVO_B200_DECODE_ATTN_V1") != nullptr;
  if (max_seqlen % TK == 0 && !force_v1 && (long long)B * max_seqlen < (1LL << 31)) {
    CUtensorMap tm;
    const uint64_t dims[3] = {(uint64_t)HD, (uint64_t)(2 * H), (uint64_t)B * (uint64_t)max_seqlen};
    const uint64_t str[2] = {(uint64_t)HD * 2, (uint64_t)2 * H * HD * 2};
    const uint32_t box[3] = {(uint32_t)HD, 1, (uint32_t)TK};
    int rc = make_tmap_nd_bf16(&tm, cache, 3, dims, str, box, false);
    if (rc) return rc;
    static unsigned long long attr_done = 0;
    if ((rc = ensure_dyn_smem(decode_attn_tma_kernel<ROWS>, ATT2_SMEM, attr_done))) return rc;
    EVO_CUDA(launch_pdl(decode_attn_tma_kernel<ROWS>, dim3(H, B, nsplit), dim3(160), (size_t)ATT2_SMEM, (cudaStream_t)stream, tm, (const bf16*)qkv, part_o, part_ml,
                        (const long long*)pos, H, (long long)max_seqlen, nsplit, softmax_scale));
    rc = check_launch(name);
    if (rc) return rc;
    EVO_CUDA(launch_pdl(decode_attn_merge_kernel, dim3(H, B), dim3(HD), 0, (cudaStream_t)stream, (const float*)part_o, (const float*)part_ml, (bf16*)out, H, nsplit));
    return check_launch("evo_decode_attn_merge");
  }
  EVO_CUDA(launch_pdl(decode_attn_kernel<ROWS>, dim3(H, B, nsplit), dim3(DT), 0, (cudaStream_t)stream, (const bf16*)qkv, (const bf16*)cache, part_o, part_ml,
                      (const long long*)pos, H, max_seqlen, nsplit, softmax_scale));
  int rc = check_launch(name);
  if (rc) return rc;
  EVO_CUDA(launch_pdl(decode_attn_merge_kernel, dim3(H, B), dim3(HD), 0, (cudaStream_t)stream, (const float*)part_o, (const float*)part_ml, (bf16*)out, H, nsplit));
  return check_launch("evo_decode_attn_merge");
}

extern "C" int evo_decode_attn(const void* qkv, const void* cache, void* out, const int64_t* pos, int B, int H, int hd,
                               int64_t max_seqlen, int nsplit, float softmax_scale, void* workspace, size_t workspace_bytes, void* stream) {
  return decode_attn<false>("evo_decode_attn", qkv, cache, out, pos, B, H, hd, max_seqlen, nsplit, softmax_scale, workspace, workspace_bytes, stream);
}

extern "C" int evo_decode_attn_rows(const void* qkv, const void* cache, void* out, const int64_t* pos, int B, int H, int hd,
                                    int64_t max_seqlen, int nsplit, float softmax_scale, void* workspace, size_t workspace_bytes, void* stream) {
  return decode_attn<true>("evo_decode_attn_rows", qkv, cache, out, pos, B, H, hd, max_seqlen, nsplit, softmax_scale, workspace, workspace_bytes, stream);
}

extern "C" int evo_advance_position(int64_t* pos, int64_t delta, void* stream) {
  add_i64_kernel<<<1, 1, 0, (cudaStream_t)stream>>>((long long*)pos, delta);
  return check_launch("evo_advance_position");
}
