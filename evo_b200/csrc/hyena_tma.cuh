// Hyena scan, TMA-staged variant (the production path for head_dim 128 / D % 256 == 0).
//
// Same operator and rounding points as hyena_scan_kernel (hyena.cu); what changes is how the
// machine is driven:
//   * a CTA owns two heads (256 channels) of one batch row and walks its L segment in tiles of
//     T2 tokens; warp 4 is a TMA producer that keeps a 4-deep mbarrier ring of z tiles
//     ([x2|x1|v] x 2 heads = six 128-column boxes, 24 KB per stage) in flight, so HBM latency is
//     never exposed to the scan;
//   * each of the 128 compute threads carries TWO adjacent channels and does all fp32 work with
//     packed fma.rn.f32x2 (FFMA2): Blackwell's FP32 pipe only reaches its 128 lanes/SM/clk
//     through the packed form, and it halves the instruction count of the 8-state recurrence;
//   * x2/x1/v are read from smem as bf16x2 words (conflict-free: lane l reads word l), y is
//     written as bf16x2 words, 128 B per warp per token.
#pragma once
#include "common.cuh"

namespace evo_hy2 {

using namespace evo;

constexpr int NS = 8;
constexpr int T2 = 16;                       // tokens per stage
constexpr int STAGES = 8;                    // maximum ring depth; the launch picks 4 (two CTAs per SM) or 8 (one)
constexpr int CH_PER_CTA = 256;              // two heads of 128
constexpr int SUB_BYTES = T2 * 128 * 2;      // one 128-column box
constexpr int STAGE_BYTES = 6 * SUB_BYTES;   // [head0: x2 x1 v][head1: x2 x1 v]
constexpr int THREADS = 160;                 // 4 compute warps + 1 producer warp
constexpr int smem_bytes(int nst) { return nst * STAGE_BYTES + 128 + 1024; }

struct Args2 {
  bf16* y;
  const bf16* z;
  const bf16* fir_w; const bf16* fir_b; const bf16* Dskip;
  const float* poles; const float* residues;
  const bf16* halo; const float* state_in;
  float* state_out;
  float* seg_states;
  int B, D, nseg, nst;
  long long L, seg_len;
  const int* lengths;          // (B) valid tokens per row (evo_hyena_fwd_ragged); NULL = every row has L
};

__device__ __forceinline__ float2 unpack2(uint32_t v) { return make_float2(bf_lo(v), bf_hi(v)); }
__device__ __forceinline__ float2 rbf2(float2 a) { return unpack2(pack_bf16(a.x, a.y)); }
__device__ __forceinline__ uint32_t lds32(uint32_t addr) { uint32_t v; asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr)); return v; }
__device__ __forceinline__ float2 ld_bf2(const bf16* p) { return unpack2(__ldg(reinterpret_cast<const unsigned int*>(p))); }

struct C2 { float2 r, i; };                  // two complex numbers (one per channel of the pair)
__device__ __forceinline__ C2 cmul2(C2 a, C2 b) {
  C2 o;
  o.r = __ffma2_rn(a.r, b.r, __fmul2_rn(make_float2(-a.i.x, -a.i.y), b.i));
  o.i = __ffma2_rn(a.r, b.i, __fmul2_rn(a.i, b.r));
  return o;
}
__device__ __forceinline__ C2 cpow2(C2 p, long long n) {
  C2 acc; acc.r = make_float2(1.f, 1.f); acc.i = make_float2(0.f, 0.f);
  while (n > 0) { if (n & 1) acc = cmul2(acc, p); p = cmul2(p, p); n >>= 1; }
  return acc;
}

template <bool STATE_ONLY>
__global__ void __launch_bounds__(THREADS, 1)
hyena_scan_tma_kernel(const __grid_constant__ CUtensorMap tmZ, const Args2 a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~(uintptr_t)127);
  const int NST = a.nst;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + NST * STAGE_BYTES);
  uint64_t* empty = full + STAGES;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cb = blockIdx.x, b = blockIdx.y, seg = blockIdx.z;
  const long long t0 = (long long)seg * a.seg_len;
  const long long t1 = min(a.L, t0 + a.seg_len);
  const int n_tiles = t1 > t0 ? (int)((t1 - t0 + T2 - 1) / T2) : 0;

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 4); }
    fence_barrier_init();
  }
  __syncthreads();

  if (warp == 4) {
    // ------------------------------------------------ TMA producer
    if (lane == 0) {
      tma_prefetch_desc(&tmZ);
      for (int k = 0; k < n_tiles; ++k) {
        const int st = k % NST;
        mbar_wait(&empty[st], ((uint32_t)(k / NST) & 1) ^ 1);
        uint8_t* dst = smem + st * STAGE_BYTES;
        const int row = (int)(t0 + (long long)k * T2);
        if (STATE_ONLY) {
          mbar_arrive_expect_tx(&full[st], 4 * SUB_BYTES);
#pragma unroll
          for (int hh = 0; hh < 2; ++hh)
#pragma unroll
            for (int w = 1; w < 3; ++w)
              tma_load_3d(dst + (hh * 3 + w) * SUB_BYTES, &tmZ, &full[st], cb * 768 + hh * 384 + w * 128, row, b);
        } else {
          mbar_arrive_expect_tx(&full[st], STAGE_BYTES);
#pragma unroll
          for (int s6 = 0; s6 < 6; ++s6)
            tma_load_3d(dst + s6 * SUB_BYTES, &tmZ, &full[st], cb * 768 + s6 * 128, row, b);
        }
      }
    }
    return;
  }

  // ------------------------------------------------ compute warps: thread = channel pair
  const int hh = warp >> 1;                               // head within the CTA
  const int j2 = ((warp & 1) * 32 + lane) * 2;            // first channel of the pair inside the head
  const int ch = cb * CH_PER_CTA + hh * 128 + j2;         // global channel (of D)
  const int zc = cb * 768 + hh * 384 + j2;                // z column of x2; x1 = +128, v = +256
  const long long C3 = 3LL * a.D;

  float2 pr[NS], pi[NS], npi[NS], rr[NS], ri[NS], sr[NS], si[NS];
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    float2 p0 = __ldg(reinterpret_cast<const float2*>(a.poles) + (long long)ch * NS + s);
    float2 p1 = __ldg(reinterpret_cast<const float2*>(a.poles) + (long long)(ch + 1) * NS + s);
    float2 r0 = __ldg(reinterpret_cast<const float2*>(a.residues) + (long long)ch * NS + s);
    float2 r1 = __ldg(reinterpret_cast<const float2*>(a.residues) + (long long)(ch + 1) * NS + s);
    pr[s] = make_float2(p0.x, p1.x); pi[s] = make_float2(p0.y, p1.y); npi[s] = make_float2(-p0.y, -p1.y);
    rr[s] = make_float2(r0.x, r1.x); ri[s] = make_float2(-r0.y, -r1.y);
    sr[s] = make_float2(0.f, 0.f); si[s] = make_float2(0.f, 0.f);
  }
  // FIR taps / bias / skip for the pair: w[k] = (tap k of channel c, tap k of channel c+1)
  float2 w1[3], wv[3], w2[3], b1, bv, b2, dsk;
  {
    auto taps = [&](int c, float2 (&w)[3]) {
      const bf16* p0 = a.fir_w + (long long)c * 3;
#pragma unroll
      for (int k = 0; k < 3; ++k) w[k] = make_float2(__bfloat162float(p0[k]), __bfloat162float(p0[3 + k]));
    };
    taps(zc + 128, w1); taps(zc + 256, wv); taps(zc, w2);
    b1 = ld_bf2(a.fir_b + zc + 128); bv = ld_bf2(a.fir_b + zc + 256); b2 = ld_bf2(a.fir_b + zc);
    dsk = ld_bf2(a.Dskip + ch);
  }

  if (!STATE_ONLY) {
    if (a.state_in) {
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        float2 v0 = __ldg(reinterpret_cast<const float2*>(a.state_in) + ((long long)b * a.D + ch) * NS + s);
        float2 v1 = __ldg(reinterpret_cast<const float2*>(a.state_in) + ((long long)b * a.D + ch + 1) * NS + s);
        sr[s] = make_float2(v0.x, v1.x); si[s] = make_float2(v0.y, v1.y);
      }
    }
    if (seg > 0) {
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        C2 p; p.r = pr[s]; p.i = pi[s];
        const C2 pl = cpow2(p, a.seg_len);
        C2 acc; acc.r = sr[s]; acc.i = si[s];
        for (int q = 0; q < seg; ++q) {
          const float2* e = reinterpret_cast<const float2*>(a.seg_states) + (((long long)b * a.nseg + q) * a.D + ch) * NS + s;
          float2 e0 = e[0], e1 = e[NS];
          acc = cmul2(pl, acc);
          acc.r = __fadd2_rn(acc.r, make_float2(e0.x, e1.x));
          acc.i = __fadd2_rn(acc.i, make_float2(e0.y, e1.y));
        }
        sr[s] = acc.r; si[s] = acc.i;
      }
    }
  }

  // FIR history z[t0-2], z[t0-1]
  const bf16* zb = a.z + (long long)b * a.L * C3;
  float2 h1[2], hv[2], h2[2];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    h1[k] = hv[k] = h2[k] = make_float2(0.f, 0.f);
    long long t = t0 - 2 + k;
    const bf16* row = nullptr;
    if (t >= 0) row = zb + t * C3;
    else if (a.halo) row = a.halo + ((long long)b * 2 + (t + 2)) * C3;
    if (row) { h1[k] = ld_bf2(row + zc + 128); hv[k] = ld_bf2(row + zc + 256); if (!STATE_ONLY) h2[k] = ld_bf2(row + zc); }
  }

  uint32_t* yrow = STATE_ONLY ? nullptr : reinterpret_cast<uint32_t*>(a.y + ((long long)b * a.L + t0) * a.D + ch);
  const long long ystride = a.D / 2;        // in 32-bit words

  // One group = G tokens.  The element-wise stages (FIR + roundings, output gating) have no
  // cross-token dependence, so they are written as straight-line code over the group: a single
  // in-order warp per SM sub-partition needs that ILP (there is no second warp to switch to).
  // Only the 8-state recurrence in the middle is sequential in t.
  constexpr int G = 8;
  auto do_group = [&](uint32_t tile, int j0, int n_valid, uint32_t* ydst) {
    uint32_t xq[G], f2q[G], ycq[G];
    // ---- stage A: short FIR (fp32 accumulate, rp) + bias (rp); x = x1*v (rp)
    float2 zin1[G], zinv[G], zin2[G];
#pragma unroll
    for (int g = 0; g < G; ++g) {
      zin1[g] = unpack2(lds32(tile + 1 * SUB_BYTES + (j0 + g) * 256));
      zinv[g] = unpack2(lds32(tile + 2 * SUB_BYTES + (j0 + g) * 256));
      if (!STATE_ONLY) zin2[g] = unpack2(lds32(tile + (j0 + g) * 256));
    }
#pragma unroll
    for (int g = 0; g < G; ++g) {
      const float2 a1 = g >= 2 ? zin1[g - 2] : h1[g], b1_ = g >= 1 ? zin1[g - 1] : h1[1];
      const float2 av = g >= 2 ? zinv[g - 2] : hv[g], bv_ = g >= 1 ? zinv[g - 1] : hv[1];
      const float2 f1 = rbf2(__fadd2_rn(rbf2(__ffma2_rn(w1[2], zin1[g], __ffma2_rn(w1[1], b1_, __fmul2_rn(w1[0], a1)))), b1));
      const float2 fv = rbf2(__fadd2_rn(rbf2(__ffma2_rn(wv[2], zinv[g], __ffma2_rn(wv[1], bv_, __fmul2_rn(wv[0], av)))), bv));
      const float2 xx = __fmul2_rn(f1, fv);
      xq[g] = pack_bf16(xx.x, xx.y);
      if (!STATE_ONLY) {
        const float2 a2 = g >= 2 ? zin2[g - 2] : h2[g], b2_ = g >= 1 ? zin2[g - 1] : h2[1];
        const float2 f2 = __fadd2_rn(rbf2(__ffma2_rn(w2[2], zin2[g], __ffma2_rn(w2[1], b2_, __fmul2_rn(w2[0], a2)))), b2);
        f2q[g] = pack_bf16(f2.x, f2.y);
      }
    }
    // FIR history for the next group = last two valid inputs of this one
    if (n_valid == G) {
      h1[0] = zin1[G - 2]; h1[1] = zin1[G - 1]; hv[0] = zinv[G - 2]; hv[1] = zinv[G - 1];
      if (!STATE_ONLY) { h2[0] = zin2[G - 2]; h2[1] = zin2[G - 1]; }
    }
    // ---- stage B: modal recurrence, sequential in t, 16 independent complex-pair chains per step
#pragma unroll
    for (int g = 0; g < G; ++g) {
      if (g < n_valid) {
        const float2 x = unpack2(xq[g]);
        // four short accumulation chains instead of two 8-long ones (FFMA2 latency is exposed: one warp per SMSP)
        float2 ar0 = make_float2(0.f, 0.f), ar1 = ar0, ai0 = ar0, ai1 = ar0;
#pragma unroll
        for (int s = 0; s < NS; ++s) {
          const float2 t_ = __ffma2_rn(npi[s], si[s], x);
          const float2 nr = __ffma2_rn(pr[s], sr[s], t_);
          const float2 ni = __ffma2_rn(pr[s], si[s], __fmul2_rn(pi[s], sr[s]));
          sr[s] = nr; si[s] = ni;
          if (!STATE_ONLY) {
            if (s & 1) { ar1 = __ffma2_rn(rr[s], nr, ar1); ai1 = __ffma2_rn(ri[s], ni, ai1); }
            else       { ar0 = __ffma2_rn(rr[s], nr, ar0); ai0 = __ffma2_rn(ri[s], ni, ai0); }
          }
        }
        if (!STATE_ONLY) { const float2 c = __fadd2_rn(__fadd2_rn(ar0, ar1), __fadd2_rn(ai0, ai1)); ycq[g] = pack_bf16(c.x, c.y); }   // y.to(bf16) (rp)
      }
    }
    // ---- stage C: y = (conv + x1v*D) * x2 with the reference's roundings, bf16x2 stores
    if (!STATE_ONLY) {
#pragma unroll
      for (int g = 0; g < G; ++g) {
        if (g < n_valid) {
          const float2 x = unpack2(xq[g]);
          const float2 u = rbf2(__fadd2_rn(unpack2(ycq[g]), rbf2(__fmul2_rn(x, dsk))));
          const float2 o = __fmul2_rn(u, unpack2(f2q[g]));
          ydst[(long long)g * ystride] = pack_bf16(o.x, o.y);
        }
      }
    }
  };

  for (int k = 0; k < n_tiles; ++k) {
    const int st = k % NST;
    mbar_wait(&full[st], (uint32_t)(k / NST) & 1);
    const uint32_t tile = smem_u32(smem) + st * STAGE_BYTES + hh * 3 * SUB_BYTES + j2 * 2;
    const int n_tok = (int)min((long long)T2, t1 - (t0 + (long long)k * T2));
    uint32_t* ytile = STATE_ONLY ? nullptr : yrow + (long long)k * T2 * ystride;
    if (n_tok == T2) {
#pragma unroll
      for (int j0 = 0; j0 < T2; j0 += G) do_group(tile, j0, G, STATE_ONLY ? nullptr : ytile + (long long)j0 * ystride);
    } else {                                   // ragged last tile of the segment
      for (int j0 = 0; j0 < n_tok; j0 += G) do_group(tile, j0, min(G, n_tok - j0), STATE_ONLY ? nullptr : ytile + (long long)j0 * ystride);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[st]);
  }

  float* dst = nullptr;
  if (STATE_ONLY) dst = a.seg_states + ((((long long)b * a.nseg + seg) * a.D + ch) * NS) * 2;
  else if (a.state_out && seg == a.nseg - 1) dst = a.state_out + (((long long)b * a.D + ch) * NS) * 2;
  if (dst && n_tiles >= 0) {
    float2* e = reinterpret_cast<float2*>(dst);
#pragma unroll
    for (int s = 0; s < NS; ++s) { e[s] = make_float2(sr[s].x, si[s].x); e[NS + s] = make_float2(sr[s].y, si[s].y); }
  }
}

}  // namespace evo_hy2
