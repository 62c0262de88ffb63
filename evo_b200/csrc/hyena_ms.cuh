// Hyena scan, mode-split variant (round 2): the production path for head_dim 128 / D % 256 == 0.
//
// Same operator, same rounding points and the same TMA ring as hyena_scan_tma_kernel (hyena_tma.cuh); what changes
// is the work assignment, because that kernel was latency-starved, not bandwidth- or pipe-bound: 128 CTAs x 4
// compute warps = ONE warp per SM sub-partition, 214 registers per thread, fma pipe 55 % busy, issue slots 47 %
// (profiles/r01_ncu_full_hyena_call5.csv).  Here
//   * a thread still carries a channel PAIR (so every fp32 op stays a packed FFMA2 -- the only way to the FP32
//     pipe's 128 lanes/SM/clk), but only FOUR of the eight modal states: lanes l and l^16 of a warp share a pair.
//     Registers per thread drop to ~half and a 256-channel CTA has 8 compute warps = two per sub-partition, so a
//     dependent FFMA2 chain in one warp is covered by the other;
//   * the element-wise work is split between the two halves instead of duplicated: half 0 runs the x1 FIR, half 1
//     the v FIR (one shuffle exchanges the bf16x2 results); half 0 gates tokens 0..3 of a group of eight, half 1
//     tokens 4..7 (one shuffle per fp32 word moves the partial residue sums to the half that needs them);
//   * every bf16 (x) bf16 -> bf16 tensor op of the reference (bias add, x1*v, D*x1v, +conv, *x2) is ONE packed
//     add.rn.bf16x2 / mul.rn.bf16x2 instead of unpack + fp32 op + pack: the product of two bf16 is exact in fp32 and
//     the sum of two bf16 is exact in fp32 or rounds to the larger operand either way, so a single rounding of the
//     exact result is bit-identical to the reference's "compute in fp32, round to bf16".
// fma-pipe instructions per token per channel pair: 68 (was 67); ALU conversions ~21 (was ~38).
#pragma once
#include "hyena_tma.cuh"

namespace evo_hy3 {

using namespace evo;
using evo_hy2::Args2;
using evo_hy2::C2;
using evo_hy2::cmul2;
using evo_hy2::cpow2;
using evo_hy2::lds32;
using evo_hy2::unpack2;

constexpr int NS = 8;
constexpr int NSH = 4;                       // modal states per thread
constexpr int T2 = evo_hy2::T2;              // tokens per stage
constexpr int STAGES = evo_hy2::STAGES;
constexpr int CH_PER_CTA = 256;
constexpr int SUB_BYTES = evo_hy2::SUB_BYTES;
constexpr int STAGE_BYTES = evo_hy2::STAGE_BYTES;
constexpr int CWARPS = 8;                    // compute warps: 4 per head, 16 channel pairs x 2 halves each
constexpr int THREADS = (CWARPS + 1) * 32;   // + 1 TMA producer warp
constexpr int G = 8;                         // tokens per group
constexpr int smem_bytes(int nst) { return evo_hy2::smem_bytes(nst); }

__device__ __forceinline__ uint32_t mul_bf2(uint32_t a, uint32_t b) { uint32_t d; asm("mul.rn.bf16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b)); return d; }
__device__ __forceinline__ uint32_t add_bf2(uint32_t a, uint32_t b) { uint32_t d; asm("add.rn.bf16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b)); return d; }
__device__ __forceinline__ uint32_t ldg32(const bf16* p) { return __ldg(reinterpret_cast<const unsigned int*>(p)); }

// RAGGED: row b holds a.lengths[b] valid tokens (right-padded to L): the scan of each segment stops at the row's length, a
// segment wholly past it is empty, and the state after the row's last token is written by the segment that holds that token.
// Every segment before that one is full, so the in-kernel carry fold needs no per-row length.  With every length == L the
// RAGGED instantiation computes exactly what the uniform one does.
template <bool STATE_ONLY, bool RAGGED = false>
__global__ void __launch_bounds__(THREADS, 1)
hyena_scan_ms_kernel(const __grid_constant__ CUtensorMap tmZ, const Args2 a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~(uintptr_t)127);
  const int NST = a.nst;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + NST * STAGE_BYTES);
  uint64_t* empty = full + STAGES;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cb = blockIdx.x, b = blockIdx.y, seg = blockIdx.z;
  const long long Lb = RAGGED ? min(a.L, (long long)max(a.lengths[b], 0)) : a.L;
  const int last_seg = RAGGED ? (Lb > 0 ? (int)((Lb - 1) / a.seg_len) : 0) : a.nseg - 1;
  const long long t0 = (long long)seg * a.seg_len;
  const long long t1 = min(Lb, t0 + a.seg_len);
  const int n_tiles = t1 > t0 ? (int)((t1 - t0 + T2 - 1) / T2) : 0;
  if (RAGGED && n_tiles == 0 && (STATE_ONLY || seg != last_seg)) {
    // nothing of this row here; the state pass still leaves a zero end state for the fold
    if (STATE_ONLY && threadIdx.x < 256)
      for (int i = threadIdx.x; i < CH_PER_CTA * NS * 2; i += 256) a.seg_states[(((long long)b * a.nseg + seg) * a.D + cb * CH_PER_CTA) * NS * 2 + i] = 0.f;
    return;
  }

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], CWARPS); }
    fence_barrier_init();
  }
  __syncthreads();

  if (warp == CWARPS) {
    // ------------------------------------------------ TMA producer (one lane)
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

  // ------------------------------------------------ compute warps: thread = (channel pair, half of the modes)
  const int hh = warp >> 2;                               // head within the CTA
  const int half = lane >> 4;                             // 0: modes 0..3, x1 FIR, tokens 0..3 | 1: modes 4..7, v FIR, tokens 4..7
  const int j2 = ((warp & 3) * 16 + (lane & 15)) * 2;     // first channel of the pair inside the head
  const int ch = cb * CH_PER_CTA + hh * 128 + j2;         // global channel (of D)
  const int zc = cb * 768 + hh * 384 + j2;                // z column of x2; x1 = +128, v = +256
  const int own = 1 + half;                               // sub-box this thread's FIR reads: 1 = x1, 2 = v
  const int m0 = half * NSH;
  const long long C3 = 3LL * a.D;

  float2 pr[NSH], pi[NSH], npi[NSH], rr[NSH], ri[NSH], sr[NSH], si[NSH];
#pragma unroll
  for (int s = 0; s < NSH; ++s) {
    const float2 p0 = __ldg(reinterpret_cast<const float2*>(a.poles) + (long long)ch * NS + m0 + s);
    const float2 p1 = __ldg(reinterpret_cast<const float2*>(a.poles) + (long long)(ch + 1) * NS + m0 + s);
    const float2 r0 = __ldg(reinterpret_cast<const float2*>(a.residues) + (long long)ch * NS + m0 + s);
    const float2 r1 = __ldg(reinterpret_cast<const float2*>(a.residues) + (long long)(ch + 1) * NS + m0 + s);
    pr[s] = make_float2(p0.x, p1.x); pi[s] = make_float2(p0.y, p1.y); npi[s] = make_float2(-p0.y, -p1.y);
    rr[s] = make_float2(r0.x, r1.x); ri[s] = make_float2(-r0.y, -r1.y);      // Re(R s) = Rr sr - Ri si
    sr[s] = make_float2(0.f, 0.f); si[s] = make_float2(0.f, 0.f);
  }
  // FIR taps of the owned channel pair and of x2; biases / skip stay packed bf16x2
  float2 wo[3], w2[3];
  {
    const bf16* p0 = a.fir_w + (long long)(zc + own * 128) * 3;
    const bf16* q0 = a.fir_w + (long long)zc * 3;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      wo[k] = make_float2(__bfloat162float(p0[k]), __bfloat162float(p0[3 + k]));
      w2[k] = make_float2(__bfloat162float(q0[k]), __bfloat162float(q0[3 + k]));
    }
  }
  const uint32_t boq = ldg32(a.fir_b + zc + own * 128);
  const uint32_t b2q = ldg32(a.fir_b + zc);
  const uint32_t dskq = ldg32(a.Dskip + ch);

  if (!STATE_ONLY) {
    if (a.state_in) {
#pragma unroll
      for (int s = 0; s < NSH; ++s) {
        const float2 v0 = __ldg(reinterpret_cast<const float2*>(a.state_in) + ((long long)b * a.D + ch) * NS + m0 + s);
        const float2 v1 = __ldg(reinterpret_cast<const float2*>(a.state_in) + ((long long)b * a.D + ch + 1) * NS + m0 + s);
        sr[s] = make_float2(v0.x, v1.x); si[s] = make_float2(v0.y, v1.y);
      }
    }
    if (seg > 0) {      // carry entering this segment: S_j = p^len S_{j-1} + E_{j-1} over the zero-start end states
#pragma unroll
      for (int s = 0; s < NSH; ++s) {
        C2 p; p.r = pr[s]; p.i = pi[s];
        const C2 pl = cpow2(p, a.seg_len);
        C2 acc; acc.r = sr[s]; acc.i = si[s];
        for (int q = 0; q < seg; ++q) {
          const float2* e = reinterpret_cast<const float2*>(a.seg_states) + (((long long)b * a.nseg + q) * a.D + ch) * NS + m0 + s;
          const float2 e0 = e[0], e1 = e[NS];
          acc = cmul2(pl, acc);
          acc.r = __fadd2_rn(acc.r, make_float2(e0.x, e1.x));
          acc.i = __fadd2_rn(acc.i, make_float2(e0.y, e1.y));
        }
        sr[s] = acc.r; si[s] = acc.i;
      }
    }
  }

  // FIR history z[t0-2], z[t0-1]: fp32 pair for the owned channel, packed words for x2 (half 0 only uses them)
  const bf16* zb = a.z + (long long)b * a.L * C3;
  float2 ho[2];
  uint32_t h2q[2];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    ho[k] = make_float2(0.f, 0.f); h2q[k] = 0u;
    const long long t = t0 - 2 + k;
    const bf16* row = nullptr;
    if (t >= 0) row = zb + t * C3;
    else if (a.halo) row = a.halo + ((long long)b * 2 + (t + 2)) * C3;
    if (row) { ho[k] = unpack2(ldg32(row + zc + own * 128)); if (!STATE_ONLY) h2q[k] = ldg32(row + zc); }
  }

  const long long ystride = a.D / 2;        // in 32-bit words
  uint32_t* yrow = STATE_ONLY ? nullptr : reinterpret_cast<uint32_t*>(a.y + ((long long)b * a.L + t0) * a.D + ch) + (long long)(4 * half) * ystride;

  auto do_group = [&](uint32_t tile, int j0, int n_valid, uint32_t* ydst) {
    // ---- stage A: the owned short FIR (fp32 accumulate, rp) + bias (rp) for all G tokens
    float2 zo[G];
#pragma unroll
    for (int g = 0; g < G; ++g) zo[g] = unpack2(lds32(tile + own * SUB_BYTES + (j0 + g) * 256));
    uint32_t xq[G];
#pragma unroll
    for (int g = 0; g < G; ++g) {
      const float2 a_ = g >= 2 ? zo[g - 2] : ho[g], b_ = g >= 1 ? zo[g - 1] : ho[1];
      const float2 acc = __ffma2_rn(wo[2], zo[g], __ffma2_rn(wo[1], b_, __fmul2_rn(wo[0], a_)));
      const uint32_t f = add_bf2(pack_bf16(acc.x, acc.y), boq);
      xq[g] = mul_bf2(f, __shfl_xor_sync(0xffffffffu, f, 16));          // x1v = x1 * v (rp): the partner holds the other factor
    }
    if (n_valid == G) { ho[0] = zo[G - 2]; ho[1] = zo[G - 1]; }
    // ---- stage A2: x2 FIR for the four tokens this half gates (window = 6 consecutive z2 rows)
    uint32_t f2q[4];
    if (!STATE_ONLY) {
      uint32_t l2[6];
#pragma unroll
      for (int i = 0; i < 4; ++i) l2[i] = lds32(tile + half * 512 + (j0 + i) * 256);      // tokens i (half 0) / i + 2 (half 1)
      l2[4] = lds32(tile + (j0 + 6) * 256); l2[5] = lds32(tile + (j0 + 7) * 256);
      float2 wf[6];
      wf[0] = unpack2(half ? l2[0] : h2q[0]); wf[1] = unpack2(half ? l2[1] : h2q[1]);
#pragma unroll
      for (int i = 2; i < 6; ++i) wf[i] = unpack2(half ? l2[i] : l2[i - 2]);
      if (n_valid == G) { h2q[0] = l2[4]; h2q[1] = l2[5]; }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float2 acc = __ffma2_rn(w2[2], wf[k + 2], __ffma2_rn(w2[1], wf[k + 1], __fmul2_rn(w2[0], wf[k])));
        f2q[k] = add_bf2(pack_bf16(acc.x, acc.y), b2q);
      }
    }
    // ---- stage B: modal recurrence on this half's four states, sequential in t; partial residue sums
    float2 pc[G];
#pragma unroll
    for (int g = 0; g < G; ++g) {
      if (g < n_valid) {
        const float2 x = unpack2(xq[g]);
        float2 ar = make_float2(0.f, 0.f), ai = ar;
#pragma unroll
        for (int s = 0; s < NSH; ++s) {
          const float2 t_ = __ffma2_rn(npi[s], si[s], x);
          const float2 nr = __ffma2_rn(pr[s], sr[s], t_);
          const float2 ni = __ffma2_rn(pr[s], si[s], __fmul2_rn(pi[s], sr[s]));
          sr[s] = nr; si[s] = ni;
          if (!STATE_ONLY) { ar = s ? __ffma2_rn(rr[s], nr, ar) : __fmul2_rn(rr[s], nr); ai = s ? __ffma2_rn(ri[s], ni, ai) : __fmul2_rn(ri[s], ni); }
        }
        if (!STATE_ONLY) pc[g] = __fadd2_rn(ar, ai);
      }
    }
    // ---- stage C: conv = partial(modes 0..3) + partial(modes 4..7) (rp to bf16); y = (conv + x1v*D) * x2 with the reference's roundings
    if (!STATE_ONLY) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float2 mine = half ? pc[4 + k] : pc[k];
        const float2 send = half ? pc[k] : pc[4 + k];
        const float2 recv = make_float2(__shfl_xor_sync(0xffffffffu, send.x, 16), __shfl_xor_sync(0xffffffffu, send.y, 16));
        const float2 c = __fadd2_rn(mine, recv);
        const uint32_t xk = half ? xq[4 + k] : xq[k];
        const uint32_t u = add_bf2(pack_bf16(c.x, c.y), mul_bf2(xk, dskq));
        if (4 * half + k < n_valid) ydst[(long long)k * ystride] = mul_bf2(u, f2q[k]);
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
  else if (a.state_out && seg == last_seg) dst = a.state_out + (((long long)b * a.D + ch) * NS) * 2;
  if (dst) {
    float2* e = reinterpret_cast<float2*>(dst) + m0;
#pragma unroll
    for (int s = 0; s < NSH; ++s) { e[s] = make_float2(sr[s].x, si[s].x); e[NS + s] = make_float2(sr[s].y, si[s].y); }
  }
}

}  // namespace evo_hy3
