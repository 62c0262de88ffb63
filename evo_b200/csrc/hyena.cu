// Fused Hyena operator for sm_100a.
//
// Replaces, in one pass over HBM, what stripedhyena 0.2.2 does with ~10 launches and
// ~60-70 B/token/channel of traffic (engine.parallel_fir -> compute_filter -> parallel_iir
// [-> prefill_via_modal_fft]):
//     z' = FIR3(z) + b                     depthwise causal short conv over 3D channels
//     (x2, x1, v) = column_split(z')       per head: [x2 | x1 | v]
//     x1v = x1 * v
//     c[t] = sum_{tau<=t} h[t-tau] x1v[tau],  h[k] = Re sum_s R_s p_s^k     (the "FFT conv")
//     y = (c + D * x1v) * x2
// The long convolution is evaluated as the exact modal recurrence it is defined by
//     s_s[t] = p_s s_s[t-1] + x1v[t],   c[t] = Re sum_s R_s s_s[t]
// (the same recurrence the reference uses for decode, engine.step_iir), so the end state
// s[L-1] -- what the reference obtains with a second set of FFTs in prefill_via_modal_fft --
// falls out for free, arbitrary L (8193!) costs nothing, and the algorithmic HBM traffic is
// 8 B per token per channel (read 3 bf16, write 1 bf16).
//
// Parallelisation: one thread per channel, sequential along L inside a segment; the grid is
// (channel blocks) x (batch) x (L segments).  With more than one segment a first pass
// computes each segment's zero-start end state (reads x1, v only) and the output pass
// starts every segment from the exactly combined carry  S_j = p^len S_{j-1} + E_{j-1}.
// The same carry algebra shards the sequence across GPUs (evo_hyena_combine_states).
//
// bf16 rounding points mirror the reference's tensor ops one for one (marked "rp").
#include "common.cuh"
#include "../../include/evo_b200.h"
#include <algorithm>
#include "hyena_tma.cuh"
#include "hyena_ms.cuh"
#include <stdlib.h>

using namespace evo;

namespace {

constexpr int NS = 8;        // state_size of Evo (evo-1-8k-base_inference.yml:14)
constexpr int TB = 8;        // tokens per software-pipelined batch
constexpr int THREADS = 128;

struct Args {
  const bf16* z; bf16* y;
  const bf16* fir_w; const bf16* fir_b; const bf16* Dskip;
  const float* poles; const float* residues;
  const bf16* halo; const float* state_in;
  float* state_out;
  float* seg_states;         // (B, nseg, D, NS, 2) zero-start end states of each segment
  int B, D, hd, nseg;
  long long L, seg_len;
};

__device__ __forceinline__ float ldbf(const bf16* p) {
  return __uint_as_float(((uint32_t)__ldg(reinterpret_cast<const unsigned short*>(p))) << 16);
}

struct Cplx { float r, i; };
__device__ __forceinline__ Cplx cmul(Cplx a, Cplx b) { return {a.r * b.r - a.i * b.i, a.r * b.i + a.i * b.r}; }
__device__ __forceinline__ Cplx cpow_int(Cplx p, long long n) {
  Cplx acc = {1.f, 0.f};
  while (n > 0) { if (n & 1) acc = cmul(acc, p); p = cmul(p, p); n >>= 1; }
  return acc;
}

// STATE_ONLY: no x2 / no output, just the zero-start end state of the segment.
template <bool STATE_ONLY>
__global__ void __launch_bounds__(THREADS) hyena_scan_kernel(const Args a) {
  const int ch = blockIdx.x * THREADS + threadIdx.x;
  if (ch >= a.D) return;
  const int b = blockIdx.y, seg = blockIdx.z;
  const long long t0 = (long long)seg * a.seg_len;
  const long long t1 = min(a.L, t0 + a.seg_len);
  if (t0 >= t1) return;
  const int head = ch / a.hd, o = ch % a.hd;
  const int c_x2 = head * 3 * a.hd + o, c_x1 = c_x2 + a.hd, c_v = c_x1 + a.hd;
  const long long C3 = 3LL * a.D;

  // per-channel constants
  float pr[NS], pi[NS], rr[NS], ri[NS], sr[NS], si[NS];
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    float2 pp = __ldg(reinterpret_cast<const float2*>(a.poles) + (long long)ch * NS + s);
    float2 rs = __ldg(reinterpret_cast<const float2*>(a.residues) + (long long)ch * NS + s);
    pr[s] = pp.x; pi[s] = pp.y; rr[s] = rs.x; ri[s] = -rs.y;   // Re(R s) = Rr sr - Ri si
    sr[s] = 0.f; si[s] = 0.f;
  }
  float w1[3], wv[3], w2[3] = {0.f, 0.f, 0.f}, b1, bv, b2 = 0.f, dsk = 0.f;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    w1[k] = ldbf(a.fir_w + (long long)c_x1 * 3 + k);
    wv[k] = ldbf(a.fir_w + (long long)c_v * 3 + k);
    if (!STATE_ONLY) w2[k] = ldbf(a.fir_w + (long long)c_x2 * 3 + k);
  }
  b1 = ldbf(a.fir_b + c_x1); bv = ldbf(a.fir_b + c_v);
  if (!STATE_ONLY) { b2 = ldbf(a.fir_b + c_x2); dsk = ldbf(a.Dskip + ch); }

  // carry entering this segment (output pass only; the state pass starts from zero)
  if (!STATE_ONLY) {
    if (a.state_in) {
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        float2 v = __ldg(reinterpret_cast<const float2*>(a.state_in) + ((long long)b * a.D + ch) * NS + s);
        sr[s] = v.x; si[s] = v.y;
      }
    }
    if (seg > 0) {
      Cplx pl[NS];
#pragma unroll
      for (int s = 0; s < NS; ++s) pl[s] = cpow_int({pr[s], pi[s]}, a.seg_len);
      for (int q = 0; q < seg; ++q) {
        const float2* e = reinterpret_cast<const float2*>(a.seg_states) + (((long long)b * a.nseg + q) * a.D + ch) * NS;
#pragma unroll
        for (int s = 0; s < NS; ++s) {
          float2 ev = e[s];
          Cplx c = cmul(pl[s], {sr[s], si[s]});
          sr[s] = c.r + ev.x; si[s] = c.i + ev.y;
        }
      }
    }
  }

  // FIR history: z[t0-2], z[t0-1] of the three channels
  const bf16* zb = a.z + (long long)b * a.L * C3;
  float h1[2] = {0.f, 0.f}, hv[2] = {0.f, 0.f}, h2[2] = {0.f, 0.f};
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    long long t = t0 - 2 + k;
    const bf16* row = nullptr;
    if (t >= 0) row = zb + t * C3;
    else if (a.halo) row = a.halo + ((long long)b * 2 + (t + 2)) * C3;
    if (row) { h1[k] = ldbf(row + c_x1); hv[k] = ldbf(row + c_v); if (!STATE_ONLY) h2[k] = ldbf(row + c_x2); }
  }

  bf16* yb = STATE_ONLY ? nullptr : a.y + (long long)b * a.L * a.D + ch;

  // software pipeline: batch n+1's loads are issued before batch n's arithmetic
  unsigned short n1[TB], nv[TB], n2[TB];
  auto load_batch = [&](long long tb) {
#pragma unroll
    for (int j = 0; j < TB; ++j) {
      long long t = tb + j;
      if (t < t1) {
        const unsigned short* row = reinterpret_cast<const unsigned short*>(zb + t * C3);
        n1[j] = __ldg(row + c_x1); nv[j] = __ldg(row + c_v);
        if (!STATE_ONLY) n2[j] = __ldg(row + c_x2);
      } else { n1[j] = 0; nv[j] = 0; n2[j] = 0; }
    }
  };
  load_batch(t0);
  for (long long tb = t0; tb < t1; tb += TB) {
    unsigned short c1[TB], cv[TB], c2[TB];
#pragma unroll
    for (int j = 0; j < TB; ++j) { c1[j] = n1[j]; cv[j] = nv[j]; c2[j] = n2[j]; }
    if (tb + TB < t1) load_batch(tb + TB);
#pragma unroll
    for (int j = 0; j < TB; ++j) {
      if (tb + j < t1) {
        float z1 = __uint_as_float((uint32_t)c1[j] << 16), zv = __uint_as_float((uint32_t)cv[j] << 16);
        // short FIR: conv (fp32 accumulate, rp) then bias (rp)
        float f1 = rbf(rbf(fmaf(w1[2], z1, fmaf(w1[1], h1[1], w1[0] * h1[0]))) + b1);
        float fv = rbf(rbf(fmaf(wv[2], zv, fmaf(wv[1], hv[1], wv[0] * hv[0]))) + bv);
        h1[0] = h1[1]; h1[1] = z1; hv[0] = hv[1]; hv[1] = zv;
        float x = rbf(f1 * fv);                                   // x1v = x1 * v (rp)
        float acc = 0.f;
#pragma unroll
        for (int s = 0; s < NS; ++s) {
          float t_ = fmaf(-pi[s], si[s], x);
          float nr = fmaf(pr[s], sr[s], t_);
          float ni = fmaf(pr[s], si[s], pi[s] * sr[s]);
          sr[s] = nr; si[s] = ni;
          if (!STATE_ONLY) { acc = fmaf(rr[s], nr, acc); acc = fmaf(ri[s], ni, acc); }
        }
        if (!STATE_ONLY) {
          float z2 = __uint_as_float((uint32_t)c2[j] << 16);
          float f2 = rbf(rbf(fmaf(w2[2], z2, fmaf(w2[1], h2[1], w2[0] * h2[0]))) + b2);
          h2[0] = h2[1]; h2[1] = z2;
          float yc = rbf(acc);                                    // y.to(bf16) (rp)
          float u = rbf(yc + rbf(x * dsk));                       // y + x1v * D (rp, rp)
          yb[(tb + j) * a.D] = __float2bfloat16_rn(u * f2);       // * x2 (rp)
        }
      }
    }
  }

  if (STATE_ONLY) {
    float2* e = reinterpret_cast<float2*>(a.seg_states) + (((long long)b * a.nseg + seg) * a.D + ch) * NS;
#pragma unroll
    for (int s = 0; s < NS; ++s) e[s] = make_float2(sr[s], si[s]);
  } else if (a.state_out && seg == a.nseg - 1) {
    float2* e = reinterpret_cast<float2*>(a.state_out) + ((long long)b * a.D + ch) * NS;
#pragma unroll
    for (int s = 0; s < NS; ++s) e[s] = make_float2(sr[s], si[s]);
  }
}

// out = p^{total_len - nseg_full... } fold: carry over all segments' zero-start end states (+ state_in).
// lengths (B) or NULL: row b's sequence ends at lengths[b] (ragged rows), so each segment contributes its effective length.
__global__ void hyena_fold_states_kernel(const float* __restrict__ seg_states, const float* __restrict__ state_in,
                                         const float* __restrict__ poles, float* __restrict__ out,
                                         int B, int D, int nseg, long long seg_len, long long L, const int* __restrict__ lengths) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;   // (b, ch, s)
  if (idx >= B * D * NS) return;
  int s = idx % NS, ch = (idx / NS) % D, b = idx / (NS * D);
  if (lengths) L = min(L, (long long)max(lengths[b], 0));
  float2 pp = reinterpret_cast<const float2*>(poles)[(long long)ch * NS + s];
  Cplx p = {pp.x, pp.y};
  Cplx acc = {0.f, 0.f};
  if (state_in) { float2 v = reinterpret_cast<const float2*>(state_in)[idx]; acc = {v.x, v.y}; }
  for (int q = 0; q < nseg; ++q) {
    long long len = max(0LL, min(seg_len, L - (long long)q * seg_len));
    float2 e = reinterpret_cast<const float2*>(seg_states)[(((long long)b * nseg + q) * D + ch) * NS + s];
    Cplx c = cmul(cpow_int(p, len), acc);
    acc = {c.r + e.x, c.i + e.y};
  }
  reinterpret_cast<float2*>(out)[idx] = make_float2(acc.r, acc.i);
}

// lengths (B) or NULL: the two rows before row b's own end (ragged rows); rows are still L apart in z
__global__ void fir_state_kernel(const bf16* __restrict__ z, const bf16* __restrict__ halo, bf16* __restrict__ out,
                                 int B, long long L, long long C3, const int* __restrict__ lengths) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // (b, c)
  if (idx >= (long long)B * C3) return;
  long long b = idx / C3, c = idx % C3;
  const long long Lb = lengths ? min(L, (long long)max(lengths[b], 0)) : L;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    long long t = Lb - 2 + k;
    bf16 v = __float2bfloat16_rn(0.f);
    if (t >= 0) v = z[(b * L + t) * C3 + c];
    else if (halo) v = halo[(b * 2 + (t + 2)) * C3 + c];
    out[idx * 2 + k] = v;
  }
}

// decode step (engine.step_fir + step_iir): 8 lanes per (b, channel).  Lane s owns modal state s (its pole, residue
// and state are one coalesced 8-byte load each); lanes 0..2 run the three FIR channels (x2, x1, v); lane 0 folds the
// eight residue products in the reference's order (sequential fma chain) and writes y.
__global__ void __launch_bounds__(256) hyena_step_kernel(const bf16* __restrict__ u, bf16* __restrict__ y, bf16* __restrict__ fir_state,
                                  float* __restrict__ state, const bf16* __restrict__ fir_w, const bf16* __restrict__ fir_b,
                                  const bf16* __restrict__ Dskip, const float* __restrict__ poles, const float* __restrict__ residues,
                                  int B, int D, int hd) {
  pdl_launch_dependents();
  static_assert(NS == 8, "one lane per modal state");
  const long long gidx = (long long)blockIdx.x * blockDim.x + threadIdx.x;      // (b, channel, s); B*D*8 is a multiple of 256
  const int s = (int)(gidx & 7);
  const long long idx = gidx >> 3;
  const int b = (int)(idx / D), ch = (int)(idx % D);
  const int head = ch / hd, o = ch % hd;
  const int base = (threadIdx.x & 31) & ~7;
  // Everything except u is older than the previous kernel (filter parameters; the states this kernel itself wrote one token ago),
  // so it is fetched BEFORE griddepcontrol.wait: under programmatic dependent launch these loads overlap the in-projection's tail.
  const float2 p = reinterpret_cast<const float2*>(poles)[(long long)ch * NS + s];
  const float2 r = reinterpret_cast<const float2*>(residues)[(long long)ch * NS + s];
  float2* st = reinterpret_cast<float2*>(state) + idx * NS + s;
  const float2 sv = *st;
  const float dskip = __bfloat162float(Dskip[ch]);
  const long long C3 = 3LL * D;
  const long long c = (long long)head * 3 * hd + (long long)(s < 3 ? s : 0) * hd + o;            // x2, x1, v (lanes 0..2)
  bf16* fs = fir_state + (b * C3 + c) * 2;
  bf16 s0_b = __float2bfloat16_rn(0.f), s1_b = s0_b;
  float w0 = 0.f, w1 = 0.f, w2 = 0.f, fb = 0.f;
  if (s < 3) {
    s0_b = fs[0]; s1_b = fs[1];
    w0 = __bfloat162float(fir_w[c * 3 + 0]); w1 = __bfloat162float(fir_w[c * 3 + 1]); w2 = __bfloat162float(fir_w[c * 3 + 2]);
    fb = __bfloat162float(fir_b[c]);
  }
  pdl_wait();
  float f = 0.f;
  if (s < 3) {
    const bf16 un_b = u[b * C3 + c];
    const float un = __bfloat162float(un_b);
    const float s0 = __bfloat162float(s0_b), s1 = __bfloat162float(s1_b);
    // y = h0*u + sum(fir_state*h) + bias, bf16 tensor ops: each product / sum rounds (rp)
    const float t0 = rbf(w2 * un);
    const float t1 = rbf(rbf(s0 * w0) + rbf(s1 * w1));          // torch.sum over two bf16 products (fp32 accumulate, rp)
    f = rbf(rbf(t0 + t1) + fb);
    fs[0] = s1_b; fs[1] = un_b;
  }
  const float x2 = __shfl_sync(0xffffffffu, f, base + 0);
  const float x1 = __shfl_sync(0xffffffffu, f, base + 1);
  const float v = __shfl_sync(0xffffffffu, f, base + 2);
  const float x = rbf(x1 * v);
  const float nr = fmaf(p.x, sv.x, fmaf(-p.y, sv.y, x));
  const float ni = fmaf(p.x, sv.y, p.y * sv.x);
  *st = make_float2(nr, ni);
  float acc = 0.f;
#pragma unroll
  for (int t = 0; t < NS; ++t) {
    const float rx = __shfl_sync(0xffffffffu, r.x, base + t), ry = __shfl_sync(0xffffffffu, r.y, base + t);
    const float nrt = __shfl_sync(0xffffffffu, nr, base + t), nit = __shfl_sync(0xffffffffu, ni, base + t);
    acc = fmaf(rx, nrt, acc); acc = fmaf(-ry, nit, acc);
  }
  // y = x2 * (res_state + D * x1v): D*x1v is a bf16 product (rp); the rest is fp32, cast to bf16 at the end
  if (s == 0) y[idx] = __float2bfloat16_rn(x2 * (acc + rbf(dskip * x)));
}

bool use_tma_path(const evo_hyena_params* p) {
  return p->D % evo_hy2::CH_PER_CTA == 0 && p->D / p->nheads == 128;
}

// Sequential-in-L is the efficient form (one HBM pass, no carry pass); split L only when the
// (channel block x batch) grid cannot occupy the chip.
int pick_segments(const evo_hyena_params* p) {
  const long long L = p->L;
  if (p->force_segments > 0) return (int)std::min<long long>(p->force_segments, std::max<long long>(1, L));
  const int per_cta = use_tma_path(p) ? evo_hy2::CH_PER_CTA : THREADS;
  long long blocks = (long long)((p->D + per_cta - 1) / per_cta) * p->B;
  int sms = device_sm_count();
  if (blocks * 5 >= sms * 3 || L < 1024) return 1;
  // ONE wave: the largest segment count whose grid still fits the SMs (16 channel blocks x 9 segments = 144 CTAs on 148 SMs;
  // rounding up to 10 gave 160 CTAs = two waves: 0.52 ms against 0.36 ms at B = 1, L = 16384, profiles/r02_hyena_micro_call2.jsonl)
  long long want = std::max<long long>(1, sms / blocks);
  long long max_by_len = std::max<long long>(1, L / 512);
  return (int)std::max<long long>(1, std::min<long long>(std::min<long long>(want, max_by_len), 64));
}

}  // namespace

extern "C" size_t evo_hyena_fwd_workspace(const evo_hyena_params* p) {
  if (p->L <= 0) return 0;
  int nseg = pick_segments(p);
  if (nseg <= 1 && !p->state_only) return 0;
  return (size_t)p->B * nseg * p->D * NS * 2 * sizeof(float);
}

// segment geometry: equal segments, none empty
static void segment_geometry(const evo_hyena_params* p, int& nseg, long long& seg_len) {
  nseg = pick_segments(p);
  seg_len = (p->L + nseg - 1) / nseg;
  nseg = (int)((p->L + seg_len - 1) / seg_len);
}

// lengths == NULL: evo_hyena_fwd; otherwise evo_hyena_fwd_ragged (mode-split TMA path only, checked by the caller)
static int hyena_fwd_impl(const evo_hyena_params* p, const int* lengths, void* workspace, size_t workspace_bytes, void* stream) {
  EVO_REQUIRE(p->S == NS, "evo_hyena_fwd: state_size %d unsupported (kernel is specialised for %d)", p->S, NS);
  EVO_REQUIRE(p->nheads > 0 && p->D % p->nheads == 0, "evo_hyena_fwd: D %% nheads != 0");
  EVO_REQUIRE(p->B > 0 && p->B <= 65535, "evo_hyena_fwd: bad batch %d", p->B);
  if (p->L == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  int nseg; long long seg_len;
  segment_geometry(p, nseg, seg_len);
  size_t need = evo_hyena_fwd_workspace(p);
  EVO_REQUIRE(workspace_bytes >= need && (need == 0 || workspace), "evo_hyena_fwd: workspace too small (%zu < %zu)", workspace_bytes, need);
  if (p->state_only) EVO_REQUIRE(p->state_out != nullptr, "evo_hyena_fwd: state_only needs state_out");
  else EVO_REQUIRE(p->y != nullptr, "evo_hyena_fwd: y is NULL");
  int rc;
  if (use_tma_path(p)) {
    using namespace evo_hy2;
    CUtensorMap tmZ;
    uint64_t dims[3] = {(uint64_t)3 * p->D, (uint64_t)p->L, (uint64_t)p->B};
    uint64_t str[2] = {(uint64_t)3 * p->D * 2, (uint64_t)p->L * 3 * p->D * 2};
    uint32_t box[3] = {128, (uint32_t)T2, 1};
    if ((rc = make_tmap_nd_bf16(&tmZ, p->z, 3, dims, str, box, false))) return rc;
    Args2 a;
    a.y = (bf16*)p->y; a.z = (const bf16*)p->z;
    a.fir_w = (const bf16*)p->fir_w; a.fir_b = (const bf16*)p->fir_b; a.Dskip = (const bf16*)p->Dskip;
    a.poles = p->poles; a.residues = p->residues; a.halo = (const bf16*)p->halo; a.state_in = p->state_in; a.state_out = p->state_out;
    a.seg_states = (float*)workspace; a.B = p->B; a.D = p->D; a.nseg = nseg; a.L = p->L; a.seg_len = seg_len;
    a.lengths = lengths;
    static unsigned long long done_s = 0, done_o = 0;
    if ((rc = ensure_dyn_smem(hyena_scan_tma_kernel<true>, smem_bytes(STAGES), done_s))) return rc;
    if ((rc = ensure_dyn_smem(hyena_scan_tma_kernel<false>, smem_bytes(STAGES), done_o))) return rc;
    // 1 (default) = mode-split kernel (hyena_ms.cuh: 8 compute warps, 4 modal states per thread); 0 = round-1 kernel
    // (4 compute warps, 8 states per thread), kept for A/B timing and as a second implementation in the parity tests
    const char* env_v = getenv("EVO_B200_HYENA_VARIANT");      // read per call: experiments flip it inside one process
    const int variant = env_v ? atoi(env_v) : 1;
    static unsigned long long done_ms = 0, done_mo = 0;
    if ((rc = ensure_dyn_smem(evo_hy3::hyena_scan_ms_kernel<true>, smem_bytes(STAGES), done_ms))) return rc;
    if ((rc = ensure_dyn_smem(evo_hy3::hyena_scan_ms_kernel<false>, smem_bytes(STAGES), done_mo))) return rc;
    dim3 grid(p->D / CH_PER_CTA, p->B, nseg), block(variant == 1 ? evo_hy3::THREADS : evo_hy2::THREADS);
    auto k_state = variant == 1 ? evo_hy3::hyena_scan_ms_kernel<true> : hyena_scan_tma_kernel<true>;
    auto k_out = variant == 1 ? evo_hy3::hyena_scan_ms_kernel<false> : hyena_scan_tma_kernel<false>;
    if (lengths) {
      EVO_REQUIRE(variant == 1, "evo_hyena_fwd_ragged: only the mode-split scan (EVO_B200_HYENA_VARIANT=1) takes per-row lengths");
      static unsigned long long done_rs = 0, done_ro = 0;
      if ((rc = ensure_dyn_smem(evo_hy3::hyena_scan_ms_kernel<true, true>, smem_bytes(STAGES), done_rs))) return rc;
      if ((rc = ensure_dyn_smem(evo_hy3::hyena_scan_ms_kernel<false, true>, smem_bytes(STAGES), done_ro))) return rc;
      k_state = evo_hy3::hyena_scan_ms_kernel<true, true>;
      k_out = evo_hy3::hyena_scan_ms_kernel<false, true>;
    }
    // ring depth 4 (96 KB): two CTAs can co-reside and hide each other's latency when the grid exceeds the SM count.
    // An 8-deep ring for single-CTA-per-SM grids was measured and did not help (1.21 vs 1.06-1.13 ms at B=8, L=8193).
    a.nst = 4;
    const int SMEM_BYTES = smem_bytes(a.nst);
    if (p->state_only) {
      k_state<<<grid, block, SMEM_BYTES, st>>>(tmZ, a);
      if ((rc = check_launch("hyena_scan<state>"))) return rc;
    } else {
      if (nseg > 1 && !p->reuse_segment_states) {
        dim3 g2(grid.x, grid.y, nseg - 1);
        k_state<<<g2, block, SMEM_BYTES, st>>>(tmZ, a);
        if ((rc = check_launch("hyena_scan<state>"))) return rc;
      }
      k_out<<<grid, block, SMEM_BYTES, st>>>(tmZ, a);
      if ((rc = check_launch("hyena_scan<out>"))) return rc;
    }
  } else {
    Args a;
    a.z = (const bf16*)p->z; a.y = (bf16*)p->y;
    a.fir_w = (const bf16*)p->fir_w; a.fir_b = (const bf16*)p->fir_b; a.Dskip = (const bf16*)p->Dskip;
    a.poles = p->poles; a.residues = p->residues;
    a.halo = (const bf16*)p->halo; a.state_in = p->state_in; a.state_out = p->state_out;
    a.seg_states = (float*)workspace;
    a.B = p->B; a.D = p->D; a.hd = p->D / p->nheads; a.nseg = nseg; a.L = p->L; a.seg_len = seg_len;
    dim3 block(THREADS);
    dim3 grid((p->D + THREADS - 1) / THREADS, p->B, nseg);
    if (p->state_only) {
      hyena_scan_kernel<true><<<grid, block, 0, st>>>(a);
      if ((rc = check_launch("hyena_scan<state>"))) return rc;
    } else {
      if (nseg > 1 && !p->reuse_segment_states) {
        dim3 g2(grid.x, grid.y, nseg - 1);     // the last segment's zero-start state is never needed
        hyena_scan_kernel<true><<<g2, block, 0, st>>>(a);
        if ((rc = check_launch("hyena_scan<state>"))) return rc;
      }
      hyena_scan_kernel<false><<<grid, block, 0, st>>>(a);
      if ((rc = check_launch("hyena_scan<out>"))) return rc;
    }
  }
  if (p->state_only) {
    int n = p->B * p->D * NS;
    hyena_fold_states_kernel<<<(n + 255) / 256, 256, 0, st>>>((const float*)workspace, p->state_in, p->poles, p->state_out, p->B, p->D, nseg, seg_len, p->L, lengths);
    if ((rc = check_launch("hyena_fold_states"))) return rc;
  }
  if (p->fir_state_out) {
    long long n = (long long)p->B * 3 * p->D;
    fir_state_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const bf16*)p->z, (const bf16*)p->halo, (bf16*)p->fir_state_out, p->B, p->L, 3LL * p->D, lengths);
    if ((rc = check_launch("fir_state"))) return rc;
  }
  return 0;
}

extern "C" int evo_hyena_fwd(const evo_hyena_params* p, void* workspace, size_t workspace_bytes, void* stream) {
  return hyena_fwd_impl(p, nullptr, workspace, workspace_bytes, stream);
}

extern "C" size_t evo_hyena_fwd_ragged_workspace(const evo_hyena_params* p) { return evo_hyena_fwd_workspace(p); }

extern "C" int evo_hyena_fwd_ragged(const evo_hyena_params* p, const int32_t* lengths_dev, void* workspace, size_t workspace_bytes, void* stream) {
  EVO_REQUIRE(lengths_dev != nullptr, "evo_hyena_fwd_ragged: lengths is NULL");
  EVO_REQUIRE(p->halo == nullptr && p->state_in == nullptr, "evo_hyena_fwd_ragged: halo / state_in (a continued prefill) are not supported with per-row lengths");
  EVO_REQUIRE(!p->reuse_segment_states, "evo_hyena_fwd_ragged: reuse_segment_states is not supported with per-row lengths");
  EVO_REQUIRE(p->nheads > 0 && p->D % p->nheads == 0 && use_tma_path(p),
              "evo_hyena_fwd_ragged: needs head_dim 128 and D %% %d == 0 (the mode-split scan)", evo_hy2::CH_PER_CTA);
  return hyena_fwd_impl(p, lengths_dev, workspace, workspace_bytes, stream);
}

extern "C" int evo_hyena_step(const void* u, void* y, void* fir_state, float* state,
                              const void* fir_w, const void* fir_b, const void* Dskip,
                              const float* poles, const float* residues,
                              int B, int D, int S, int nheads, void* stream) {
  EVO_REQUIRE(S == NS, "evo_hyena_step: state_size %d unsupported", S);
  long long n = (long long)B * D * NS;
  if (n == 0) return 0;
  EVO_REQUIRE(D % 32 == 0, "evo_hyena_step: D (%d) must be a multiple of 32", D);
  EVO_CUDA(launch_pdl_at(4, hyena_step_kernel, dim3((unsigned)(n / 256)), dim3(256), 0, (cudaStream_t)stream, (const bf16*)u, (bf16*)y, (bf16*)fir_state, state,
      (const bf16*)fir_w, (const bf16*)fir_b, (const bf16*)Dskip, poles, residues, B, D, D / nheads));
  return check_launch("evo_hyena_step");
}

__global__ void combine_states_kernel(const float* __restrict__ ends, float* __restrict__ state_in, const float* __restrict__ poles,
                                      int rank, long long seg_len, int B, int D) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;   // (b, ch, s)
  if (idx >= B * D * NS) return;
  int s = idx % NS, ch = (idx / NS) % D;
  float2 pp = reinterpret_cast<const float2*>(poles)[(long long)ch * NS + s];
  Cplx pl = cpow_int({pp.x, pp.y}, seg_len);
  Cplx acc = {0.f, 0.f};
  long long per = (long long)B * D * NS;
  for (int q = 0; q < rank; ++q) {
    float2 e = reinterpret_cast<const float2*>(ends)[q * per + idx];
    Cplx c = cmul(pl, acc);
    acc = {c.r + e.x, c.i + e.y};
  }
  reinterpret_cast<float2*>(state_in)[idx] = make_float2(acc.r, acc.i);
}

extern "C" int evo_hyena_combine_states(const float* ends, float* state_in, const float* poles,
                                        int rank, int nranks, int64_t seg_len, int B, int D, int S, void* stream) {
  EVO_REQUIRE(S == NS, "evo_hyena_combine_states: state_size %d unsupported", S);
  EVO_REQUIRE(rank >= 0 && rank < nranks, "evo_hyena_combine_states: bad rank");
  int n = B * D * NS;
  combine_states_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(ends, state_in, poles, rank, seg_len, B, D);
  return check_launch("evo_hyena_combine_states");
}

// ---------------------------------------------------------------------------------------------
// Sequence-parallel carry exchange over NVLink peer memory (no NCCL on the Hyena layers).
// Every rank owns a symmetric buffer set; a rank PUSHES its data into its slot of every peer's
// buffer with plain stores through the NVLink aperture, then raises a per-sender flag on the
// peer (release at system scope); consumers spin on their local flags (acquire) inside the
// kernel that needs the data, so the transfer overlaps whatever else the stream is doing and
// costs no collective launch.  Flags carry a monotonically increasing epoch.
// ---------------------------------------------------------------------------------------------
namespace {

__device__ __forceinline__ void st_release_sys(int* p, int v) { asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ int ld_acquire_sys(const int* p) { int v; asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }

__device__ __forceinline__ void wait_flag(const int* flag, int epoch) {
  unsigned spins = 0;
  while (ld_acquire_sys(flag) < epoch) {
    __nanosleep(64);
    if (++spins > (1u << 28)) __trap();     // ~20 s: a peer died; fail loudly instead of hanging the box
  }
}

// copy `n16` 16-byte words from src into slot `rank` of each destination in dsts[first..last], then flag
__global__ void peer_publish_kernel(const uint4* __restrict__ src, long long n16, uint4* const* __restrict__ dsts, int* const* __restrict__ flags,
                                    long long slot_stride16, int rank, int first, int last, int epoch, int* __restrict__ block_counter) {
  for (int p = first; p <= last; ++p) {
    uint4* d = dsts[p] + (long long)rank * slot_stride16;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (long long)gridDim.x * blockDim.x) d[i] = src[i];
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    int prev = atomicAdd(block_counter, 1);
    if (prev == (int)gridDim.x - 1) {
      *block_counter = 0;
      __threadfence_system();
      for (int p = first; p <= last; ++p) st_release_sys(flags[p] + rank, epoch);
    }
  }
}

__global__ void wait_flags_kernel(const int* __restrict__ flags, int first, int last, int epoch) {
  int q = first + threadIdx.x;
  if (q <= last) wait_flag(flags + q, epoch);
}

}  // namespace

extern "C" int evo_peer_publish(const void* src, int64_t bytes, void* const* peer_dsts, int* const* peer_flags, int64_t slot_stride_bytes,
                                int rank, int first_peer, int last_peer, int epoch, int* block_counter, void* stream) {
  EVO_REQUIRE(bytes % 16 == 0 && slot_stride_bytes % 16 == 0, "evo_peer_publish: sizes must be multiples of 16 bytes");
  if (first_peer > last_peer) return 0;
  long long n16 = bytes / 16;
  int blocks = (int)std::min<long long>(64, std::max<long long>(1, (n16 + 255) / 256));
  peer_publish_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((const uint4*)src, n16, (uint4* const*)peer_dsts, peer_flags, slot_stride_bytes / 16,
                                                               rank, first_peer, last_peer, epoch, block_counter);
  return check_launch("evo_peer_publish");
}

extern "C" int evo_peer_wait(const int* flags, int first, int last, int epoch, void* stream) {
  if (first > last) return 0;
  EVO_REQUIRE(last - first < 64, "evo_peer_wait: too many peers");
  wait_flags_kernel<<<1, 64, 0, (cudaStream_t)stream>>>(flags, first, last, epoch);
  return check_launch("evo_peer_wait");
}
