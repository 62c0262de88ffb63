"""`StripedHyena` with the object protocol evo-design/evo relies on, executed by libevo_b200.so.

Boundary obligations (SURVEY.md section 8b), each pinned by a reference call site:
  StripedHyena(cfg)                                  evo/models.py:146
  .load_state_dict(sd, strict=True) with HF names    evo/models.py:124-147
  .to_bfloat16_except_poles_residues(); .to(device)  evo/models.py:148-150
  model(ids) -> (logits, None)                       evo/scoring.py:81,116
  model(x, inference_params_dict=d) -> (logits, d)   evo/generation.py:152
  model.initialize_inference_params()                evo/generation.py:117

The module tree only exists to carry parameters under the checkpoint's key names; `forward`
never calls a torch op on activations.  torch supplies device memory and the stream.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from typing import Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import _lib
from .._lib import (EPI_BIAS, EPI_BIAS_RESID, EPI_BIAS_ROPE, EPI_GELU_GATE, EPI_HYENA_STEP, EPI_NONE, EPI_RESID, AttnParams, GemmParams,
                    GemmSmallMParams, HyenaParams, check, ptr)
from .cache import InferenceParams, RecurrentInferenceParams

# kernel variants (see include/evo_b200.h); overridable for experiments
# measured on B200, same box, interleaved A/B inside the power-capped 0.7 s step (profiles/r01_gemm_variant_ab_call32.txt):
# the 2-CTA 256x256 tile (variant 0) gives 93.1-93.2 k nt/s against 88.3-88.5 k for the 1-CTA 128x256 tile -- each CTA
# stages 32 KB instead of 48 KB per k-block, so the same FLOPs cost less operand traffic and power.  (An early-round
# comparison had the 1-CTA tile ahead by 2 %; that was before the traffic-aware rasterisation and with a
# release.cluster arrive in the pair's epilogue.)
GEMM_VARIANT = int(os.environ.get("EVO_B200_GEMM_VARIANT", "0"))
GEMM_VARIANT_GATE = int(os.environ.get("EVO_B200_GEMM_VARIANT_GATE", "0"))
# attention: 2 = ping-pong kernel (two query tiles per CTA, P in TMEM): 0.89-1.07 PFLOP/s vs 0.86-1.07 for variant 1
ATTN_VARIANT = int(os.environ.get("EVO_B200_ATTN_VARIANT", "2"))


def _round_up(x: int, m: int) -> int:
    return (x + m - 1) // m * m


# ----------------------------------------------------------------------------- parameter carriers
class _Scale(nn.Module):
    def __init__(self, dim):
        super().__init__()
        self.scale = nn.Parameter(torch.ones(dim))


class _Linear(nn.Module):
    def __init__(self, fan_in, fan_out, bias):
        super().__init__()
        self.weight = nn.Parameter(torch.empty(fan_out, fan_in).normal_(0.0, 1.0 / math.sqrt(fan_in)))
        self.bias = nn.Parameter(torch.zeros(fan_out)) if bias else None


def pack_w12(l1: torch.Tensor, l2: torch.Tensor, ipad: int) -> torch.Tensor:
    """(inner, K) x 2 -> (2*ipad, K): rows interleaved in 128-row groups [l1 rows g*128.. | l2 rows g*128..], zero rows past
    `inner`, so one 128x256 accumulator tile holds l1.x and l2.x of the same 128 inner features (gate fused in the epilogue)."""
    inner, k = l1.shape
    out = l1.new_zeros(ipad // 128, 2, 128, k)
    out[:, 0] = F.pad(l1, (0, 0, 0, ipad - inner)).view(ipad // 128, 128, k)
    out[:, 1] = F.pad(l2, (0, 0, 0, ipad - inner)).view(ipad // 128, 128, k)
    return out.view(2 * ipad, k)


def unpack_w12(w12: torch.Tensor, inner: int):
    ipad, k = w12.shape[0] // 2, w12.shape[1]
    v = w12.view(ipad // 128, 2, 128, k)
    return v[:, 0].reshape(ipad, k)[:inner], v[:, 1].reshape(ipad, k)[:inner]


class _GatedMLP(nn.Module):
    """ParallelGatedMLP parameters, held ONLY in the layouts the GEMMs read (SURVEY 8f-3: no second copy):
      w12 (2*ipad, D)  l1 / l2 interleaved per 128 rows, zero-padded 10928 -> 11008 (pack_w12)
      w3  (D, ipad)    l3 zero-padded along K
    The checkpoint's key names (mlp.l1.weight, mlp.l2.weight, mlp.l3.weight; evo/models.py:124-147) are what state_dict()
    shows and what load_state_dict() accepts: two hooks translate at the module boundary."""

    def __init__(self, cfg):
        super().__init__()
        d = cfg.hidden_size
        mult = cfg.get("inner_size_multiple_of", 64) * (cfg.get("model_parallel_size") or 1)
        inner = mult * ((int(2 * d * 4 / 3) + mult - 1) // mult)
        if cfg.get("inner_mlp_size") is not None:
            inner = cfg.get("inner_mlp_size")
        if (cfg.get("mlp_activation") or "silu") != "gelu":
            raise NotImplementedError("evo_b200 implements the Evo configs' exact-erf GELU gate only")
        self.inner, self.ipad = inner, _round_up(inner, 128)
        mk = lambda fo, fi: torch.empty(fo, fi).normal_(0.0, 1.0 / math.sqrt(fi))
        self.w12 = nn.Parameter(pack_w12(mk(inner, d), mk(inner, d), self.ipad))
        self.w3 = nn.Parameter(F.pad(mk(d, inner), (0, self.ipad - inner)))
        self._register_state_dict_hook(self._export_reference_keys)
        self._register_load_state_dict_pre_hook(self._import_reference_keys)

    @staticmethod
    def _export_reference_keys(module, state_dict, prefix, local_metadata):
        w12, w3 = state_dict.pop(prefix + "w12"), state_dict.pop(prefix + "w3")
        l1, l2 = unpack_w12(w12, module.inner)
        state_dict[prefix + "l1.weight"], state_dict[prefix + "l2.weight"] = l1.contiguous(), l2.contiguous()
        state_dict[prefix + "l3.weight"] = w3[:, :module.inner].contiguous()

    def _import_reference_keys(self, state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys, error_msgs):
        names = [prefix + n for n in ("l1.weight", "l2.weight", "l3.weight")]
        have = [n in state_dict for n in names]
        d = self.w3.shape[0]
        for n, ok, shape in zip(names, have, ((self.inner, d), (self.inner, d), (d, self.inner))):
            if not ok:
                missing_keys.append(n)
            elif tuple(state_dict[n].shape) != shape:
                error_msgs.append(f"size mismatch for {n}: copying a param with shape {tuple(state_dict[n].shape)} from checkpoint, the shape in current model is {shape}.")
                have = [False] * 3
        if have[0] and have[1]:
            state_dict[prefix + "w12"] = pack_w12(state_dict[names[0]], state_dict[names[1]], self.ipad)
        else:
            state_dict[prefix + "w12"] = self.w12.data         # reported above under the reference's own key names
        state_dict[prefix + "w3"] = F.pad(state_dict[names[2]], (0, self.ipad - self.inner)) if have[2] else self.w3.data
        for n in names:
            state_dict.pop(n, None)


class _HyenaFilter(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        d, s, k = cfg.hidden_size, cfg.state_size, cfg.short_filter_length
        if k != 3 or s != 8:
            raise NotImplementedError("kernels are specialised for short_filter_length=3, state_size=8 (the Evo configs)")
        if (cfg.get("hyena_filter_groups") or 1) != 1:
            raise NotImplementedError("hyena_filter_groups != 1")
        self.short_filter_weight = nn.Parameter(torch.randn(3 * d, 1, k) * 0.3)
        self.short_filter_bias = nn.Parameter(torch.randn(3 * d) * 0.1)
        self.D = nn.Parameter(torch.zeros(d))
        mag = 0.5 + 0.45 * torch.rand(d, s, 1)
        ang = (torch.rand(d, s, 1) * 2 - 1) * math.pi
        self.poles = nn.Parameter(torch.stack([mag * torch.cos(ang), mag * torch.sin(ang)], dim=-1))
        self.residues = nn.Parameter(torch.randn(d, s, 1, 2) * 0.3)


class _Rotary(nn.Module):
    """Carrier of `inv_freq`.  flash_attn registers it as a NON-persistent buffer (layers/rotary.py:366); stripedhyena re-registers it
    as a persistent one, so its checkpoints carry `...rotary_emb.inv_freq`.  That second fact is recalled, not verified here (SURVEY.md
    A.7), so loading accepts both: a checkpoint value is used when present, the constructor's analytic value when absent -- what the
    reference ends up with in either world."""

    def __init__(self, head_dim, base):
        super().__init__()
        self.head_dim, self.base = head_dim, base
        self.register_buffer("inv_freq", self.analytic())

    def analytic(self, device=None):
        return 1.0 / (self.base ** (torch.arange(0, self.head_dim, 2, dtype=torch.float32, device=device) / self.head_dim))

    def _load_from_state_dict(self, state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys, error_msgs):
        if prefix + "inv_freq" not in state_dict:
            state_dict = {**state_dict, prefix + "inv_freq": self.inv_freq if self.inv_freq.device.type != "meta" else self.analytic()}
        super()._load_from_state_dict(state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys, error_msgs)


class _MHA(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        d = cfg.hidden_size
        if (cfg.get("proj_groups") or 1) != 1:
            raise NotImplementedError("proj_groups != 1 (GQA) is not an Evo configuration")
        self.Wqkv = _Linear(d, 3 * d, bool(cfg.get("qkv_proj_bias", True)))
        self.out_proj = _Linear(d, d, bool(cfg.get("mha_out_proj_bias", True)))
        self.rotary_emb = _Rotary(d // cfg.num_attention_heads, cfg.get("rotary_emb_base") or 10000)


class _HyenaBlock(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        d = cfg.hidden_size
        self.pre_norm, self.post_norm = _Scale(d), _Scale(d)
        self.filter = _HyenaFilter(cfg)
        self.projections = _Linear(d, 3 * d, True)
        self.out_filter_dense = _Linear(d, d, True)
        self.mlp = _GatedMLP(cfg)


class _AttentionBlock(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        d = cfg.hidden_size
        self.pre_norm, self.post_norm = _Scale(d), _Scale(d)
        self.inner_mha_cls = _MHA(cfg)
        self.mlp = _GatedMLP(cfg)


class _Embedding(nn.Module):
    def __init__(self, vocab, dim):
        super().__init__()
        self.weight = nn.Parameter(torch.randn(vocab, dim) * (2.5 / math.sqrt(dim)))


# ----------------------------------------------------------------------------- the model
class StripedHyena(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.config = config
        d = config.hidden_size
        self.embedding_layer = _Embedding(config.vocab_size, d)
        self.norm = _Scale(d) if config.get("final_norm", True) else None
        self.unembed = self.embedding_layer if config.tie_embeddings else _Embedding(config.vocab_size, d)
        attn = set(config.attn_layer_idxs or [])
        self.blocks = nn.ModuleList(
            _AttentionBlock(config) if i in attn else _HyenaBlock(config) for i in range(config.num_layers))
        self._attn_idxs = attn
        self._packed = None
        self._rope = None
        self.gemm_variant = GEMM_VARIANT
        self.gemm_variant_gate = GEMM_VARIANT_GATE
        self.attn_variant = ATTN_VARIANT
        self.decode_graph = os.environ.get("EVO_B200_DECODE_GRAPH", "1") != "0"
        # rotary embedding inside the Wqkv GEMM's epilogue (EVO_EPI_BIAS_ROPE) instead of a separate pass over qkv; "0" = separate evo_rotary_qk
        self.fused_rope = os.environ.get("EVO_B200_FUSED_ROPE", "1") != "0"
        # tile-major weight copies for decode (GEMM variant 3): validated bit-identical but no faster on B200 (6.57 vs 6.65 ms/step:
        # the small-M GEMM is bound by bytes in flight per CTA and by too few CTAs at N=4096, not by DRAM page locality), so off
        self.decode_tiled = os.environ.get("EVO_B200_DECODE_TILED", "0") != "0"
        # decode-step GEMMs: stream-K weight-streaming kernel (csrc/gemm_smallm.cu) for batch <= 64; "0" = the 128x64 tiles
        self.decode_streamk = os.environ.get("EVO_B200_DECODE_STREAMK", "1") != "0"
        # programmatic dependent launch inside a decode step (evo_set_pdl): 0 off, 1 every kernel, 2 weight-streaming GEMMs only
        self.decode_pdl = int(os.environ.get("EVO_B200_DECODE_PDL", "4"))
        # the Hyena decode step inside the in-projection GEMM's epilogue (EVO_EPI_HYENA_STEP).  Bit-identical to the separate
        # evo_hyena_step launch but SLOWER on B200 (5.12 vs 4.30 ms/step at batch 16, profiles/r02_decode_fused_step_call8.txt): the
        # step of a tile runs on the 128 epilogue threads of its last contributor -- 16 batch rows x 8 states of dependent
        # load -> update -> store per thread in the GEMM's serial tail -- where the stand-alone kernel spreads the same 8 MB of state
        # traffic over 524 288 threads.  Off by default; kept as a tested option.
        self.decode_fused_step = os.environ.get("EVO_B200_DECODE_FUSED_STEP", "0") != "0"
        self._smallm_ws = None
        self._tiled = None   # tile-major weight copies for the weight-streaming decode GEMMs
        self._decode = None  # cached CUDA graph of one decode step (see _decode_forward)
        self._loop = None    # cached CUDA graph of one step of the on-device generation loop (see decode_loop)
        self._loop_ragged = None   # the same for prompts of different lengths (see decode_loop_ragged)
        self._prof = None   # set to a list to record (kind, algorithmic work, start event, end event) per kernel call

    # ---- reference API ------------------------------------------------------------------
    def to_bfloat16_except_poles_residues(self):
        for name, p in self.named_parameters():
            if "poles" not in name and "residues" not in name:
                p.data = p.data.to(torch.bfloat16)
        self._packed = None
        return self

    def initialize_inference_params(self):
        return {
            "mha": InferenceParams(max_seqlen=self.config.get("max_seqlen") or 8192,
                                   max_batch_size=self.config.get("max_batch_size") or 1, seqlen_offset=0),
            "hyena": RecurrentInferenceParams(fir_filter_length=self.config.short_filter_length,
                                              state_dim=self.config.state_size, seqlen_offset=0),
        }

    def load_state_dict(self, state_dict, strict: bool = True, **kw):
        out = super().load_state_dict(state_dict, strict=strict, **kw)
        self._packed = None
        self._decode = None
        self._loop = None
        self._loop_ragged = None
        self._tiled = None
        return out

    def _apply(self, fn, *a, **kw):
        out = super()._apply(fn, *a, **kw)
        self._packed = None
        self._rope = None
        self._decode = None
        self._loop = None
        self._loop_ragged = None
        self._tiled = None
        return out

    # ---- weight packing (once per load / move) ---------------------------------------------
    def _ensure_packed(self):
        if self._packed is not None:
            return self._packed
        dev = self.embedding_layer.weight.device
        if dev.type != "cuda":
            raise _lib.EvoError("evo_b200 runs on CUDA (sm_100a) only: move the model with .to('cuda:N'); there is no CPU path")
        for name, p in self.named_parameters():
            want = torch.float32 if ("poles" in name or "residues" in name) else torch.bfloat16
            if p.dtype != want:
                raise _lib.EvoError(f"parameter {name} is {p.dtype}; call to_bfloat16_except_poles_residues() (evo/models.py:148)")
            if p.device != dev:
                raise _lib.EvoError(f"parameter {name} is on {p.device}, expected {dev}")
        packed = {}
        for i, blk in enumerate(self.blocks):
            # the MLP parameters already live in the GEMM layouts (see _GatedMLP): nothing is copied here
            packed[i] = {"w12": blk.mlp.w12.data, "w3": blk.mlp.w3.data, "ipad": blk.mlp.ipad}
        hd = self.config.hidden_size // self.config.num_attention_heads
        base = self.config.get("rotary_emb_base") or 10000
        # flash_attn keeps the checkpoint's inv_freq buffer when it is fp32 and recomputes it in fp32 otherwise
        # (layers/rotary.py:386-401); one table per model: every attention block must then agree
        analytic = (1.0 / (base ** (torch.arange(0, hd, 2, dtype=torch.float32) / hd))).to(dev)
        bufs = [self.blocks[i].inner_mha_cls.rotary_emb.inv_freq for i in sorted(self._attn_idxs)]
        if bufs and bufs[0].dtype == torch.float32:
            for b_ in bufs[1:]:
                if b_.dtype != torch.float32 or not torch.equal(b_, bufs[0]):
                    raise _lib.EvoError("attention blocks carry different rotary inv_freq buffers; one rope table per model is supported")
            packed["inv_freq"] = bufs[0].detach().to(dev).contiguous()
        else:
            packed["inv_freq"] = analytic
        self._packed = packed
        return packed

    # ---- thin wrappers over the C ABI ------------------------------------------------------------
    @staticmethod
    def _stream():
        return C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def _record(self, kind, work, launch):
        """Run `launch()`; when profiling is on, bracket it with CUDA events on the launch stream."""
        if self._prof is None:
            return launch()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        launch()
        e1.record()
        self._prof.append((kind, work, e0, e1))

    def _gemm(self, a, w, out, M, N, K, epi, bias=None, resid=None, ldc=None, variant=None, rope=None, peers=None):
        """rope = (cos_ptr, sin_ptr, tokens_per_sequence, rotated_columns) for EPI_BIAS_ROPE;
        peers = (ctypes array of peer pointers, n, period, inner, row0): peer-scattered output (see evo_gemm_params), out may be None."""
        if variant is None:
            variant = self.gemm_variant_gate if epi == EPI_GELU_GATE else self.gemm_variant
        p = GemmParams(A=a.data_ptr(), lda=K, W=w.data_ptr(), C=out.data_ptr() if out is not None else None, ldc=ldc or N,
                       bias=bias.data_ptr() if bias is not None else None,
                       residual=resid.data_ptr() if resid is not None else None, ldr=ldc or N,
                       M=M, N=N, K=K, epilogue=epi, variant=variant)
        if rope is not None:
            p.rope_cos, p.rope_sin, p.rope_L, p.rope_cols = rope
        if peers is not None:
            arr, n, period, inner, row0 = peers
            p.c_peers, p.n_c_peers, p.peer_period, p.peer_inner, p.peer_row0 = C.cast(arr, C.c_void_p), n, period, inner, row0
        self._record(f"gemm/{N}x{K}/e{epi}/v{variant}", 2.0 * M * N * K, lambda: check(_lib.lib().evo_gemm(C.byref(p), self._stream()), "evo_gemm"))

    def _gemm_smallm(self, a, w, out, M, N, K, epi, bias=None, resid=None, step=None):
        """Decode-step linear layer (M <= 64): stream-K weight-streaming kernel, gate epilogue fused.
        step = (fir_state, state_real, filter module) for EPI_HYENA_STEP: the in-projection with the operator's decode step
        in its epilogue (out is then y (M, N/3))."""
        lib = _lib.lib()
        need = lib.evo_gemm_smallm_workspace(M, N, K, epi)
        ws = self._smallm_ws
        if ws is None or ws.numel() < need or ws.device != a.device:
            self._decode = None      # a captured decode graph holds the old workspace address
            ws = self._smallm_ws = torch.zeros(max(need, lib.evo_gemm_smallm_workspace(M, 256, 64, EPI_GELU_GATE), lib.evo_gemm_smallm_workspace(M, 384, 64, EPI_HYENA_STEP)),
                                               dtype=torch.uint8, device=a.device)
        n_out = N // 2 if epi == EPI_GELU_GATE else (N // 3 if epi == EPI_HYENA_STEP else N)
        p = GemmSmallMParams(A=a.data_ptr(), lda=K, W=w.data_ptr(), C=out.data_ptr(), ldc=n_out,
                             bias=bias.data_ptr() if bias is not None else None,
                             residual=resid.data_ptr() if resid is not None else None, ldr=n_out,
                             M=M, N=N, K=K, epilogue=epi, workspace=ws.data_ptr(), workspace_bytes=ws.numel())
        if step is not None:
            fs, st, f = step
            p.fir_state, p.state = fs.data_ptr(), st.data_ptr()
            p.fir_w, p.fir_b, p.Dskip = f.short_filter_weight.data_ptr(), f.short_filter_bias.data_ptr(), f.D.data_ptr()
            p.poles, p.residues = f.poles.data_ptr(), f.residues.data_ptr()
        self._record(f"gemm/{N}x{K}/e{epi}/streamk", 2.0 * M * N * K, lambda: check(lib.evo_gemm_smallm(C.byref(p), self._stream()), "evo_gemm_smallm"))

    def _rmsnorm(self, x, scale, out, rows):
        self._record("rmsnorm", 4.0 * rows * self.config.hidden_size, lambda: check(_lib.lib().evo_rmsnorm(
            ptr(x), ptr(scale), ptr(out), rows, self.config.hidden_size, float(self.config.eps), self._stream()), "evo_rmsnorm"))

    def _rope_tables(self, n_pos, dev):
        if self._rope is None or self._rope[0].shape[0] < n_pos:
            hd2 = self.config.hidden_size // self.config.num_attention_heads // 2
            scaling = float(self.config.get("rotary_emb_scaling_factor") or 1.0) if self.config.get("use_interpolated_rotary_pos_emb") else 1.0
            n = max(n_pos, 2048)
            cos = torch.empty(n, hd2, dtype=torch.bfloat16, device=dev)
            sin = torch.empty_like(cos)
            check(_lib.lib().evo_rope_tables(ptr(cos), ptr(sin), ptr(self._packed["inv_freq"]), 0, n, hd2, scaling, self._stream()), "evo_rope_tables")
            self._rope = (cos, sin)
            self._decode = None      # a captured decode graph holds the old tables' addresses
        return self._rope

    def _mlp_residual(self, i, blk, u, M):
        """out = l3(gelu(l1 n) * l2 n) + u with n = post_norm(u); returns a new (M, D) tensor."""
        d = self.config.hidden_size
        pk = self._packed[i]
        xn = torch.empty_like(u)
        self._rmsnorm(u, blk.post_norm.scale, xn, M)
        g = torch.empty(M, pk["ipad"], dtype=torch.bfloat16, device=u.device)
        self._gemm(xn, pk["w12"], g, M, 2 * pk["ipad"], d, EPI_GELU_GATE, ldc=pk["ipad"])
        out = xn  # reuse
        self._gemm(g, pk["w3"], out, M, d, pk["ipad"], EPI_RESID, resid=u)
        return out

    def _hyena_block(self, i, blk, u, B, L, ip: Optional[RecurrentInferenceParams], lengths=None):
        cfg = self.config
        d, H = cfg.hidden_size, cfg.num_attention_heads
        M = B * L
        dev = u.device
        f = blk.filter
        xn = torch.empty_like(u)
        self._rmsnorm(u, blk.pre_norm.scale, xn, M)
        z = torch.empty(M, 3 * d, dtype=torch.bfloat16, device=dev)
        self._gemm(xn, blk.projections.weight, z, M, 3 * d, d, EPI_BIAS, bias=blk.projections.bias)
        y = xn  # (M, D) buffer reuse
        lib = _lib.lib()
        have_state = ip is not None and i in ip.fir_state_dict
        if have_state and L == 1:
            st = ip.state_dict[i]
            if not st.is_contiguous():
                st = st.contiguous(); ip.state_dict[i] = st
            fs = ip.fir_state_dict[i]
            if not fs.is_contiguous():
                fs = fs.contiguous(); ip.fir_state_dict[i] = fs
            check(lib.evo_hyena_step(ptr(z), ptr(y), ptr(fs), ptr(torch.view_as_real(st)), ptr(f.short_filter_weight),
                                     ptr(f.short_filter_bias), ptr(f.D), ptr(f.poles), ptr(f.residues),
                                     B, d, cfg.state_size, H, self._stream()), "evo_hyena_step")
        else:
            hp = HyenaParams(z=z.data_ptr(), y=y.data_ptr(), fir_w=f.short_filter_weight.data_ptr(), fir_b=f.short_filter_bias.data_ptr(),
                             Dskip=f.D.data_ptr(), poles=f.poles.data_ptr(), residues=f.residues.data_ptr(),
                             B=B, L=L, D=d, S=cfg.state_size, nheads=H, force_segments=0, state_only=0)
            keep = []
            if have_state:  # continued prefill: history = stored states
                halo = ip.fir_state_dict[i].permute(0, 2, 1).contiguous()
                sin_ = torch.view_as_real(ip.state_dict[i].contiguous()).contiguous()
                hp.halo, hp.state_in = halo.data_ptr(), sin_.data_ptr()
                keep += [halo, sin_]
            if ip is not None:
                st_out = torch.empty(B, d, cfg.state_size, 2, dtype=torch.float32, device=dev)
                fs_out = torch.empty(B, 3 * d, 2, dtype=torch.bfloat16, device=dev)
                hp.state_out, hp.fir_state_out = st_out.data_ptr(), fs_out.data_ptr()
            if lengths is not None:     # right-padded rows (prefill_ragged): each row's scan and states end at its own length
                ws_bytes = lib.evo_hyena_fwd_ragged_workspace(C.byref(hp))
                ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
                self._record("hyena", 8.0 * B * L * d, lambda: check(lib.evo_hyena_fwd_ragged(C.byref(hp), ptr(lengths), ptr(ws), ws_bytes, self._stream()), "evo_hyena_fwd_ragged"))
            else:
                ws_bytes = lib.evo_hyena_fwd_workspace(C.byref(hp))
                ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
                self._record("hyena", 8.0 * B * L * d, lambda: check(lib.evo_hyena_fwd(C.byref(hp), ptr(ws), ws_bytes, self._stream()), "evo_hyena_fwd"))
            if ip is not None:
                ip.state_dict[i] = torch.view_as_complex(st_out)
                ip.fir_state_dict[i] = fs_out
        u2 = torch.empty_like(u)
        self._gemm(y, blk.out_filter_dense.weight, u2, M, d, d, EPI_BIAS_RESID, bias=blk.out_filter_dense.bias, resid=u)
        return self._mlp_residual(i, blk, u2, M)

    def _attention_block(self, i, blk, u, B, L, ip: Optional[InferenceParams]):
        cfg = self.config
        d, H = cfg.hidden_size, cfg.num_attention_heads
        hd = d // H
        M = B * L
        dev = u.device
        mha = blk.inner_mha_cls
        lib = _lib.lib()
        xn = torch.empty_like(u)
        self._rmsnorm(u, blk.pre_norm.scale, xn, M)
        qkv = torch.empty(M, 3 * d, dtype=torch.bfloat16, device=dev)
        off = int(ip.seqlen_offset) if ip is not None else 0
        cos, sin = self._rope_tables(off + L, dev)
        hd2 = hd // 2
        cos_p, sin_p = cos.data_ptr() + off * hd2 * 2, sin.data_ptr() + off * hd2 * 2
        if self.fused_rope and mha.Wqkv.bias is not None and hd == 128 and self.gemm_variant in (0, 1):
            # rotary applied in the projection's epilogue, where flash_attn's MHA applies it (mha.py:635-648): no second pass over qkv
            self._gemm(xn, mha.Wqkv.weight, qkv, M, 3 * d, d, EPI_BIAS_ROPE, bias=mha.Wqkv.bias, rope=(cos_p, sin_p, L, 2 * d))
        else:
            self._gemm(xn, mha.Wqkv.weight, qkv, M, 3 * d, d, EPI_BIAS if mha.Wqkv.bias is not None else EPI_NONE, bias=mha.Wqkv.bias)
            self._record("rotary", 8.0 * M * d, lambda: check(lib.evo_rotary_qk(ptr(qkv), C.c_void_p(cos_p), C.c_void_p(sin_p), B, L, H, hd, self._stream()), "evo_rotary_qk"))
        ctx = xn  # reuse
        ap = AttnParams(out=ctx.data_ptr(), B=B, Lq=L, H=H, hd=hd, q_pos0=off, softmax_scale=1.0 / math.sqrt(hd))
        ap.q, ap.q_tok_stride, ap.q_batch_stride = qkv.data_ptr(), 3 * d, L * 3 * d
        if ip is None:
            ap.k, ap.v = qkv.data_ptr() + d * 2, qkv.data_ptr() + 2 * d * 2
            ap.kv_tok_stride, ap.kv_batch_stride, ap.Lk = 3 * d, L * 3 * d, L
        else:
            if i not in ip.key_value_memory_dict:  # flash_attn/modules/mha.py:344-353 (zeros instead of empty: quirk Q1)
                ip.key_value_memory_dict[i] = torch.zeros(ip.max_batch_size, ip.max_seqlen, 2, H, hd, dtype=torch.bfloat16, device=dev)
            cache = ip.key_value_memory_dict[i]
            if B > cache.shape[0] or off + L > cache.shape[1]:
                raise _lib.EvoError(f"KV cache too small: batch {B} > {cache.shape[0]} or length {off + L} > {cache.shape[1]} (mha.py:366-367)")
            check(lib.evo_kv_append(ptr(qkv), ptr(cache), B, L, H, hd, off, cache.shape[1], self._stream()), "evo_kv_append")
            ap.k, ap.v = cache.data_ptr(), cache.data_ptr() + d * 2
            ap.kv_tok_stride, ap.kv_batch_stride, ap.Lk = 2 * d, cache.shape[1] * 2 * d, off + L
        ws_bytes = lib.evo_attn_fwd_workspace(C.byref(ap), self.attn_variant)
        ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
        causal_flops = 4.0 * B * H * hd * (L * (off + (L + 1) / 2.0))   # QK^T + PV over the visible (query, key) pairs
        self._record("attn", causal_flops, lambda: check(lib.evo_attn_fwd_ws(C.byref(ap), self.attn_variant, ptr(ws), ws_bytes, self._stream()), "evo_attn_fwd"))
        u2 = torch.empty_like(u)
        self._gemm(ctx, mha.out_proj.weight, u2, M, d, d, EPI_BIAS_RESID if mha.out_proj.bias is not None else EPI_RESID,
                   bias=mha.out_proj.bias, resid=u)
        return self._mlp_residual(i, blk, u2, M)

    # ---- forward ---------------------------------------------------------------------------------
    def forward(self, x, inference_params_dict=None, padding_mask=None):
        if padding_mask is not None:
            raise NotImplementedError("padding_mask is never passed by evo (evo/scoring.py:81); not implemented")
        if x.dim() != 2:
            raise ValueError("input ids must be (batch, length)")
        if x.dtype not in (torch.int32, torch.int64):
            raise TypeError("input ids must be int32 or int64")
        self._ensure_packed()
        dev = self.embedding_layer.weight.device
        if x.device != dev:
            raise _lib.EvoError(f"input ids on {x.device}, model on {dev}")
        x = x.contiguous()
        B, L = x.shape
        M = B * L
        d = self.config.hidden_size
        V = self.config.vocab_size
        if L == 1 and inference_params_dict is not None and self._can_step(inference_params_dict, B):
            with torch.cuda.device(dev), torch.no_grad():
                return self._decode_forward(x, inference_params_dict), inference_params_dict
        with torch.cuda.device(dev), torch.no_grad():
            u = self._backbone(x, B, L, inference_params_dict)
            logits = torch.empty(M, V, dtype=torch.bfloat16, device=dev)
            self._gemm(u, self.unembed.weight, logits, M, V, d, EPI_NONE)
        return logits.view(B, L, V), inference_params_dict

    def _backbone(self, x, B, L, inference_params_dict=None, lengths=None):
        """embed -> all blocks -> final norm: the (B*L, D) bf16 input of the unembedding.
        lengths: (B) int32 on the device for right-padded rows (see prefill_ragged), else None."""
        M, d, V = B * L, self.config.hidden_size, self.config.vocab_size
        dev = x.device
        u = torch.empty(M, d, dtype=torch.bfloat16, device=dev)
        check(_lib.lib().evo_embed(ptr(x), int(x.dtype == torch.int64), ptr(self.embedding_layer.weight), ptr(u),
                                   M, d, V, self._stream()), "evo_embed")
        for i, blk in enumerate(self.blocks):
            if i in self._attn_idxs:
                ip = inference_params_dict["mha"] if inference_params_dict is not None else None
                u = self._attention_block(i, blk, u, B, L, ip)
            else:
                ip = inference_params_dict["hyena"] if inference_params_dict is not None else None
                u = self._hyena_block(i, blk, u, B, L, ip, lengths)
        if self.norm is not None:
            xn = torch.empty_like(u)
            self._rmsnorm(u, self.norm.scale, xn, M)
            u = xn
        return u

    def prefill_ragged(self, ids, lengths, ipd):
        """Prefill of prompts of different lengths in one batch: ids (B, W) right-padded, row b's prompt is ids[b, :lengths[b]].
        Populates the fresh inference params `ipd` as B separate prefills would -- Hyena state and FIR state after each row's
        own last token (evo_hyena_fwd_ragged), keys and values of positions [0, lengths[b]) in the KV cache -- and returns the
        (B, V) bf16 logits at each row's last prompt position.  Positions past a row's length are computed and discarded:
        attention is causal, so they never reach a valid position, and their KV slots are overwritten by the row's decode
        steps before any step reads them.  Only the B rows the caller needs go through the unembedding."""
        if ids.dim() != 2 or ids.dtype not in (torch.int32, torch.int64):
            raise TypeError("input ids must be (batch, length) int32/int64")
        self._ensure_packed()
        dev = self.embedding_layer.weight.device
        if ids.device != dev:
            raise _lib.EvoError(f"input ids on {ids.device}, model on {dev}")
        B, W = ids.shape
        lens = [int(n) for n in lengths]
        if len(lens) != B or (B and (min(lens) < 1 or max(lens) > W)):
            raise ValueError(f"lengths must be {B} values in [1, {W}], got {lens}")
        mha_ip, hy_ip = ipd["mha"], ipd["hyena"]
        if mha_ip.seqlen_offset or hy_ip.seqlen_offset or mha_ip.key_value_memory_dict or hy_ip.state_dict or hy_ip.fir_state_dict:
            raise _lib.EvoError("prefill_ragged needs fresh inference params (initialize_inference_params())")
        d, V = self.config.hidden_size, self.config.vocab_size
        x = ids.contiguous()
        with torch.cuda.device(dev), torch.no_grad():
            prev = self._loop_ragged
            if prev is not None:
                # the KV caches the ragged loop's captured step was recorded with: zeroed (what a fresh cache holds) and reused,
                # so a second call of the same shape replays that step instead of capturing a new one
                H = self.config.num_attention_heads
                want = (mha_ip.max_batch_size, mha_ip.max_seqlen, 2, H, d // H)
                with torch.inference_mode():
                    for i, c in prev["kv"].items():
                        if tuple(c.shape) == want:
                            mha_ip.key_value_memory_dict[i] = c.zero_()
            lens_dev = torch.tensor(lens, dtype=torch.int32, device=dev)
            u = self._backbone(x, B, W, ipd, lengths=lens_dev)
            last = torch.tensor([b * W + n - 1 for b, n in enumerate(lens)], dtype=torch.int64, device=dev)
            rows = torch.empty(B, d, dtype=torch.bfloat16, device=dev)
            check(_lib.lib().evo_embed(ptr(last), 1, ptr(u), ptr(rows), B, d, B * W, self._stream()), "evo_embed")   # row gather
            logits = torch.empty(B, V, dtype=torch.bfloat16, device=dev)
            self._gemm(rows, self.unembed.weight, logits, B, V, d, EPI_NONE)
        return logits

    def score_tokens(self, input_ids, want_logprobs=True, want_entropy=False):
        """Fused scoring head (SURVEY 8f-1): what evo/scoring.py computes from `model(input_ids)` -- log_softmax of the
        logits gathered at the NEXT token (logits_to_logprobs, :36-59) and the per-position entropy (:119-121) -- without
        the (B, L, 512) logits ever reaching HBM: the unembed GEMM's epilogue keeps max / sum-exp / sum-exp*logit / target
        logit per row (evo_unembed_score).  Returns (logprobs (B, L) fp32 or None, entropy (B, L) fp32 or None);
        logprobs[b, t] = log p(ids[b, t+1] | ids[b, :t+1]), 0 at the last position."""
        if input_ids.dim() != 2 or input_ids.dtype not in (torch.int32, torch.int64):
            raise TypeError("input ids must be (batch, length) int32/int64")
        self._ensure_packed()
        dev = self.embedding_layer.weight.device
        if input_ids.device != dev:
            raise _lib.EvoError(f"input ids on {input_ids.device}, model on {dev}")
        x = input_ids.contiguous()
        B, L = x.shape
        M, d, V = B * L, self.config.hidden_size, self.config.vocab_size
        lib = _lib.lib()
        with torch.cuda.device(dev), torch.no_grad():
            u = self._backbone(x, B, L, None)
            targets = torch.full((B, L), -1, dtype=torch.long, device=dev)
            targets[:, :-1] = x[:, 1:]
            lp = torch.empty(B, L, dtype=torch.float32, device=dev) if want_logprobs else None
            ent = torch.empty(B, L, dtype=torch.float32, device=dev) if want_entropy else None
            n = lib.evo_unembed_score_workspace(M, V)
            ws = torch.empty(max(n, 1), dtype=torch.uint8, device=dev)
            sp = _lib.ScoreParams(x=u.data_ptr(), W=self.unembed.weight.data_ptr(), targets=targets.data_ptr(), logprobs=lp.data_ptr() if lp is not None else None,
                                  entropy=ent.data_ptr() if ent is not None else None, M=M, V=V, K=d, workspace=ws.data_ptr(), workspace_bytes=n)
            self._record(f"gemm/{V}x{d}/score", 2.0 * M * V * d, lambda: check(lib.evo_unembed_score(C.byref(sp), self._stream()), "evo_unembed_score"))
        return lp, ent

    # ---- decode step: small-M weight-streaming GEMM tiles + device-side position + CUDA graph ------
    def _can_step(self, ipd, B):
        mha, hy = ipd["mha"], ipd["hyena"]
        for i in range(len(self.blocks)):
            if i in self._attn_idxs:
                c = mha.key_value_memory_dict.get(i)
                if c is None or c.shape[0] < B:
                    return False
            elif i not in hy.fir_state_dict or i not in hy.state_dict:
                return False
        return True

    @staticmethod
    def _tile64(w):
        """(N, K) row-major -> (N/64, K/64, 64, 64): each 64x64 tile is one contiguous 8 KB block, so the decode GEMM's TMA
        boxes use every DRAM page they open (row-major tiles touch 64 pages for 128 bytes each: measured 2.2-3.5 TB/s)."""
        n, k = w.shape
        return w.view(n // 64, 64, k // 64, 64).permute(0, 2, 1, 3).contiguous()

    def _ensure_tiled(self):
        if self._tiled is not None:
            return self._tiled
        t = {}
        with torch.no_grad():
            for i, blk in enumerate(self.blocks):
                pk = self._packed[i]
                e = {"w12": self._tile64(pk["w12"]), "w3": self._tile64(pk["w3"])}
                if i in self._attn_idxs:
                    e["in"], e["out"] = self._tile64(blk.inner_mha_cls.Wqkv.weight.data), self._tile64(blk.inner_mha_cls.out_proj.weight.data)
                else:
                    e["in"], e["out"] = self._tile64(blk.projections.weight.data), self._tile64(blk.out_filter_dense.weight.data)
                t[i] = e
            t["unembed"] = self._tile64(self.unembed.weight.data)
        self._tiled = t
        return t

    def _decode_body(self, x, pos_dev, ipd, B, rows=False):
        """One token per sequence through all blocks; every launch reads the position from pos_dev.
        rows: pos_dev is a (B) vector, one position per row (the *_rows attention kernels); else one (1) position."""
        lib = _lib.lib()
        prev = lib.evo_set_pdl(int(self.decode_pdl))
        try:
            return self._decode_body_impl(x, pos_dev, ipd, B, rows)
        finally:
            lib.evo_set_pdl(prev)

    def _decode_body_impl(self, x, pos_dev, ipd, B, rows=False):
        cfg = self.config
        d, H, V = cfg.hidden_size, cfg.num_attention_heads, cfg.vocab_size
        hd = d // H
        dev = x.device
        lib = _lib.lib()
        mha_ip, hy_ip = ipd["mha"], ipd["hyena"]
        streamk = self.decode_streamk and B <= 64
        tiled = self._ensure_tiled() if (self.decode_tiled and not streamk) else None
        G2 = 3 if tiled is not None else 2       # weight-streaming tiles (3: tile-major weights)
        wsel = (lambda i, name, w: tiled[i][name]) if tiled is not None else (lambda i, name, w: w)

        def lin(a, w, out, N, K, epi, bias=None, resid=None):
            if streamk:
                self._gemm_smallm(a, w, out, B, N, K, epi, bias=bias, resid=resid)
            else:
                self._gemm(a, w, out, B, N, K, epi, bias=bias, resid=resid, variant=G2)

        qkv_prep, attn = (lib.evo_decode_qkv_prep_rows, lib.evo_decode_attn_rows) if rows else (lib.evo_decode_qkv_prep, lib.evo_decode_attn)
        u = torch.empty(B, d, dtype=torch.bfloat16, device=dev)
        check(lib.evo_embed(ptr(x), int(x.dtype == torch.int64), ptr(self.embedding_layer.weight), ptr(u), B, d, V, self._stream()), "evo_embed")
        nsplit = max(1, min(16, -(-8 * torch.cuda.get_device_properties(dev).multi_processor_count // (H * B))))   # >= ~4 waves of 2 CTAs/SM
        for i, blk in enumerate(self.blocks):
            xn = torch.empty_like(u)
            self._rmsnorm(u, blk.pre_norm.scale, xn, B)
            u2 = torch.empty_like(u)
            if i in self._attn_idxs:
                mha = blk.inner_mha_cls
                qkv = torch.empty(B, 3 * d, dtype=torch.bfloat16, device=dev)
                lin(xn, wsel(i, "in", mha.Wqkv.weight), qkv, 3 * d, d, EPI_BIAS if mha.Wqkv.bias is not None else EPI_NONE, bias=mha.Wqkv.bias)
                cache = mha_ip.key_value_memory_dict[i]
                cos, sin = self._rope_tables(cache.shape[1], dev)
                check(qkv_prep(ptr(qkv), ptr(cache), ptr(cos), ptr(sin), ptr(pos_dev), B, H, hd, cache.shape[1], self._stream()), "evo_decode_qkv_prep")
                nws = lib.evo_decode_attn_workspace(B, H, nsplit)
                ws = torch.empty(nws, dtype=torch.uint8, device=dev)
                ctx = xn
                check(attn(ptr(qkv), ptr(cache), ptr(ctx), ptr(pos_dev), B, H, hd, cache.shape[1], nsplit,
                                          1.0 / math.sqrt(hd), ptr(ws), nws, self._stream()), "evo_decode_attn")
                lin(ctx, wsel(i, "out", mha.out_proj.weight), u2, d, d, EPI_BIAS_RESID if mha.out_proj.bias is not None else EPI_RESID,
                    bias=mha.out_proj.bias, resid=u)
            else:
                f = blk.filter
                if streamk and self.decode_fused_step and hd == 128:
                    # in-projection with engine.step_fir + step_iir in its epilogue: z never leaves the SM, one launch less per layer
                    y = torch.empty(B, d, dtype=torch.bfloat16, device=dev)
                    self._gemm_smallm(xn, blk.projections.weight, y, B, 3 * d, d, EPI_HYENA_STEP, bias=blk.projections.bias,
                                      step=(hy_ip.fir_state_dict[i], torch.view_as_real(hy_ip.state_dict[i]), f))
                else:
                    z = torch.empty(B, 3 * d, dtype=torch.bfloat16, device=dev)
                    lin(xn, wsel(i, "in", blk.projections.weight), z, 3 * d, d, EPI_BIAS, bias=blk.projections.bias)
                    y = xn
                    check(lib.evo_hyena_step(ptr(z), ptr(y), ptr(hy_ip.fir_state_dict[i]), ptr(torch.view_as_real(hy_ip.state_dict[i])),
                                             ptr(f.short_filter_weight), ptr(f.short_filter_bias), ptr(f.D), ptr(f.poles), ptr(f.residues),
                                             B, d, cfg.state_size, H, self._stream()), "evo_hyena_step")
                lin(y, wsel(i, "out", blk.out_filter_dense.weight), u2, d, d, EPI_BIAS_RESID, bias=blk.out_filter_dense.bias, resid=u)
            pk = self._packed[i]
            xn2 = xn
            self._rmsnorm(u2, blk.post_norm.scale, xn2, B)
            g = torch.empty(B, pk["ipad"], dtype=torch.bfloat16, device=dev)
            if streamk:
                self._gemm_smallm(xn2, pk["w12"], g, B, 2 * pk["ipad"], d, EPI_GELU_GATE)
            else:
                t = torch.empty(B, 2 * pk["ipad"], dtype=torch.bfloat16, device=dev)
                self._gemm(xn2, wsel(i, "w12", pk["w12"]), t, B, 2 * pk["ipad"], d, EPI_NONE, variant=G2)
                check(lib.evo_gelu_gate_interleaved(ptr(t), ptr(g), B, pk["ipad"], self._stream()), "evo_gelu_gate_interleaved")
            u = torch.empty_like(u2)
            lin(g, wsel(i, "w3", pk["w3"]), u, d, pk["ipad"], EPI_RESID, resid=u2)
        if self.norm is not None:
            xn = torch.empty_like(u)
            self._rmsnorm(u, self.norm.scale, xn, B)
            u = xn
        logits = torch.empty(B, V, dtype=torch.bfloat16, device=dev)
        lin(u, tiled["unembed"] if tiled is not None else self.unembed.weight, logits, V, d, EPI_NONE)
        return logits

    # ---- on-device generation loop (SURVEY 8f-2): token pick + bookkeeping + feedback inside the captured step ------
    def decode_loop(self, first_token, ipd, n_steps, start_pos, *, top_k=1, top_p=0.0, temperature=1.0, forced=None, n_out=None, seed=None):
        """Run `n_steps` single-token steps without returning to the host in between.

        first_token (B,) or (B, 1): the input of step 0; ipd: populated state (after a prefill); start_pos: sequence
        position of step 0 (the reference sets the FULL prompt length here, evo/generation.py:143).  Step i feeds the
        token of step i-1; the token of step i is forced[:, i] while i < forced.shape[1] (teacher-forced prompt tail,
        evo/generation.py:156-160), afterwards it is picked on the device by evo_sample_step.
        Returns (picked (B, n_out) int64, kept_logits (B, n_out, V) fp32) for the sampled steps; the state holders'
        seqlen_offset end at the value the per-token protocol would leave.
        One CUDA graph = one whole step (all blocks + sampler + counters); the host only replays it."""
        lib = _lib.lib()
        dev = self.embedding_layer.weight.device
        x = first_token.reshape(-1, 1).contiguous()
        B = x.shape[0]
        V = self.config.vocab_size
        if not self._can_step(ipd, B):
            raise _lib.EvoError("decode_loop needs populated inference params (run the prefill first)")
        mha_ip, hy_ip = ipd["mha"], ipd["hyena"]
        n_forced = 0 if forced is None else int(forced.shape[1])
        n_out = n_steps - n_forced if n_out is None else n_out
        if n_out < 0:
            raise ValueError("more forced tokens than steps")
        for i in mha_ip.key_value_memory_dict:
            if start_pos + n_steps > mha_ip.key_value_memory_dict[i].shape[1]:
                raise _lib.EvoError(f"sequence length {start_pos + n_steps} exceeds the KV cache ({mha_ip.key_value_memory_dict[i].shape[1]}) (mha.py:367)")
        with torch.cuda.device(dev), torch.no_grad():
            self._ensure_packed()
            for i in list(hy_ip.state_dict):
                hy_ip.state_dict[i] = hy_ip.state_dict[i].contiguous()
                hy_ip.fir_state_dict[i] = hy_ip.fir_state_dict[i].contiguous()
            picked = torch.empty(B, max(n_out, 1), dtype=torch.long, device=dev)
            kept = torch.empty(B, max(n_out, 1), V, dtype=torch.float32, device=dev)
            forced_c = forced.to(dev, torch.long).contiguous() if n_forced else None
            if seed is None:
                seed = int(torch.randint(0, 2 ** 62, (1,)).item())          # torch.manual_seed() governs reproducibility
            lp = _lib.LoopParams(forced=forced_c.data_ptr() if n_forced else None, n_forced=n_forced, forced_stride=n_forced,
                                 picked=picked.data_ptr(), picked_stride=picked.shape[1], kept_logits=kept.data_ptr(), n_out=n_out,
                                 top_k=int(top_k), top_p=float(top_p), temperature=float(temperature), seed=seed, step0=0)
            key = ("loop", B, tuple(hy_ip.state_dict[i].data_ptr() for i in sorted(hy_ip.state_dict)),
                   tuple(hy_ip.fir_state_dict[i].data_ptr() for i in sorted(hy_ip.fir_state_dict)),
                   tuple((mha_ip.key_value_memory_dict[i].data_ptr(), mha_ip.key_value_memory_dict[i].shape[1]) for i in sorted(mha_ip.key_value_memory_dict)))
            st = self._loop
            if st is None or st["key"] != key:
                st = {"key": key, "graph": None, "x": torch.empty(B, 1, dtype=torch.long, device=dev), "pos": torch.zeros(1, dtype=torch.int64, device=dev),
                      "step": torch.zeros(1, dtype=torch.int64, device=dev), "lp": torch.zeros(C.sizeof(_lib.LoopParams), dtype=torch.uint8, device=dev),
                      "lp_host": torch.zeros(C.sizeof(_lib.LoopParams), dtype=torch.uint8).pin_memory()}
                self._loop = st
            if st.get("lp_copied") is not None:
                st["lp_copied"].synchronize()       # a previous call's async copy may not have left the pinned staging buffer yet
            C.memmove(st["lp_host"].data_ptr(), C.addressof(lp), C.sizeof(lp))
            st["lp"].copy_(st["lp_host"], non_blocking=True)
            st["lp_copied"] = torch.cuda.Event()
            st["lp_copied"].record()
            st["pos"].fill_(int(start_pos))
            st["step"].zero_()
            st["x"].copy_(x.to(torch.long))

            def one_step():
                logits = self._decode_body(st["x"], st["pos"], ipd, B)
                prev = lib.evo_set_pdl(int(self.decode_pdl))
                try:
                    check(lib.evo_sample_step(ptr(logits), ptr(st["x"]), B, V, ptr(st["lp"]), ptr(st["step"]), self._stream()), "evo_sample_step")
                    check(lib.evo_advance_counters(ptr(st["pos"]), ptr(st["step"]), 1, self._stream()), "evo_advance_counters")
                finally:
                    lib.evo_set_pdl(prev)

            done = 0
            if st["graph"] is None or st.get("ptrs") != self._graph_ptrs():
                one_step()                      # eager step: allocates rope tables / workspaces the capture must not
                done = 1
                if self.decode_graph and n_steps > 1:
                    g = torch.cuda.CUDAGraph()
                    torch.cuda.synchronize()
                    n0 = lib.evo_launch_count()
                    with torch.cuda.graph(g):
                        one_step()
                    st["graph"], st["launches"], st["ptrs"] = g, lib.evo_launch_count() - n0, self._graph_ptrs()
                    lib.evo_note_graph_replay(-st["launches"])
            for _ in range(done, n_steps):
                if st["graph"] is not None:
                    st["graph"].replay()
                    lib.evo_note_graph_replay(st["launches"])
                else:
                    one_step()
            end = int(start_pos) + n_steps - 1          # the position the last step ran at (what the per-token protocol leaves)
            mha_ip.seqlen_offset = hy_ip.seqlen_offset = end
            # the captured graph and its buffers stay alive in self._loop; the outputs are this call's own tensors
            return picked[:, :n_out], kept[:, :n_out]

    def decode_loop_ragged(self, first_token, ipd, start, n_forced, n_out, *, forced=None, out_cols=None, top_k=1, top_p=0.0,
                           temperature=1.0, seed=None):
        """decode_loop for rows that sit at different positions (prompts of different lengths, after prefill_ragged).

        Row b starts at position start[b], feeds first_token[b] at step 0, is teacher-forced with forced[b, :n_forced[b]],
        then samples n_out[b] tokens; it runs n_forced[b] + n_out[b] steps and then stands still (keeps its position,
        records nothing) while the longer rows finish.  Returns (picked (B, out_cols) int64, kept_logits (B, out_cols, V)
        fp32): row b's tokens fill its LAST n_out[b] columns; columns before those are not written.
        One CUDA graph per step, like decode_loop, with its own graph cache.  The cache keeps the state tensors the step was
        captured with (the KV caches included) until the model is moved or reloaded; prefill_ragged and the next call of the
        same shape reuse them, so that call replays the captured step.  The state holders' seqlen_offset are left as they
        are: the rows end at different positions, so the state is not resumable through them."""
        lib = _lib.lib()
        dev = self.embedding_layer.weight.device
        x = first_token.reshape(-1, 1).contiguous()
        B = x.shape[0]
        V = self.config.vocab_size
        start, n_forced, n_out = ([int(v) for v in a] for a in (start, n_forced, n_out))
        if not (len(start) == len(n_forced) == len(n_out) == B):
            raise ValueError("start, n_forced and n_out need one entry per row")
        if B > 64:
            raise _lib.EvoError(f"decode_loop_ragged: batch {B} > 64 (the stream-K decode GEMM's limit)")
        if min(n_forced + n_out) < 0:
            raise ValueError("negative step counts")
        out_cols = max(n_out) if out_cols is None else int(out_cols)
        if max(n_out) > out_cols:
            raise ValueError("n_out exceeds out_cols")
        F = max(n_forced)
        if F and (forced is None or forced.shape[0] != B or forced.shape[1] < F):
            raise ValueError(f"forced must be (B, >= {F})")
        if not self._can_step(ipd, B):
            raise _lib.EvoError("decode_loop_ragged needs populated inference params (run prefill_ragged first)")
        mha_ip, hy_ip = ipd["mha"], ipd["hyena"]
        steps = [f + o for f, o in zip(n_forced, n_out)]
        for i in mha_ip.key_value_memory_dict:
            cap = mha_ip.key_value_memory_dict[i].shape[1]
            for b in range(B):
                if start[b] + steps[b] > cap:
                    raise _lib.EvoError(f"row {b}: sequence length {start[b] + steps[b]} exceeds the KV cache ({cap}) (mha.py:367)")
        n_steps = max(steps)
        with torch.cuda.device(dev), torch.no_grad():
            picked = torch.empty(B, max(out_cols, 1), dtype=torch.long, device=dev)
            kept = torch.empty(B, max(out_cols, 1), V, dtype=torch.float32, device=dev)
            if n_steps == 0:
                return picked[:, :out_cols], kept[:, :out_cols]
            self._ensure_packed()
            for i in list(hy_ip.state_dict):
                hy_ip.state_dict[i] = hy_ip.state_dict[i].contiguous()
                hy_ip.fir_state_dict[i] = hy_ip.fir_state_dict[i].contiguous()
            prev = self._loop_ragged
            if prev is not None:
                # move the Hyena states into the tensors the captured step was recorded with (a few MB per layer)
                # (inference mode: the held tensors were made by a prefill under torch.inference_mode, as generate() runs it)
                with torch.inference_mode():
                    for store, held in ((hy_ip.state_dict, prev["hy"]), (hy_ip.fir_state_dict, prev["fir"])):
                        for i, t in held.items():
                            if i in store and store[i].shape == t.shape and store[i].dtype == t.dtype and store[i].data_ptr() != t.data_ptr():
                                store[i] = t.copy_(store[i])
            per_row = torch.tensor([n_forced, n_out, start], dtype=torch.int64, device=dev)
            forced_c = forced[:, :F].to(dev, torch.long).contiguous() if F else None
            if seed is None:
                seed = int(torch.randint(0, 2 ** 62, (1,)).item())          # torch.manual_seed() governs reproducibility
            lp = _lib.RaggedLoopParams(n_forced=per_row[0].data_ptr(), n_out=per_row[1].data_ptr(), start=per_row[2].data_ptr(),
                                       forced=forced_c.data_ptr() if F else None, forced_stride=F,
                                       picked=picked.data_ptr(), kept_logits=kept.data_ptr(), out_cols=picked.shape[1],
                                       top_k=int(top_k), top_p=float(top_p), temperature=float(temperature), seed=seed)
            key = ("ragged", B, tuple(hy_ip.state_dict[i].data_ptr() for i in sorted(hy_ip.state_dict)),
                   tuple(hy_ip.fir_state_dict[i].data_ptr() for i in sorted(hy_ip.fir_state_dict)),
                   tuple((mha_ip.key_value_memory_dict[i].data_ptr(), mha_ip.key_value_memory_dict[i].shape[1]) for i in sorted(mha_ip.key_value_memory_dict)))
            st = self._loop_ragged
            if st is None or st["key"] != key:
                st = {"key": key, "graph": None, "x": torch.empty(B, 1, dtype=torch.long, device=dev), "pos": torch.zeros(B, dtype=torch.int64, device=dev),
                      "step": torch.zeros(1, dtype=torch.int64, device=dev), "lp": torch.zeros(C.sizeof(_lib.RaggedLoopParams), dtype=torch.uint8, device=dev),
                      "lp_host": torch.zeros(C.sizeof(_lib.RaggedLoopParams), dtype=torch.uint8).pin_memory(),
                      # the state tensors the step is captured with stay alive here, so the next call can reuse them
                      "hy": dict(hy_ip.state_dict), "fir": dict(hy_ip.fir_state_dict), "kv": dict(mha_ip.key_value_memory_dict)}
                self._loop_ragged = st
            if st.get("lp_copied") is not None:
                st["lp_copied"].synchronize()       # a previous call's async copy may not have left the pinned staging buffer yet
            C.memmove(st["lp_host"].data_ptr(), C.addressof(lp), C.sizeof(lp))
            st["lp"].copy_(st["lp_host"], non_blocking=True)
            st["lp_copied"] = torch.cuda.Event()
            st["lp_copied"].record()
            st["pos"].copy_(per_row[2])
            st["step"].zero_()
            st["x"].copy_(x.to(torch.long))

            def one_step():
                logits = self._decode_body(st["x"], st["pos"], ipd, B, rows=True)
                prev = lib.evo_set_pdl(int(self.decode_pdl))
                try:
                    check(lib.evo_sample_step_rows(ptr(logits), ptr(st["x"]), B, V, ptr(st["lp"]), ptr(st["step"]), self._stream()), "evo_sample_step_rows")
                    check(lib.evo_ragged_advance(ptr(st["pos"]), ptr(st["step"]), ptr(st["lp"]), B, self._stream()), "evo_ragged_advance")
                finally:
                    lib.evo_set_pdl(prev)

            done = 0
            if st["graph"] is None or st.get("ptrs") != self._graph_ptrs():
                one_step()                      # eager step: allocates rope tables / workspaces the capture must not
                done = 1
                if self.decode_graph and n_steps > 1:
                    g = torch.cuda.CUDAGraph()
                    torch.cuda.synchronize()
                    n0 = lib.evo_launch_count()
                    with torch.cuda.graph(g):
                        one_step()
                    st["graph"], st["launches"], st["ptrs"] = g, lib.evo_launch_count() - n0, self._graph_ptrs()
                    lib.evo_note_graph_replay(-st["launches"])
            for _ in range(done, n_steps):
                if st["graph"] is not None:
                    st["graph"].replay()
                    lib.evo_note_graph_replay(st["launches"])
                else:
                    one_step()
            return picked[:, :out_cols], kept[:, :out_cols]

    def _graph_ptrs(self):
        """Addresses a captured step bakes in besides the state tensors: rope tables and the stream-K workspace."""
        return (tuple(t.data_ptr() for t in (self._rope or ())), self._smallm_ws.data_ptr() if self._smallm_ws is not None else 0)

    def _decode_forward(self, x, ipd):
        """L == 1 with populated states.  Step 1 after a prefill runs eagerly (and makes the state
        tensors contiguous / resident); step 2 captures the whole step into a CUDA graph; later
        steps replay it: one host call per token instead of ~15 launches per block."""
        mha_ip, hy_ip = ipd["mha"], ipd["hyena"]
        dev = x.device
        B = x.shape[0]
        for i in list(hy_ip.state_dict):
            if not hy_ip.state_dict[i].is_contiguous():
                hy_ip.state_dict[i] = hy_ip.state_dict[i].contiguous()
            if not hy_ip.fir_state_dict[i].is_contiguous():
                hy_ip.fir_state_dict[i] = hy_ip.fir_state_dict[i].contiguous()
        key = (B, x.dtype, tuple(hy_ip.state_dict[i].data_ptr() for i in sorted(hy_ip.state_dict)),
               tuple(hy_ip.fir_state_dict[i].data_ptr() for i in sorted(hy_ip.fir_state_dict)),
               tuple((mha_ip.key_value_memory_dict[i].data_ptr(), mha_ip.key_value_memory_dict[i].shape[1]) for i in sorted(mha_ip.key_value_memory_dict)),
               # every other address the captured launches bake in: rope tables, stream-K workspace
               tuple(t.data_ptr() for t in (self._rope or ())), self._smallm_ws.data_ptr() if self._smallm_ws is not None else 0)
        off = int(mha_ip.seqlen_offset)
        for i in mha_ip.key_value_memory_dict:
            if off >= mha_ip.key_value_memory_dict[i].shape[1]:
                raise _lib.EvoError(f"sequence length {off + 1} exceeds the KV cache ({mha_ip.key_value_memory_dict[i].shape[1]}) (mha.py:367)")
        st = self._decode
        if st is None or st["key"] != key:
            st = {"key": key, "graph": None, "x": torch.empty_like(x), "pos": torch.zeros(1, dtype=torch.int64, device=dev), "logits": None, "steps": 0}
            self._decode = st
        st["pos"].fill_(off)
        st["x"].copy_(x)
        if not self.decode_graph or self._prof is not None or st["steps"] == 0:
            st["steps"] += 1
            return self._decode_body(st["x"], st["pos"], ipd, B).view(B, 1, -1)
        if st["graph"] is None:
            g = torch.cuda.CUDAGraph()
            torch.cuda.synchronize()
            n0 = _lib.lib().evo_launch_count()
            with torch.cuda.graph(g):
                st["logits"] = self._decode_body(st["x"], st["pos"], ipd, B)
            st["graph"] = g
            st["launches"] = _lib.lib().evo_launch_count() - n0      # counted while capturing, when nothing ran: undo, then count per replay
            _lib.lib().evo_note_graph_replay(-st["launches"])
        st["graph"].replay()
        _lib.lib().evo_note_graph_replay(st["launches"])
        st["steps"] += 1
        return st["logits"].clone().view(B, 1, -1)
