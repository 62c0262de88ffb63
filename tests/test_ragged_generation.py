"""Batched generation of prompts of different lengths (generate(..., ragged=True)), the parts that need no GPU:
  * ragged_schedule -- the per-row bookkeeping shared by the one-prompt device loop and the ragged loop -- reproduces,
    prompt by prompt, the model calls the reference's own generation code made (tests/golden/reference_host.json):
    the prefill slice length, then the seqlen_offset of every single-token step, Q1's jump to the full prompt included;
  * where the ragged path does not apply (a model without the device loop: here the CPU oracle) generate(ragged=True)
    is generate() exactly: texts, scores, calls;
  * every new C entry point rejects bad arguments with a negative code and a reason in evo_last_error(), before launching."""
import ctypes
import json
import math
import os
import sys
import warnings

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import evo_b200                                                     # noqa: E402
from evo_b200 import CharLevelTokenizer, _lib                       # noqa: E402
from evo_b200.generation import ragged_schedule                     # noqa: E402
from oracle import stripedhyena_oracle as O                         # noqa: E402


@pytest.fixture(scope="module")
def gen_cases(golden_dir):
    with open(os.path.join(golden_dir, "reference_host.json")) as f:
        return json.load(f)["generation"]


def split_calls(calls):
    """[[shape, mha_offset, hyena_offset], ...] -> one (batch, prefill length, [step offsets]) per prefill."""
    groups = []
    for shape, off, off_h in calls:
        assert off == off_h
        if off == 0:
            groups.append((shape[0], shape[1], []))
        else:
            assert shape[1] == 1
            groups[-1][2].append(off)
    return groups


def trace(s):
    return s.prefill, [s.start + i for i in range(s.steps)]


@pytest.mark.parametrize("case", ["ragged_cached", "prompt_forcing_q1", "batched_cached", "one_token"])
def test_schedule_reproduces_the_reference_call_trace(gen_cases, case):
    want = gen_cases[case]
    kw = want["kwargs"]
    plan = ragged_schedule([len(p) for p in want["prompts"]], kw.get("force_prompt_threshold", 128), kw["n_tokens"])
    groups = split_calls(want["calls"])
    rows = []                                    # the reference's trace of each prompt (a batch of B shares one trace)
    for batch, prefill, steps in groups:
        rows += [(prefill, steps)] * batch
    assert len(rows) == len(plan)
    for s, (prefill, steps) in zip(plan, rows):
        assert trace(s) == (prefill, steps)
        assert s.steps == s.n_forced + s.n_out
        first = 0 if s.start > s.prefill else 1   # the prefill's logits give token 0 unless a tail is forced
        assert first + s.n_out == kw["n_tokens"]


def test_schedule_of_the_issue_example():
    s = ragged_schedule([8], 3, 5)[0]            # prompt_forcing_q1: prefill 3, steps at positions 8..16
    assert (s.prefill, s.start, s.n_forced, s.n_out, s.steps) == (3, 8, 4, 5, 9)
    assert trace(s) == (3, list(range(8, 17)))
    # a tail of one token: nothing forced inside the loop, all n_tokens sampled there
    assert ragged_schedule([4], 3, 2)[0] == (3, 4, 0, 2, 2)
    # no tail: the first token comes from the prefill
    assert ragged_schedule([1, 5], 128, 1) == [(1, 1, 0, 0, 0), (5, 5, 0, 0, 0)]


class OracleAsModel:
    """The fixture's model (seed 7, 3 layers, attention at layer 1) behind the model protocol, logging every call."""

    def __init__(self):
        cfg = O.tiny_config(num_layers=3, attn_layer_idxs=(1,), hidden_size=256, num_heads=2)
        cfg["max_seqlen"] = 128
        self.m = O.OracleStripedHyena(cfg, O.random_state_dict(cfg, seed=7), torch.float64)
        self.calls = []

    def eval(self):
        return self

    def initialize_inference_params(self):
        return self.m.initialize_inference_params()

    def __call__(self, x, inference_params_dict=None):
        d = inference_params_dict
        self.calls.append([list(x.shape), None if d is None else int(d["mha"].seqlen_offset), None if d is None else int(d["hyena"].seqlen_offset)])
        return self.m(x, d)


@pytest.mark.parametrize("case", ["ragged_cached", "prompt_forcing_q1", "batched_cached", "one_token", "unbatched_by_request"])
def test_ragged_flag_changes_nothing_without_the_device_loop(gen_cases, case, capsys):
    want = gen_cases[case]
    outs = []
    for ragged in (False, True):
        model = OracleAsModel()
        with np.errstate(all="ignore"), warnings.catch_warnings():
            warnings.simplefilter("ignore")                                  # n_tokens=1: mean of an empty slice
            texts, scores = evo_b200.generate(want["prompts"], model, CharLevelTokenizer(512), top_k=1, verbose=1, device="cpu",
                                              ragged=ragged, **want["kwargs"])
        outs.append((texts, scores, model.calls, capsys.readouterr()))
    (t0, s0, c0, io0), (t1, s1, c1, io1) = outs
    assert t1 == t0 == want["texts"] and c1 == c0 == want["calls"]
    assert all((math.isnan(a) and math.isnan(b)) or a == b for a, b in zip(s0, s1))
    assert (io1.out, io1.err) == (io0.out, io0.err)                           # the notes included


def test_ragged_loop_checks_the_kv_cache_per_row_before_launching():
    """A row whose start + steps passes the KV cache raises EvoError; nothing reaches the device (the model is on the CPU)."""
    from evo_b200.stripedhyena import StripedHyena, dotdict
    from evo_b200.stripedhyena.cache import InferenceParams, RecurrentInferenceParams
    cfg = O.tiny_config(num_layers=2, attn_layer_idxs=(1,), hidden_size=256, num_heads=2)
    m = StripedHyena(dotdict(cfg))
    ipd = {"mha": InferenceParams(max_seqlen=16, max_batch_size=2, seqlen_offset=0),
           "hyena": RecurrentInferenceParams(fir_filter_length=3, state_dim=8, seqlen_offset=0)}
    ipd["mha"].key_value_memory_dict[1] = torch.zeros(2, 16, 2, 2, 128, dtype=torch.bfloat16)
    ipd["hyena"].state_dict[0] = torch.zeros(2, 256, 8, dtype=torch.complex64)
    ipd["hyena"].fir_state_dict[0] = torch.zeros(2, 768, 2, dtype=torch.bfloat16)
    first = torch.zeros(2, dtype=torch.long)
    with pytest.raises(_lib.EvoError, match=r"row 1: sequence length 17 exceeds the KV cache \(16\)"):
        m.decode_loop_ragged(first, ipd, start=[3, 12], n_forced=[0, 0], n_out=[4, 5])
    with pytest.raises(_lib.EvoError, match="batch 65 > 64"):
        m.decode_loop_ragged(torch.zeros(65, dtype=torch.long), ipd, start=[1] * 65, n_forced=[0] * 65, n_out=[1] * 65)
    with pytest.raises(ValueError, match="forced must be"):
        m.decode_loop_ragged(first, ipd, start=[3, 4], n_forced=[2, 0], n_out=[1, 1])


def test_new_entry_points_reject_bad_arguments_without_a_gpu():
    lib = _lib.lib()
    p = ctypes.c_void_p

    def err():
        return lib.evo_last_error().decode()

    assert lib.evo_decode_qkv_prep_rows(p(0x1000), p(0x2000), p(0x3000), p(0x4000), p(0x5000), 2, 2, 64, 16, None) < 0
    assert "evo_decode_qkv_prep_rows: head_dim 64 unsupported" in err()
    assert lib.evo_decode_attn_rows(p(0x1000), p(0x2000), p(0x3000), p(0x4000), 2, 2, 96, 16, 1, 0.1, p(0x5000), 1 << 20, None) < 0
    assert "evo_decode_attn_rows: head_dim 96 unsupported" in err()
    assert lib.evo_decode_attn_rows(p(0x1000), p(0x2000), p(0x3000), p(0x4000), 2, 2, 128, 16, 0, 0.1, p(0x5000), 1 << 20, None) < 0
    assert "bad nsplit 0" in err()
    need = lib.evo_decode_attn_workspace(2, 2, 4)
    assert lib.evo_decode_attn_rows(p(0x1000), p(0x2000), p(0x3000), p(0x4000), 2, 2, 128, 16, 4, 0.1, p(0x5000), need - 1, None) < 0
    assert "evo_decode_attn_rows: workspace too small" in err()
    assert lib.evo_sample_step_rows(p(0x1000), p(0x2000), 2, 2000, p(0x3000), p(0x4000), None) < 0
    assert "evo_sample_step_rows: vocabulary 2000 unsupported" in err()
    assert lib.evo_ragged_advance(p(0x1000), p(0x2000), p(0x3000), 2000, None) < 0
    assert "evo_ragged_advance: batch 2000 unsupported" in err()
    assert lib.evo_ragged_advance(p(0x1000), p(0x2000), p(0x3000), 0, None) < 0

    hp = _lib.HyenaParams(z=0x1000, y=0x2000, fir_w=0x3000, fir_b=0x4000, Dskip=0x5000, poles=0x6000, residues=0x7000,
                          B=2, L=40, D=256, S=8, nheads=2)
    lengths = p(0x8000)
    assert lib.evo_hyena_fwd_ragged(ctypes.byref(hp), None, None, 0, None) < 0 and "lengths is NULL" in err()
    hp.halo = 0x9000
    assert lib.evo_hyena_fwd_ragged(ctypes.byref(hp), lengths, None, 0, None) < 0 and "halo / state_in" in err()
    hp.halo, hp.state_in = None, 0x9000
    assert lib.evo_hyena_fwd_ragged(ctypes.byref(hp), lengths, None, 0, None) < 0 and "halo / state_in" in err()
    hp.state_in, hp.nheads = None, 4                       # head_dim 64: not the mode-split scan
    assert lib.evo_hyena_fwd_ragged(ctypes.byref(hp), lengths, None, 0, None) < 0 and "mode-split" in err()
    hp.nheads, hp.S = 2, 4
    assert lib.evo_hyena_fwd_ragged(ctypes.byref(hp), lengths, None, 0, None) < 0 and "state_size 4 unsupported" in err()
    hp.S, hp.force_segments = 8, 4                         # a split scan needs its workspace
    assert lib.evo_hyena_fwd_ragged_workspace(ctypes.byref(hp)) == lib.evo_hyena_fwd_workspace(ctypes.byref(hp)) > 0
    assert lib.evo_hyena_fwd_ragged(ctypes.byref(hp), lengths, None, 0, None) < 0 and "workspace too small" in err()
