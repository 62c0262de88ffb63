"""evo_b200's host layer against outputs of the REFERENCE'S OWN host code (tests/golden/reference_host.{json,npz}).

The fixtures were produced by tests/golden/make_reference_host_golden.py: the reference's evo/{tokenizer,scoring,generation,
models}.py imported unmodified (with a stand-in for the absent `stripedhyena` package) and driven on CPU with the oracle model.
Here the same oracle model is put behind evo_b200's tokenizer / scoring / generation / checkpoint code: every id, every model
call (prompt slice and seqlen_offset), every generated string and every score must come out as the reference's did.
This pins the host side of the path (SURVEY.md 8b, 8f).  It does not pin the model arithmetic: the oracle is a restatement."""
import json
import math
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import evo_b200                                                     # noqa: E402
from evo_b200 import CharLevelTokenizer                             # noqa: E402
from evo_b200.generation import Generator                           # noqa: E402
from evo_b200.scoring import logits_to_logprobs, positional_entropies, prepare_batch, score_sequences  # noqa: E402
from oracle import stripedhyena_oracle as O                         # noqa: E402


@pytest.fixture(scope="module")
def ref(golden_dir):
    with open(os.path.join(golden_dir, "reference_host.json")) as f:
        doc = json.load(f)
    return doc, np.load(os.path.join(golden_dir, "reference_host.npz"))


class OracleAsModel:
    """Same wrapper as the generating script's: the oracle behind the model protocol, logging every call."""

    def __init__(self, dtype=torch.float64):
        cfg = O.tiny_config(num_layers=3, attn_layer_idxs=(1,), hidden_size=256, num_heads=2)
        cfg["max_seqlen"] = 128
        self.m = O.OracleStripedHyena(cfg, O.random_state_dict(cfg, seed=7), dtype)
        self.calls = []

    def eval(self):
        return self

    def initialize_inference_params(self):
        return self.m.initialize_inference_params()

    def __call__(self, x, inference_params_dict=None):
        d = inference_params_dict
        self.calls.append([list(x.shape), None if d is None else int(d["mha"].seqlen_offset), None if d is None else int(d["hyena"].seqlen_offset)])
        return self.m(x, d)


class RecordedBf16Model(OracleAsModel):
    """The bf16 oracle as the reference's scoring code saw it: the fixture's logits for the fixture's batch.  A bf16 matmul on
    CPU rounds differently with and without AMX, so recomputing them would tie the expected scores to the host CPU."""

    def __init__(self, arr):
        self.ids = torch.from_numpy(arr["prepare_batch_ids_bos1"])
        self.logits = torch.from_numpy(arr["score_logits_bf16"]).to(torch.bfloat16)
        self.calls = []

    def __call__(self, x, inference_params_dict=None):
        assert inference_params_dict is None and torch.equal(x, self.ids)
        self.calls.append([list(x.shape), None, None])
        return self.logits.clone(), None


def test_fixture_was_made_from_the_reference_modules(ref):
    doc, arr = ref
    assert sorted(doc["reference_modules"]) == ["evo.generation", "evo.models", "evo.scoring", "evo.tokenizer"]
    assert all(len(d) == 16 and int(d, 16) >= 0 for d in doc["reference_modules"].values())       # sha256 prefixes of the files run
    # the stored bf16 logits are this oracle's, up to the bf16 rounding a different CPU matmul path gives (<= 2 ulp at |x| < 16)
    live = OracleAsModel(torch.bfloat16)(torch.from_numpy(arr["prepare_batch_ids_bos1"]))[0].float()
    d = (live - torch.from_numpy(arr["score_logits_bf16"])).abs()
    assert d.max().item() <= 0.125 and d.mean().item() < 0.02, (d.max().item(), d.mean().item())


def test_tokenizer_matches_the_reference(ref):
    want = ref[0]["tokenizer"]
    tok = CharLevelTokenizer(512)
    assert [tok.vocab_size, tok.eod_id, tok.eos_id, tok.pad_id, tok.eod, tok.eos] == [want[k] for k in ("vocab_size", "eod_id", "eos_id", "pad_id", "eod", "eos")]
    for text, ids in want["tokenize"]:
        assert [int(i) for i in tok.tokenize(text)] == ids
    assert [[int(i) for i in row] for row in tok.tokenize_batch([t for t, _ in want["tokenize"][:3]])] == want["tokenize_batch"]
    for ids, text in want["detokenize"]:
        assert tok.detokenize(ids) == text
    assert tok.detokenize_batch([ids for ids, _ in want["detokenize"]]) == want["detokenize_batch_list"]
    assert tok.detokenize_batch(torch.tensor([[65, 67, 10, 3], [84, 84, 200, 511]])) == want["detokenize_batch_tensor"]
    assert [[n, tok.clamp(n)] for n, _ in want["clamp"]] == want["clamp"]


def test_prepare_batch_and_logits_to_logprobs_match_the_reference(ref):
    doc, arr = ref
    tok = CharLevelTokenizer(512)
    for bos in (True, False):
        ids, lengths = prepare_batch(doc["scoring"]["seqs"], tok, prepend_bos=bos, device="cpu")
        assert ids.dtype == torch.long and np.array_equal(ids.numpy(), arr[f"prepare_batch_ids_bos{int(bos)}"])
        assert list(lengths) == doc["scoring"][f"prepare_batch_lengths_bos{int(bos)}"]
    logits, ids = torch.from_numpy(arr["l2l_logits"]), torch.from_numpy(arr["l2l_ids"])
    for name, lg in (("fp32", logits), ("bf16", logits.to(torch.bfloat16))):
        for trim in (True, False):
            got = logits_to_logprobs(lg, ids, trim_bos=trim)
            assert got.dtype == lg.dtype                                         # Q4: the reduction runs in the logits' dtype
            assert np.array_equal(got.float().numpy(), arr[f"l2l_{name}_trim{int(trim)}"])


@pytest.mark.parametrize("name,dtype", [("fp64", torch.float64), ("bf16", torch.bfloat16)])
def test_scores_and_entropies_match_the_reference(ref, name, dtype):
    doc, arr = ref
    sc = doc["scoring"]
    tok = CharLevelTokenizer(512)
    make = (lambda: OracleAsModel(dtype)) if name == "fp64" else (lambda: RecordedBf16Model(arr))
    for red in ("mean", "sum"):
        model = make()
        got = score_sequences(sc["seqs"], model, tok, reduce_method=red, device="cpu")
        assert model.calls == sc[f"score_calls_{name}"]                          # ONE padded batch, no state
        assert np.allclose(np.asarray(got, dtype=np.float64), sc[f"score_{red}_{name}"], rtol=1e-6, atol=1e-6)
    ent = positional_entropies(sc["seqs"], make(), tok, device="cpu")
    assert [len(e) for e in ent] == [len(s) for s in sc["seqs"]]
    for k, e in enumerate(ent):
        # fp64: same arithmetic; bf16: the reference's softmax runs in bf16 (Q4), evo_b200's entropy in fp32 -- the documented improvement
        tol = 1e-5 if name == "fp64" else 0.06
        assert np.abs(np.asarray(e, dtype=np.float64) - arr[f"entropy_{name}_{k}"]).max() <= tol
    with pytest.raises(ValueError) as ex:
        score_sequences(sc["seqs"], make(), tok, reduce_method="median", device="cpu")
    assert str(ex.value) == sc["bad_reduce"]


@pytest.mark.parametrize("case", ["batched_cached", "ragged_cached", "unbatched_by_request", "prompt_forcing_q1", "prepend_bos", "one_token"])
def test_generate_matches_the_reference(ref, case):
    want = ref[0]["generation"][case]
    model = OracleAsModel()
    with np.errstate(all="ignore"):
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")                                      # n_tokens=1: mean of an empty slice, as in the reference
            texts, scores = evo_b200.generate(want["prompts"], model, CharLevelTokenizer(512), top_k=1, verbose=0, device="cpu", **want["kwargs"])
    assert texts == want["texts"]
    assert model.calls == want["calls"]                                          # prompt slices and seqlen_offsets, Q1's jump included
    for g, w in zip(scores, want["scores"]):
        assert (math.isnan(g) and math.isnan(w)) or abs(g - w) <= 1e-5 * max(1.0, abs(w))     # Q3's alignment is part of the number


@pytest.mark.parametrize("case", ["sampled_topk4", "sampled_topk50_topp", "sampled_full_vocab"])
def test_sampled_generation_matches_the_reference_under_the_same_seed(ref, case):
    """Not greedy: the reference's loop draws one torch.multinomial per step from the global generator (its `sample` here is
    flash_attn.utils.generation.sample, the function stripedhyena/sample.py copies); evo_b200's host loop and host sampler must
    consume the generator identically -- same seed, same strings, same scores."""
    want = ref[0]["generation"][case]
    model = OracleAsModel()
    torch.manual_seed(want["seed"])
    texts, scores = evo_b200.generate(want["prompts"], model, CharLevelTokenizer(512), verbose=0, device="cpu", **want["kwargs"])
    assert texts == want["texts"] and model.calls == want["calls"]
    assert np.allclose(scores, want["scores"], rtol=1e-5, atol=1e-5)


def test_uncached_generation_where_the_reference_raises(ref):
    """evo/generation.py:132 reads `prefilled`, which is only assigned when generation is cached or a state is passed in: the
    reference's generate(cached_generation=False) -- its default -- dies with UnboundLocalError before the first forward.
    evo_b200 runs the uncached loop (full forward per token); its greedy tokens equal the cached path's."""
    want = ref[0]["generation"]["batched_uncached"]
    assert want["raises"][0] == "UnboundLocalError" and want["calls"] == []
    model = OracleAsModel()
    texts, _ = evo_b200.generate(want["prompts"], model, CharLevelTokenizer(512), top_k=1, verbose=0, device="cpu", **want["kwargs"])
    cached = ref[0]["generation"]["batched_cached"]["texts"]
    n = want["kwargs"]["n_tokens"]
    assert texts == [t[:n] for t in cached]
    assert [c[0] for c in model.calls] == [[2, 8 + k] for k in range(n)] and all(c[1] is None for c in model.calls)


def test_generator_resume_protocol_matches_the_reference(ref):
    doc, arr = ref
    want = doc["generation"]["resume"]
    tok = CharLevelTokenizer(512)
    model = OracleAsModel()
    g = Generator(model, tok, top_k=1)
    ids, _ = prepare_batch(["ACGTACGT", "TTGACCAA"], tok, prepend_bos=False, device="cpu")
    new_ids, new_logits, state = g.generate(device="cpu", input_ids=ids, num_tokens=4, cached_generation=True, print_generation=False, stop_at_eos=False)
    assert np.array_equal(new_ids.numpy(), arr["gen_first_ids"]) and new_logits.dtype == torch.float32
    assert np.allclose(new_logits.numpy(), arr["gen_first_logits"], rtol=0, atol=1e-5)
    assert [int(state["mha"].seqlen_offset), int(state["hyena"].seqlen_offset)] == want["offsets_after_first"]
    more_ids, more_logits, state2 = g.generate(device="cpu", input_ids=new_ids[:, -1:], num_tokens=3, print_generation=False, stop_at_eos=False,
                                                inference_params_dict=state)
    assert (state2 is state) == want["same_state_object"]
    assert np.array_equal(more_ids.numpy(), arr["gen_resumed_ids"]) and np.allclose(more_logits.numpy(), arr["gen_resumed_logits"], rtol=0, atol=1e-5)
    assert model.calls == want["calls"]
    assert [int(state["mha"].seqlen_offset), int(state["hyena"].seqlen_offset)] == want["offsets_after_resume"]
    assert {"kv": sorted(state["mha"].key_value_memory_dict), "fir": sorted(state["hyena"].fir_state_dict), "iir": sorted(state["hyena"].state_dict)} == want["state_keys"]
    assert [int(state["mha"].max_batch_size), int(state["hyena"].max_batch_size)] == want["max_batch_size"]


def test_generator_input_string_and_max_seqlen_match_the_reference(ref):
    doc, arr = ref
    model = OracleAsModel()
    g = Generator(model, CharLevelTokenizer(512), top_k=1)
    ids, _, _ = g.generate(device="cpu", input_string="ACGTACGTTT", num_tokens=3, cached_generation=True, print_generation=False, stop_at_eos=False, max_seqlen=6)
    assert np.array_equal(ids.numpy(), arr["gen_string_ids"])
    assert model.calls == doc["generation"]["input_string_max_seqlen"]["calls"]         # window cropped to 6, offset set from the uncropped 10


def test_checkpoint_ingest_matches_the_reference(ref, tmp_path, monkeypatch):
    """Model name -> HF repo / revision / config, and what reaches the model from a two-shard snapshot with the HF 'backbone.'
    prefix and no unembed.weight, as the reference's Evo(...) / load_checkpoint did it (recorded through a stand-in model)."""
    import hashlib
    import huggingface_hub
    import yaml
    from safetensors.torch import save_file
    from evo_b200.configs import MODEL_NAMES, get_config
    from evo_b200.models import Evo, load_checkpoint
    want = ref[0]["checkpoint"]
    assert MODEL_NAMES == list(want["models"]) or sorted(MODEL_NAMES) == sorted(want["models"])
    for name, w in want["models"].items():
        assert get_config(name) == w["config"], name                              # every key and value of the reference's YAML
        assert w["strict"] is True and w["call_order"] == ["StripedHyena", "load_state_dict", "to_bfloat16_except_poles_residues", "to"]
    with pytest.raises(ValueError) as ex:
        Evo("evo-2-7b")
    assert str(ex.value) == want["bad_name"]
    # the same snapshot on disk
    cfg = O.tiny_config(num_layers=3, attn_layer_idxs=(1,), hidden_size=256, num_heads=2)
    cfg["max_seqlen"] = 128
    sd = O.random_state_dict(cfg, seed=7)
    sd.pop("unembed.weight")
    names = sorted(sd)
    assert ["backbone." + k for k in names] == want["source_checkpoint"]["keys_on_disk"]
    weight_map = {}
    for fname, keys in (("model-00001-of-00002.safetensors", names[: len(names) // 2]), ("model-00002-of-00002.safetensors", names[len(names) // 2:])):
        save_file({"backbone." + k: sd[k].contiguous() for k in keys}, str(tmp_path / fname))
        weight_map.update({"backbone." + k: fname for k in keys})
    (tmp_path / "model.safetensors.index.json").write_text(json.dumps({"weight_map": weight_map}))
    cfg_path = tmp_path / "tiny.yml"
    cfg_path.write_text(yaml.safe_dump(cfg))
    asked = []
    monkeypatch.setattr(huggingface_hub, "snapshot_download", lambda repo, revision=None, **kw: (asked.append([repo, revision]), str(tmp_path))[1])
    digest = lambda t: hashlib.sha256(t.detach().cpu().contiguous().view(torch.uint8).numpy().tobytes()).hexdigest()[:16]
    for name, w in want["models"].items():
        for streaming in (True, False):
            asked.clear()
            m = load_checkpoint(name, config_path=str(cfg_path), streaming=streaming)
            assert asked == [w["snapshot_download"]], (name, asked)
            got = m.state_dict()
            assert sorted(got) == sorted(want["state_dict"])
            for k, (shape, dtype, sha) in want["state_dict"].items():
                t = got[k]
                if k.endswith("rotary_emb.inv_freq"):
                    # a buffer, not a parameter: load_state_dict copies the checkpoint's values into the module's fp32 buffer
                    # (flash_attn layers/rotary.py:386-401 keeps an fp32 inv_freq); the VALUES are the checkpoint's
                    assert t.dtype == torch.float32
                    t = t.to(getattr(torch, dtype.split(".")[1]))
                assert [list(t.shape), str(t.dtype), digest(t)] == [shape, dtype, sha], (name, streaming, k)
    empty = tmp_path / "empty"
    empty.mkdir()
    monkeypatch.setattr(huggingface_hub, "snapshot_download", lambda repo, revision=None, **kw: str(empty))
    with pytest.raises(FileNotFoundError) as ex:
        load_checkpoint("evo-1-8k-base", config_path=str(cfg_path), streaming=False)
    assert str(ex.value).replace(str(empty), "<dir>") == want["no_files"]


class _FakeEvo:
    """Evo(...) without a checkpoint: the fixture's oracle model behind the scripts' `Evo` name."""
    made = []

    def __init__(self, model_name, device=None, **kw):
        class Model(OracleAsModel):
            def to(self, device):
                return self
        self.model, self.tokenizer = Model(), CharLevelTokenizer(512)
        _FakeEvo.made.append([model_name, device])


def test_score_cli_writes_the_reference_tsv(ref, tmp_path, monkeypatch, capsys):
    """scripts/score.py main(): same file-order rows, same header, same float text as the pandas TSV of the reference's script."""
    import scripts.score as cli
    want = ref[0]["cli"]["score"]
    monkeypatch.setattr(cli, "Evo", _FakeEvo)
    tsv = tmp_path / "scores.tsv"
    argv = [a if a != "<tsv>" else str(tsv) for a in want["argv"]]
    argv[argv.index("examples/example_seqs.fasta")] = os.path.join(ROOT, "examples", "example_seqs.fasta")
    cli.main(argv)
    assert tsv.read_text() == want["tsv"]
    assert capsys.readouterr().out == want["stdout"]
    assert _FakeEvo.made[-1][0] == want["evo_args"][0]                           # default model name


def test_generate_cli_prints_what_the_reference_prints(ref, monkeypatch, capsys):
    import scripts.generate as cli
    want = ref[0]["cli"]["generate"]
    monkeypatch.setattr(cli, "Evo", _FakeEvo)
    cli.main(want["argv"])
    assert capsys.readouterr().out == want["stdout"]
    assert _FakeEvo.made[-1][0] == want["evo_args"][0]


def test_length_buckets_match_the_reference_read_prompts(ref, tmp_path):
    """frontend.read_prompts_csv + length_buckets(mode="exact") = semantic_design.read_prompts (BOM, header row, quoted field,
    first-seen order of the lengths, batches of <= batch_size identical-length prompts)."""
    from evo_b200.frontend import length_buckets, read_prompts_csv
    want = ref[0]["bucketing"]
    path = tmp_path / "prompts.csv"
    with open(path, "w", encoding="utf-8", newline="") as f:
        f.write(want["csv"])
    seqs = read_prompts_csv(str(path))
    assert seqs == want["unbatched"]
    for bs in (150, 2, 1):
        got = [[seqs[i] for i in idx] for idx in length_buckets(seqs, batch_size=bs, mode="exact")]
        assert got == want[f"batched_{bs}"], bs
