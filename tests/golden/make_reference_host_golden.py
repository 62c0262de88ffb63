"""Generates tests/golden/reference_host.{json,npz}: outputs of the REFERENCE'S OWN host code, run on CPU.

What is pinned.  evo/{tokenizer,scoring,generation,models}.py of the reference checkout are the reference for everything on either
side of the model call (SURVEY.md 8b, 8f-1..4): tokenisation, batch preparation, the logits -> log-likelihood / entropy
reductions, the generation loop's state protocol (which slices of the prompt the model sees and which `seqlen_offset` it is
handed at every call, quirks Q1-Q4 included) and checkpoint ingest (HF repo / revision, 'backbone.' strip, tied unembed,
YAML config, strict load, dtype policy call order).  Those files import `stripedhyena`, which does not exist here
(SURVEY.md 0.1) -- so this script registers a stand-in `stripedhyena` package whose `StripedHyena` is a recorder, whose
`sample` is flash_attn.utils.generation.sample (installed here; the function stripedhyena/sample.py copies) and whose `dotdict`
is a plain attribute dict, imports the reference's modules UNMODIFIED from the checkout, and drives them on CPU with the
oracle model (oracle/stripedhyena_oracle.py) standing where the real model would.  The bf16 oracle's logits are stored too:
a bf16 matmul on CPU rounds differently with and without AMX, so the test replays them instead of recomputing them.

What is NOT pinned by this: the model arithmetic (the oracle stays a restatement; "parity unpinned" in its header stands).
The fixtures pin the host layer: tests/test_reference_host_golden.py runs evo_b200's host code over the SAME oracle model and
must reproduce every id, call, string and score; the GPU tests compare the CUDA path's scores with the fp64 numbers.

    python tests/golden/make_reference_host_golden.py <path of the reference checkout>
"""
import hashlib
import json
import os
import sys
import tempfile
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.normpath(os.path.join(HERE, "..", ".."))
REFERENCE = None          # the reference checkout, from the command line
sys.path.insert(0, ROOT)

from oracle import stripedhyena_oracle as O  # noqa: E402

SEQS = ["ACGTTGCAACGTACGTAGCTAGCTAGGATC", "ACGTAC", "TTTTGGGGCCCCAAAA"]          # tests/test_gpu_parity.py's public-API case
PROMPTS = ["ACGTACGT", "TTGACCAA"]
TOKENIZER_TEXTS = ["ACGT", "acgtn", "", "A C\tG\nT", "|d__Bacteria;p__Pseudomonadota|", "~\x7f\x01\x1f !", "N" * 40]
TOKENIZER_IDS = [[65, 67, 71, 84], [0, 1, 31, 32, 33, 126, 127, 128, 255, 300, 511, 512, 600], []]


class Recorder:
    """Stands where stripedhyena.model.StripedHyena would inside evo/models.py: notes what load_checkpoint does to it."""
    log = []

    def __init__(self, config):
        Recorder.log.append(["StripedHyena", {k: v for k, v in dict(config).items() if k != "Loader"}, sorted(k for k in dict(config) if k == "Loader")])

    def load_state_dict(self, state_dict, strict=None):
        Recorder.log.append(["load_state_dict", {"strict": strict, "tensors": {
            k: [list(v.shape), str(v.dtype), hashlib.sha256(v.contiguous().view(torch.uint8).numpy().tobytes()).hexdigest()[:16], int(v.data_ptr())]
            for k, v in state_dict.items()}}])

    def to_bfloat16_except_poles_residues(self):
        Recorder.log.append(["to_bfloat16_except_poles_residues"])

    def to(self, device):
        Recorder.log.append(["to", str(device)])
        return self


class dotdict(dict):
    __getattr__ = dict.get
    __setattr__ = dict.__setitem__
    __delattr__ = dict.__delitem__


def install_stand_in():
    pkg = types.ModuleType("stripedhyena")
    pkg.__path__ = []
    from flash_attn.utils.generation import sample as flash_attn_sample       # the code stripedhyena/sample.py copies; pure torch
    for name, attrs in (("model", {"StripedHyena": Recorder}), ("sample", {"sample": flash_attn_sample}), ("utils", {"dotdict": dotdict}),
                        ("tokenizer", {})):
        mod = types.ModuleType("stripedhyena." + name)
        mod.__dict__.update(attrs)
        sys.modules["stripedhyena." + name] = mod
        setattr(pkg, name, mod)
    sys.modules["stripedhyena"] = pkg


class OracleAsModel:
    """The oracle behind the object protocol evo/ uses; logs every call the reference's host code makes."""

    def __init__(self, cfg, sd, dtype):
        self.m = O.OracleStripedHyena(cfg, sd, dtype)
        self.calls = []
        self.logits = []

    def eval(self):
        return self

    def initialize_inference_params(self):
        return self.m.initialize_inference_params()

    def __call__(self, x, inference_params_dict=None):
        d = inference_params_dict
        self.calls.append([list(x.shape), None if d is None else int(d["mha"].seqlen_offset), None if d is None else int(d["hyena"].seqlen_offset)])
        out = self.m(x, d)
        self.logits.append(out[0])
        return out


def tiny():
    cfg = O.tiny_config(num_layers=3, attn_layer_idxs=(1,), hidden_size=256, num_heads=2)      # = _tiny(layers=3, attn=(1,)) of the GPU tests
    cfg["max_seqlen"] = 128
    return cfg, O.random_state_dict(cfg, seed=7)


def tokenizer_cases(RT):
    tok = RT.CharLevelTokenizer(512)
    out = {"vocab_size": tok.vocab_size, "eod_id": tok.eod_id, "eos_id": tok.eos_id, "pad_id": tok.pad_id, "eod": tok.eod, "eos": tok.eos,
           "tokenize": [[t, [int(i) for i in tok.tokenize(t)]] for t in TOKENIZER_TEXTS],
           "tokenize_batch": [[int(i) for i in row] for row in tok.tokenize_batch(TOKENIZER_TEXTS[:3])],
           "detokenize": [[ids, tok.detokenize(ids)] for ids in TOKENIZER_IDS],
           "detokenize_batch_list": tok.detokenize_batch(TOKENIZER_IDS),
           "detokenize_batch_tensor": tok.detokenize_batch(torch.tensor([[65, 67, 10, 3], [84, 84, 200, 511]])),
           "clamp": [[n, tok.clamp(n)] for n in (-5, 0, 31, 32, 100, 511, 512, 9999)]}
    return out


def scoring_cases(RS, RT, arrays):
    tok = RT.CharLevelTokenizer(512)
    out = {"seqs": SEQS}
    for bos in (True, False):
        ids, lengths = RS.prepare_batch(SEQS, tok, prepend_bos=bos, device="cpu")
        assert ids.dtype == torch.long
        arrays[f"prepare_batch_ids_bos{int(bos)}"] = ids.numpy()
        out[f"prepare_batch_lengths_bos{int(bos)}"] = [int(n) for n in lengths]
    # logits -> log-likelihoods on fixed logits, both trims, fp32 and bf16 (Q4: the softmax runs in the logits' dtype)
    g = torch.Generator().manual_seed(11)
    logits = torch.randn(2, 9, 512, generator=g) * 3.0
    ids = torch.randint(0, 512, (2, 9), generator=g)
    arrays["l2l_logits"], arrays["l2l_ids"] = logits.numpy(), ids.numpy()
    for name, lg in (("fp32", logits), ("bf16", logits.to(torch.bfloat16))):
        for trim in (True, False):
            got = RS.logits_to_logprobs(lg, ids, trim_bos=trim)
            assert got.dtype == lg.dtype
            arrays[f"l2l_{name}_trim{int(trim)}"] = got.float().numpy()
    cfg, sd = tiny()
    for name, dtype in (("fp64", torch.float64), ("bf16", torch.bfloat16)):
        for red in ("mean", "sum"):
            model = OracleAsModel(cfg, sd, dtype)
            out[f"score_{red}_{name}"] = [float(s) for s in RS.score_sequences(SEQS, model, tok, reduce_method=red, device="cpu")]
            out[f"score_calls_{name}"] = model.calls
        if dtype == torch.bfloat16:
            arrays["score_logits_bf16"] = model.logits[0].float().numpy()       # exact: bf16 values fit in fp32
        model = OracleAsModel(cfg, sd, dtype)
        ent = RS.positional_entropies(SEQS, model, tok, device="cpu")
        if dtype == torch.bfloat16:
            assert np.array_equal(model.logits[0].float().numpy(), arrays["score_logits_bf16"])    # one batch feeds both reductions
        for k, e in enumerate(ent):
            arrays[f"entropy_{name}_{k}"] = np.asarray(e, dtype=np.float32)
    try:
        RS.score_sequences(SEQS, OracleAsModel(cfg, sd, torch.float64), tok, reduce_method="median", device="cpu")
        out["bad_reduce"] = None
    except ValueError as ex:
        out["bad_reduce"] = str(ex)
    return out


def generation_cases(RG, RS, RT, arrays):
    tok = RT.CharLevelTokenizer(512)
    cfg, sd = tiny()
    out = {}

    def run(tag, prompts, **kw):
        model = OracleAsModel(cfg, sd, torch.float64)
        try:
            texts, scores = RG.generate(prompts, model, tok, top_k=1, verbose=0, device="cpu", **kw)
        except Exception as ex:          # recorded, not hidden: what the reference does with these arguments
            out[tag] = {"prompts": prompts, "kwargs": kw, "raises": [type(ex).__name__, str(ex)], "calls": model.calls}
            return
        out[tag] = {"prompts": prompts, "kwargs": kw, "texts": texts, "scores": [float(s) for s in scores], "calls": model.calls}

    run("batched_cached", PROMPTS, n_tokens=12, cached_generation=True)
    run("batched_uncached", PROMPTS, n_tokens=6, cached_generation=False)
    run("ragged_cached", ["ACGTACGT", "TTGAC"], n_tokens=5, cached_generation=True)
    run("unbatched_by_request", PROMPTS, n_tokens=4, cached_generation=True, batched=False)
    run("prompt_forcing_q1", PROMPTS, n_tokens=5, cached_generation=True, force_prompt_threshold=3)
    run("prepend_bos", PROMPTS, n_tokens=5, cached_generation=True, prepend_bos=True)
    run("one_token", ["ACGT"], n_tokens=1, cached_generation=True)

    # sampled (not greedy): one torch.multinomial draw per step from the global generator, so the seed fixes the strings
    def run_sampled(tag, prompts, seed, **kw):
        model = OracleAsModel(cfg, sd, torch.float64)
        torch.manual_seed(seed)
        texts, scores = RG.generate(prompts, model, tok, verbose=0, device="cpu", **kw)
        out[tag] = {"prompts": prompts, "seed": seed, "kwargs": kw, "texts": texts, "scores": [float(s) for s in scores], "calls": model.calls}

    run_sampled("sampled_topk4", PROMPTS, 123, n_tokens=8, cached_generation=True, top_k=4, temperature=0.8)
    run_sampled("sampled_topk50_topp", PROMPTS, 124, n_tokens=8, cached_generation=True, top_k=50, top_p=0.7, temperature=1.0)
    run_sampled("sampled_full_vocab", ["ACGTAC"], 125, n_tokens=6, cached_generation=True, top_k=0, top_p=0.9, temperature=1.2)

    # Generator.generate directly: returned tensors, then a resumed call on the returned state (evo/generation.py:105-114,140-148)
    model = OracleAsModel(cfg, sd, torch.float64)
    g = RG.Generator(model, tok, top_k=1)
    ids, _ = RS.prepare_batch(PROMPTS, tok, prepend_bos=False, device="cpu")
    new_ids, new_logits, state = g.generate(device="cpu", input_ids=ids, num_tokens=4, cached_generation=True, print_generation=False, stop_at_eos=False)
    arrays["gen_first_ids"], arrays["gen_first_logits"] = new_ids.numpy(), new_logits.numpy()
    offs_after_first = [int(state["mha"].seqlen_offset), int(state["hyena"].seqlen_offset)]
    more_ids, more_logits, state2 = g.generate(device="cpu", input_ids=new_ids[:, -1:], num_tokens=3, print_generation=False, stop_at_eos=False,
                                                inference_params_dict=state)
    arrays["gen_resumed_ids"], arrays["gen_resumed_logits"] = more_ids.numpy(), more_logits.numpy()
    out["resume"] = {"calls": model.calls, "offsets_after_first": offs_after_first, "same_state_object": state2 is state,
                     "offsets_after_resume": [int(state["mha"].seqlen_offset), int(state["hyena"].seqlen_offset)],
                     "state_keys": {"kv": sorted(int(k) for k in state["mha"].key_value_memory_dict), "fir": sorted(int(k) for k in state["hyena"].fir_state_dict),
                                    "iir": sorted(int(k) for k in state["hyena"].state_dict)},
                     "max_batch_size": [int(state["mha"].max_batch_size), int(state["hyena"].max_batch_size)]}
    # input_string instead of input_ids, and max_seqlen cropping the prompt window
    model = OracleAsModel(cfg, sd, torch.float64)
    g = RG.Generator(model, tok, top_k=1)
    s_ids, s_logits, _ = g.generate(device="cpu", input_string="ACGTACGTTT", num_tokens=3, cached_generation=True, print_generation=False, stop_at_eos=False, max_seqlen=6)
    arrays["gen_string_ids"] = s_ids.numpy()
    out["input_string_max_seqlen"] = {"calls": model.calls}
    return out


def checkpoint_cases(RM):
    """The real Evo(...) / load_checkpoint against a local two-shard snapshot and the recorder."""
    import huggingface_hub
    from safetensors.torch import save_file
    cfg, sd = tiny()
    sd = dict(sd)
    sd.pop("unembed.weight")
    names = sorted(sd)
    out = {"models": {}}
    with tempfile.TemporaryDirectory() as tmp:
        shards = {"model-00001-of-00002.safetensors": names[: len(names) // 2], "model-00002-of-00002.safetensors": names[len(names) // 2:]}
        weight_map = {}
        for fname, keys in shards.items():
            save_file({"backbone." + k: sd[k].contiguous() for k in keys}, os.path.join(tmp, fname))
            weight_map.update({"backbone." + k: fname for k in keys})
        with open(os.path.join(tmp, "model.safetensors.index.json"), "w") as f:
            json.dump({"weight_map": weight_map}, f)
        asked = []

        def fake_snapshot_download(repo, revision=None, **kw):
            asked.append([repo, revision])
            return tmp

        real = huggingface_hub.snapshot_download
        huggingface_hub.snapshot_download = fake_snapshot_download
        try:
            for name in RM.MODEL_NAMES:
                Recorder.log, asked[:] = [], []
                evo = RM.Evo(name, device="cpu")
                log = Recorder.log
                assert [e[0] for e in log] == ["StripedHyena", "load_state_dict", "to_bfloat16_except_poles_residues", "to"], [e[0] for e in log]
                tensors = log[1][1]["tensors"]
                out["models"][name] = {"snapshot_download": asked[0], "config": log[0][1], "config_extra_keys": log[0][2], "strict": log[1][1]["strict"],
                                       "call_order": [e[0] for e in log], "to": log[3][1], "tokenizer_vocab": evo.tokenizer.vocab_size,
                                       "tied_unembed_is_same_tensor": tensors["unembed.weight"][3] == tensors["embedding_layer.weight"][3]}
                if "state_dict" not in out:
                    out["state_dict"] = {k: v[:3] for k, v in tensors.items()}
            Recorder.log = []
            try:
                RM.Evo("evo-2-7b")
                out["bad_name"] = None
            except ValueError as ex:
                out["bad_name"] = str(ex)
            # a snapshot directory without safetensors files
            with tempfile.TemporaryDirectory() as empty:
                huggingface_hub.snapshot_download = lambda repo, revision=None, **kw: empty
                try:
                    RM.load_checkpoint("evo-1-8k-base", config_path="configs/evo-1-8k-base_inference.yml")
                    out["no_files"] = None
                except FileNotFoundError as ex:
                    out["no_files"] = str(ex).replace(empty, "<dir>")
        finally:
            huggingface_hub.snapshot_download = real
    out["source_checkpoint"] = {"keys_on_disk": ["backbone." + k for k in names], "oracle_state_dict": "random_state_dict(tiny_config(3 layers, attn (1,), D 256, 2 heads), seed=7) minus unembed.weight"}
    return out


def _load_reference_script(name):
    """A file under the reference's scripts/ as a module of its own (the repo has a `scripts` package of the same name)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("reference_scripts_" + name, os.path.join(REFERENCE, "scripts", name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def cli_cases(RT, RM):
    """scripts/score.py and scripts/generate.py of the reference, main() run as written.  Stand-ins: Biopython is not installed, so
    `Bio.SeqIO.parse` is a 10-line FASTA reader (what is pinned is everything AFTER the parse: batching in file order, the TSV
    pandas writes, what is printed); `Evo(name)` returns the oracle model instead of downloading a checkpoint."""
    import contextlib
    import io

    class Record:
        def __init__(self, seq):
            self.seq = seq

    def parse(path, fmt):
        assert fmt == "fasta"
        cur = None
        for line in open(path):
            line = line.strip()
            if line.startswith(">"):
                if cur is not None:
                    yield Record("".join(cur))
                cur = []
            elif line and cur is not None:
                cur.append(line)
        if cur is not None:
            yield Record("".join(cur))

    bio, seqio = types.ModuleType("Bio"), types.ModuleType("Bio.SeqIO")
    seqio.parse = parse
    bio.SeqIO = seqio
    sys.modules["Bio"], sys.modules["Bio.SeqIO"] = bio, seqio
    cfg, sd = tiny()
    made = []

    class ModelWithTo(OracleAsModel):
        def to(self, device):
            self.moved_to = str(device)
            return self

    class FakeEvo:
        def __init__(self, model_name, device=None):
            self.model, self.tokenizer = ModelWithTo(cfg, sd, torch.float64), RT.CharLevelTokenizer(512)
            made.append([model_name, device])

    out = {}
    fasta = os.path.join(ROOT, "examples", "example_seqs.fasta")
    score = _load_reference_script("score")
    score.Evo = FakeEvo
    with tempfile.TemporaryDirectory() as tmp:
        tsv = os.path.join(tmp, "scores.tsv")
        argv, buf = sys.argv, io.StringIO()
        sys.argv = ["score.py", "--input-fasta", fasta, "--output-tsv", tsv, "--device", "cpu", "--batch-size", "2"]
        try:
            with contextlib.redirect_stdout(buf), contextlib.redirect_stderr(io.StringIO()):
                score.main()
        finally:
            sys.argv = argv
        out["score"] = {"argv": ["--input-fasta", "examples/example_seqs.fasta", "--output-tsv", "<tsv>", "--device", "cpu", "--batch-size", "2"],
                        "tsv": open(tsv).read(), "stdout": buf.getvalue(), "evo_args": made[-1]}
    gen = _load_reference_script("generate")
    gen.Evo = FakeEvo
    argv, buf = sys.argv, io.StringIO()
    sys.argv = ["generate.py", "--prompt", "ACGTAC", "--n-samples", "2", "--n-tokens", "6", "--top-k", "1", "--device", "cpu"]
    try:
        with contextlib.redirect_stdout(buf), contextlib.redirect_stderr(io.StringIO()):
            gen.main()
    finally:
        sys.argv = argv
    out["generate"] = {"argv": sys.argv and ["--prompt", "ACGTAC", "--n-samples", "2", "--n-tokens", "6", "--top-k", "1", "--device", "cpu"], "stdout": buf.getvalue(), "evo_args": made[-1]}
    return out


PROMPT_CSV = "\ufeffSequence,Note\r\nACGTACGT,a\r\nTTGA,b\r\nGGGGCCCC,c\r\nAC,d\r\nTTTTAAAA,e\r\nCCCC,f\r\nACGTACGA,g\r\nAAAATTTT,h\r\n\"ACGT,ACGT\",quoted\r\n"


def bucketing_cases():
    """semantic_design/semantic_design.py:read_prompts (:39-100), imported with the rest of its module (Biopython stand-ins for the
    names the module imports at the top; read_prompts itself uses csv only)."""
    bio = sys.modules.get("Bio") or types.ModuleType("Bio")
    for sub, names in (("SeqIO", ()), ("AlignIO", ()), ("Seq", ("Seq",)), ("SeqRecord", ("SeqRecord",))):
        mod = sys.modules.get("Bio." + sub) or types.ModuleType("Bio." + sub)
        for n in names:
            setattr(mod, n, type(n, (), {}))
        sys.modules["Bio." + sub] = mod
        setattr(bio, sub, mod)
    sys.modules["Bio"] = bio
    import importlib.util
    spec = importlib.util.spec_from_file_location("reference_semantic_design", os.path.join(REFERENCE, "semantic_design", "semantic_design.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    out = {"csv": PROMPT_CSV}
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "prompts.csv")
        with open(path, "w", encoding="utf-8", newline="") as f:
            f.write(PROMPT_CSV)
        out["unbatched"] = mod.read_prompts(path, batched=False)
        for bs in (150, 2, 1):
            out[f"batched_{bs}"] = mod.read_prompts(path, batched=True, batch_size=bs)
    return out


def main():
    global REFERENCE
    if len(sys.argv) != 2 or not os.path.isdir(os.path.join(sys.argv[1], "evo")):
        raise SystemExit("usage: make_reference_host_golden.py <path of the reference checkout (the directory holding evo/)>")
    REFERENCE = os.path.realpath(sys.argv[1])
    install_stand_in()
    sys.path.insert(0, REFERENCE)
    import evo.generation as RG
    import evo.models as RM
    import evo.scoring as RS
    import evo.tokenizer as RT
    for mod in (RG, RM, RS, RT):
        assert os.path.realpath(mod.__file__).startswith(REFERENCE + "/"), mod.__file__
    torch.manual_seed(0)
    arrays = {}
    doc = {"generated_by": "tests/golden/make_reference_host_golden.py",
           "reference_modules": {m.__name__: hashlib.sha256(open(m.__file__, "rb").read()).hexdigest()[:16] for m in (RG, RM, RS, RT)},
           "stand_ins": "stripedhyena.model.StripedHyena = recorder; stripedhyena.sample.sample = flash_attn.utils.generation.sample; stripedhyena.utils.dotdict = attribute dict; "
                        "the model object = oracle/stripedhyena_oracle.OracleStripedHyena (restatement, unpinned)",
           "tokenizer": tokenizer_cases(RT)}
    doc["scoring"] = scoring_cases(RS, RT, arrays)
    doc["generation"] = generation_cases(RG, RS, RT, arrays)
    doc["checkpoint"] = checkpoint_cases(RM)
    doc["cli"] = cli_cases(RT, RM)
    doc["bucketing"] = bucketing_cases()
    with open(os.path.join(HERE, "reference_host.json"), "w") as f:
        json.dump(doc, f, indent=1, sort_keys=True)
    np.savez_compressed(os.path.join(HERE, "reference_host.npz"), **arrays)
    for f in ("reference_host.json", "reference_host.npz"):
        print(f, os.path.getsize(os.path.join(HERE, f)))


if __name__ == "__main__":
    main()
