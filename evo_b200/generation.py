"""Token-by-token generation on top of the stateful call `model(x, inference_params_dict=d)`.

Same entry points, arguments and observable behaviour as the reference's evo/generation.py
(class Generator :38-204, function generate :207-297):
  * the first `force_prompt_threshold` prompt tokens go through one parallel forward, the rest of
    the prompt is teacher-forced one step at a time, then `num_tokens` tokens are sampled;
  * the position bookkeeping the caller-visible state objects expose (`seqlen_offset` on both
    holders) follows the reference, including its jump to the full prompt length after a
    truncated prefill (quirk Q1) and its report-only EOS check (Q2);
  * the per-sequence "scores" keep the reference's one-off alignment (Q3, SURVEY.md 8c).
What differs is underneath: the Hyena prefill state comes out of the scan kernel, so a prompt of
any length can be prefilled in one pass (`force_prompt_threshold >= len(prompt)`); there is no
(B, D, 8, 2L) FFT temporary that forces the 128-token cap."""
from __future__ import annotations

import os
import sys
from typing import List, NamedTuple, Optional, Sequence, Tuple

import numpy as np
import torch

from .scoring import logits_to_logprobs, prepare_batch
from .stripedhyena.sample import sample
from .tokenizer import CharLevelTokenizer


def _gb(device) -> float:
    return torch.cuda.memory_allocated(device=device) / 1e9 if torch.cuda.is_available() else 0.0


# rows per batch of the ragged path: the stream-K decode GEMM takes at most 64 rows
RAGGED_CHUNK = 64


class RowSchedule(NamedTuple):
    prefill: int     # P_b = min(force_prompt_threshold, len_b): tokens of the parallel prefill
    start: int       # position of loop step 0: the FULL prompt length, even after a truncated prefill (Q1)
    n_forced: int    # prompt tokens teacher-forced inside the loop (the tail after its first token)
    n_out: int       # tokens sampled inside the loop (n_tokens - 1 when the prefill logits give the first one)
    steps: int       # single-token steps the loop runs = n_forced + n_out


def ragged_schedule(lengths: Sequence[int], threshold: int, n_tokens: int) -> List[RowSchedule]:
    """The cached generation protocol of each prompt, as the device loop runs it (evo/generation.py:131-189): prefill the
    first P = min(threshold, len) tokens in parallel; if the prompt has a tail past P, the prefill's logits are dropped,
    loop step 0 feeds tail[0] at position len (Q1: positions P..len-1 are skipped) and the rest of the tail is forced
    before n_tokens tokens are sampled; otherwise the prefill's logits give the first token and the loop samples the
    other n_tokens - 1, starting at position len.  Step i of a row runs at position start + i."""
    out = []
    for n in lengths:
        n = int(n)
        prefill = min(int(threshold), n)
        tail = n - prefill
        n_forced = max(tail - 1, 0)
        n_out = int(n_tokens) if tail else max(int(n_tokens) - 1, 0)
        out.append(RowSchedule(prefill, n, n_forced, n_out, n_forced + n_out))
    return out


class Generator:
    def __init__(self, model, tokenizer: CharLevelTokenizer, top_k: int = 50, top_p: float = 0.7, temperature: float = 1.0):
        self.model, self.tokenizer = model, tokenizer
        self.top_k, self.top_p, self.temperature = top_k, top_p, temperature
        self.untils = ["\n\n"]
        # the token loop runs on the GPU (model.decode_loop) whenever generation is cached; "0" keeps the per-token host loop
        self.device_loop = os.environ.get("EVO_B200_DEVICE_LOOP", "1") != "0"

    # -- pieces of generate() -------------------------------------------------------------
    def _state_for(self, batch: int, device, cached: bool, given: Optional[dict]):
        """(state dict or None, cached?, already prefilled?).  A caller-held state is moved to the
        prompt's device and resumed (evo/generation.py:105-114); otherwise a fresh one is made."""
        if given is not None:
            holders = (given["mha"].key_value_memory_dict, given["hyena"].fir_state_dict, given["hyena"].state_dict)
            for store in holders:
                for key in list(store):
                    store[key] = store[key].to(device)
            return given, True, True
        if not cached:
            return None, False, False
        fresh = self.model.initialize_inference_params()
        for holder in (fresh["mha"], fresh["hyena"]):
            holder.max_batch_size = batch
        return fresh, True, False

    @staticmethod
    def _advance(state: dict, full_prompt_len: int) -> None:
        attn, rec = state["mha"], state["hyena"]
        if attn.seqlen_offset == 0:
            # first step after the prefill: the reference sets the FULL prompt length even if only
            # `force_prompt_threshold` tokens were prefilled (Q1) -- reproduced, not repaired
            attn.seqlen_offset = rec.seqlen_offset = full_prompt_len
        else:
            attn.seqlen_offset += 1
            rec.seqlen_offset += 1

    def _pick(self, last_logits: torch.Tensor) -> torch.Tensor:
        return sample(last_logits, top_k=self.top_k, top_p=self.top_p, temperature=self.temperature)

    def _generate_on_device(self, window, full_prompt, x, tail, num_tokens, state, resumed, stop_at_eos, print_generation, verbose, input_string):
        """Same token sequence as the per-token loop below, with the loop itself on the GPU (SURVEY 8f-2): the prompt goes
        through one parallel forward, then ONE captured CUDA graph per token runs all blocks, picks the token
        (evo_sample_step: forced prompt tail first, then top-k/top-p/temperature or argmax), records it and its logits and
        feeds it back -- no host synchronisation until the end.  Differences from the reference, all report-only: the
        per-token print and the EOS notice (Q2) come out after the loop instead of during it."""
        tk = self.tokenizer
        n_seq, n_tail = window.shape[0], tail.shape[1]
        dev = window.device
        total = n_tail + num_tokens
        plan = ragged_schedule([window.shape[1]], x.shape[1], num_tokens)[0]     # the same bookkeeping as the ragged path
        picked = torch.empty(n_seq, num_tokens, dtype=torch.long, device=dev)
        kept_logits = torch.empty(n_seq, num_tokens, tk.vocab_size, dtype=torch.float, device=dev)
        pick_args = dict(top_k=self.top_k, top_p=self.top_p, temperature=self.temperature)
        first = 0
        if resumed:
            token = x[:, -1]
            attn = state["mha"]
            start = full_prompt.shape[-1] if attn.seqlen_offset == 0 else attn.seqlen_offset + 1
            forced, n_loop = tail, total
        else:
            with torch.inference_mode():
                logits, state = self.model(x, inference_params_dict=state)
            head = logits[:, -1].contiguous()
            if n_tail:
                token = tail[:, 0]
            else:
                token = self._pick_device(head)
                kept_logits[:, 0], picked[:, 0] = head, token
                first = 1
            start = full_prompt.shape[-1]                      # the reference's jump to the full prompt length (Q1)
            forced, n_loop = tail[:, 1:], plan.steps
        if n_loop > 0:
            got, got_logits = self.model.decode_loop(token, state, n_loop, start, forced=forced if forced.shape[1] else None,
                                                     n_out=plan.n_out if not resumed else num_tokens - first, **pick_args)
            picked[:, first:], kept_logits[:, first:] = got, got_logits
        if stop_at_eos and num_tokens >= 2 and bool((picked[0, -2:] == tk.eos).all()):
            print("Stopping generation at EOS")              # report only, as in the reference (Q2)
        if print_generation and verbose and n_seq == 1:
            for t in torch.cat([tail[0], picked[0]]).tolist():
                print(tk.detokenize([t]), end=" ")
        if verbose:
            shown = tk.detokenize_batch(picked)
            shown = [t.split(stop)[0] if stop in t else t for t in shown for stop in self.untils[:1]]
            print(f"\n[generate] in: {input_string} | out: {shown} | {_gb(dev):.2f} GB allocated")
        return picked, kept_logits, state

    def _pick_device(self, head: torch.Tensor) -> torch.Tensor:
        """One call of the device sampler (evo_sample) on (B, V) bf16 logits."""
        import ctypes as C
        from . import _lib
        out = torch.empty(head.shape[0], dtype=torch.long, device=head.device)
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        head = head.to(torch.bfloat16).contiguous()
        _lib.check(_lib.lib().evo_sample(_lib.ptr(head), _lib.ptr(out), head.shape[0], head.shape[1], int(self.top_k), float(self.top_p), float(self.temperature),
                                         seed, 0, C.c_void_p(torch.cuda.current_stream(head.device).cuda_stream)), "evo_sample")
        return out

    def can_run_ragged(self, device, cached_generation: bool) -> bool:
        """Whether generate_ragged applies: cached generation with the loop on a CUDA device (model.decode_loop_ragged)."""
        return (bool(cached_generation) and self.device_loop and hasattr(self.model, "decode_loop_ragged")
                and torch.device(device).type == "cuda")

    def generate_ragged(self, device: str, prompts_ids: Sequence[torch.Tensor], num_tokens: int = 32, force_prompt_threshold: int = 128,
                        seed: Optional[int] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        """Prompts of different lengths as ONE batch through the on-device loop.  Row b produces what generate() produces for
        prompts_ids[b] alone with cached generation (same prefill slice, same teacher-forced tail, Q1's position jump, same
        token/logit alignment), up to the rounding of a different batch shape.  prompts_ids: 1-D (or (1, n)) id tensors,
        at most 64.  Returns (picked (B, num_tokens) int64, kept_logits (B, num_tokens, V) fp32); there is no resumable
        state, since the rows end at different positions."""
        from ._lib import EvoError
        rows = [torch.as_tensor(p).reshape(-1).to(device=device, dtype=torch.long) for p in prompts_ids]
        B, num_tokens = len(rows), int(num_tokens)
        if not 1 <= B <= RAGGED_CHUNK:
            raise ValueError(f"generate_ragged takes 1..{RAGGED_CHUNK} prompts, got {B}")
        if min(r.numel() for r in rows) < 1 or num_tokens < 1:
            raise ValueError("every prompt needs a token and num_tokens must be >= 1")
        plan = ragged_schedule([r.numel() for r in rows], force_prompt_threshold, num_tokens)
        W = max(s.prefill for s in plan)
        F = max(s.n_forced for s in plan)
        ids = torch.zeros(B, W, dtype=torch.long, device=device)
        forced = torch.zeros(B, max(F, 1), dtype=torch.long, device=device)
        tail0 = torch.zeros(B, dtype=torch.long, device=device)
        for b, (r, s) in enumerate(zip(rows, plan)):
            ids[b, :s.prefill] = r[:s.prefill]
            if r.numel() > s.prefill:
                tail0[b] = r[s.prefill]
                forced[b, :s.n_forced] = r[s.prefill + 1:]
        has_tail = torch.tensor([r.numel() > s.prefill for r, s in zip(rows, plan)], device=device)
        state = self.model.initialize_inference_params()
        for holder in (state["mha"], state["hyena"]):
            holder.max_batch_size = B
        cap = state["mha"].max_seqlen
        for b, s in enumerate(plan):                           # checked per row, before anything runs (mha.py:367)
            if s.start + s.steps > cap:
                raise EvoError(f"row {b}: sequence length {s.start + s.steps} exceeds the KV cache ({cap}) (mha.py:367)")
        with torch.inference_mode():
            head = self.model.prefill_ragged(ids, [s.prefill for s in plan], state)
        sampled = self._pick_device(head)
        token = torch.where(has_tail, tail0, sampled)
        pick_args = dict(top_k=self.top_k, top_p=self.top_p, temperature=self.temperature)
        picked, kept = self.model.decode_loop_ragged(token, state, [s.start for s in plan], [s.n_forced for s in plan], [s.n_out for s in plan],
                                                     forced=forced if F else None, out_cols=num_tokens, seed=seed, **pick_args)
        first = ~has_tail                                      # rows whose first token came from the prefill's logits
        picked[first, 0] = sampled[first]
        kept[first, 0] = head[first].float()
        return picked, kept

    # -- public ---------------------------------------------------------------------------
    def generate(self, device: str, input_string: str = None, input_ids: torch.Tensor = None, num_tokens: int = 32,
                 cached_generation: bool = True, force_prompt_threshold: int = 128, print_generation: bool = True,
                 verbose: bool = False, skip_special_tokens: bool = False, stop_at_eos: bool = True,
                 max_seqlen: int = None, inference_params_dict: dict = None) -> Tuple[torch.Tensor, torch.Tensor, dict]:
        tk = self.tokenizer
        full_prompt = input_ids if input_ids is not None else torch.tensor(tk.tokenize(input_string), dtype=torch.long, device=device)[None]
        window = full_prompt if max_seqlen is None else full_prompt[:, -max_seqlen:]
        num_tokens = int(num_tokens)
        n_seq, n_prompt = window.shape
        dev = window.device

        # prompt split: [prefilled in parallel | teacher-forced step by step]
        tail = window[:, force_prompt_threshold:] if n_prompt > force_prompt_threshold else window[:, :0]
        x = window[:, :force_prompt_threshold] if tail.shape[1] else window
        n_tail = tail.shape[1]

        picked = torch.empty(n_seq, num_tokens, dtype=torch.long, device=dev)
        kept_logits = torch.empty(n_seq, num_tokens, tk.vocab_size, dtype=torch.float, device=dev)
        eos = torch.tensor([tk.eos], dtype=torch.long, device=device)
        state, cached_generation, resumed = self._state_for(n_seq, dev, cached_generation, inference_params_dict)

        if verbose:
            what = f"prompt {input_string!r}" if input_string is not None else f"prompt ids {tuple(input_ids.shape)}"
            print(f"[generate] {what}; {_gb(dev):.2f} GB allocated; prefill {x.shape[1]} + forced {n_tail} + new {num_tokens}")

        if cached_generation and self.device_loop and hasattr(self.model, "decode_loop") and window.is_cuda and n_tail + num_tokens > 0:
            return self._generate_on_device(window, full_prompt, x, tail, num_tokens, state, resumed, stop_at_eos, print_generation, verbose, input_string)

        last_step = -1
        for last_step in range(n_tail + num_tokens):
            one_token = resumed or (cached_generation and last_step > 0)
            if one_token:
                x = x[:, -1:]
                self._advance(state, full_prompt.shape[-1])
            with torch.inference_mode():
                logits, state = self.model(x, inference_params_dict=state)
            head = logits[:, -1]
            token = tail[:, last_step] if last_step < n_tail else self._pick(head)

            if stop_at_eos and num_tokens >= 2 and bool((picked[0, -2:] == eos).all()):
                print("Stopping generation at EOS")              # report only, as in the reference (Q2)
            if print_generation and verbose and n_seq == 1:
                print(tk.detokenize([token.item()]), end=" ")

            k = last_step - n_tail
            if k >= 0:
                kept_logits[:, k], picked[:, k] = head, token
            x = token[:, None] if one_token else torch.cat([x, token[:, None]], dim=-1)

        done = last_step + 1
        if verbose:
            shown = tk.detokenize_batch(picked[:, :done])
            shown = [t.split(stop)[0] if stop in t else t for t in shown for stop in self.untils[:1]]
            print(f"\n[generate] in: {input_string} | out: {shown} | {_gb(dev):.2f} GB allocated")
        return picked[:, :done], kept_logits[:, :done], state


def generate(prompt_seqs: List[str], model, tokenizer: CharLevelTokenizer, n_tokens: int = 100, temperature: float = 0.0,
             top_k: int = 1, top_p: float = 1.0, batched: bool = True, prepend_bos: bool = False,
             cached_generation: bool = False, force_prompt_threshold: int = 128, verbose: int = 1,
             device: str = "cuda:0", ragged: bool = False, **kwargs) -> Tuple[List[str], List[float]]:
    """Sequences and mean log-likelihood "scores" for a list of prompts.  Prompts of one common
    length run as one batch; anything else falls back to one prompt at a time (with a note on stderr).
    ragged=True: prompts of different lengths run as batches of up to 64 through the on-device loop
    (Generator.generate_ragged); each row produces what its prompt produces alone.  It applies to cached generation
    with the loop on a CUDA device; otherwise generate() behaves as without it."""
    model.eval()
    engine = Generator(model, tokenizer, top_k=top_k, top_p=top_p, temperature=temperature)
    uniform = len({len(p) for p in prompt_seqs}) <= 1
    if ragged and batched and not uniform and engine.can_run_ragged(device, cached_generation):
        return _generate_ragged(engine, prompt_seqs, tokenizer, n_tokens, prepend_bos, force_prompt_threshold, verbose, device)
    if batched and uniform:
        work = [list(prompt_seqs)]
    else:
        if verbose and not uniform:
            sys.stderr.write("Note: Prompts are of different lengths.\n")
        if verbose:
            sys.stderr.write("Note: Will not do batched generation.\n")
        work = [[p] for p in prompt_seqs]

    chatty = verbose > 1
    texts: List[str] = []
    scores: List[float] = []
    for group in work:
        ids, _ = prepare_batch(group, tokenizer, prepend_bos=prepend_bos, device=device)
        new_ids, new_logits, _ = engine.generate(device=device, input_ids=ids, num_tokens=n_tokens, stop_at_eos=False,
                                                 cached_generation=cached_generation, force_prompt_threshold=force_prompt_threshold,
                                                 print_generation=chatty, verbose=chatty)
        if chatty:
            print(f"[generate] ids {tuple(ids.shape)} -> new ids {tuple(new_ids.shape)}, logits {tuple(new_logits.shape)}")
        decoded = tokenizer.detokenize_batch(new_ids)
        if len(decoded) != ids.shape[0]:
            raise AssertionError("batch size mismatch after detokenisation")
        texts.extend(decoded)
        # logits_to_logprobs(trim_bos=True) pairs logits[i] with token[i+1]: the reference's alignment (Q3)
        per_token = logits_to_logprobs(new_logits, new_ids).float().cpu().numpy()
        scores.extend(float(np.mean(row)) for row in per_token)

    if verbose:
        for prompt, text, score in zip(prompt_seqs, texts, scores):
            print(f'Prompt: "{prompt}",\tOutput: "{text}",\tScore: {score}')
    return texts, scores


def _generate_ragged(engine: Generator, prompt_seqs: List[str], tokenizer: CharLevelTokenizer, n_tokens: int, prepend_bos: bool,
                     force_prompt_threshold: int, verbose: int, device: str) -> Tuple[List[str], List[float]]:
    """generate(ragged=True): prompts sorted by length, cut into batches of at most RAGGED_CHUNK rows, results back in
    input order.  Texts and scores are computed per row exactly as for a batch of one."""
    ids = [prepare_batch([p], tokenizer, prepend_bos=prepend_bos, device=device)[0][0] for p in prompt_seqs]
    order = sorted(range(len(ids)), key=lambda i: ids[i].numel())
    texts: List[Optional[str]] = [None] * len(ids)
    scores: List[Optional[float]] = [None] * len(ids)
    for c in range(0, len(order), RAGGED_CHUNK):
        chunk = order[c:c + RAGGED_CHUNK]
        new_ids, new_logits = engine.generate_ragged(device, [ids[i] for i in chunk], num_tokens=n_tokens, force_prompt_threshold=force_prompt_threshold)
        decoded = tokenizer.detokenize_batch(new_ids)
        for r, i in enumerate(chunk):
            texts[i] = decoded[r]
            # logits_to_logprobs(trim_bos=True) pairs logits[i] with token[i+1]: the reference's alignment (Q3)
            scores[i] = float(np.mean(logits_to_logprobs(new_logits[r:r + 1], new_ids[r:r + 1]).float().cpu().numpy()[0]))
    if verbose:
        for prompt, text, score in zip(prompt_seqs, texts, scores):
            print(f'Prompt: "{prompt}",\tOutput: "{text}",\tScore: {score}')
    return texts, scores
