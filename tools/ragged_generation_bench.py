"""Generation throughput for prompts of different lengths: today's fallback against the ragged batch.

Random-init evo-1.5-8k-base on one GPU, a seeded set of prompts whose lengths are drawn from 200, 300, ..., 1100 nt (a
few lengths repeat, as in real prompt sets), greedy, `--tokens` new tokens per prompt, for each force_prompt_threshold
in `--thresholds` (2 is what semantic-design style scripts pass, 128 the default).  Three arms, timed alternately:
  (a) generate(prompts)               prompts of different lengths: one prompt at a time
  (b) exact-length groups             one generate() call per group of prompts that share a length
  (c) generate(prompts, ragged=True)  one ragged batch through the on-device loop
Reported per arm: generated nt/s (prompts x tokens / wall time, prefill and prompt forcing included).  Also reported:
the decode-step time of the uniform loop at batch B (all prompts cut to one length) against the ragged loop at batch B,
the batch-1 step time, the card's name and power limit, and whether (c) produced the same greedy tokens as (a).
Prints one JSON line; writes nothing."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card(index: int):
    name = torch.cuda.get_device_name(index)
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        power, clock = (float(v) for v in out.split(","))
    except Exception:                                    # noqa: BLE001 -- the numbers are still reported without it
        power = clock = None
    return {"name": name, "power_limit_w": power, "max_sm_clock_mhz": clock}


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def step_ms(model, prompts_ids, ragged: bool, n_steps: int) -> float:
    """ms per decode step of the loop alone (after its prefill), CUDA events around the replayed steps."""
    from evo_b200.generation import ragged_schedule
    B = len(prompts_ids)
    state = model.initialize_inference_params()
    for holder in (state["mha"], state["hyena"]):
        holder.max_batch_size = B
    with torch.inference_mode():
        if ragged:
            plan = ragged_schedule([p.numel() for p in prompts_ids], 10 ** 9, n_steps + 1)
            W = max(s.prefill for s in plan)
            ids = torch.zeros(B, W, dtype=torch.long, device=prompts_ids[0].device)
            for b, p in enumerate(prompts_ids):
                ids[b, :p.numel()] = p
            head = model.prefill_ragged(ids, [s.prefill for s in plan], state)
            run = lambda: model.decode_loop_ragged(head.argmax(-1), state, [s.start for s in plan], [0] * B, [n_steps] * B, top_k=1)
        else:
            ids = torch.stack(prompts_ids)
            logits, state = model(ids, inference_params_dict=state)
            start = ids.shape[1]
            run = lambda: model.decode_loop(logits[:, -1].argmax(-1), state, n_steps, start, top_k=1)
        run()                                            # captures the step graph
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run()
        e1.record()
        torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n_steps


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--prompts", type=int, default=16)
    ap.add_argument("--tokens", type=int, default=256)
    ap.add_argument("--thresholds", type=int, nargs="+", default=[2, 128])
    ap.add_argument("--repeats", type=int, default=2, help="alternating rounds of the three arms")
    ap.add_argument("--step-iters", type=int, default=128, help="decode steps per per-step timing")
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()

    import evo_b200
    from evo_b200 import CharLevelTokenizer
    from evo_b200.models import load_checkpoint

    dev = "cuda:0"
    model = load_checkpoint("evo-1.5-8k-base", device=dev, random_init=True, seed=0)
    tok = CharLevelTokenizer(512)
    rng = np.random.default_rng(args.seed)
    lengths = [int(n) for n in rng.choice(np.arange(200, 1101, 100), size=args.prompts)]
    prompts = ["".join(rng.choice(list("ACGT"), size=n)) for n in lengths]
    kw = dict(n_tokens=args.tokens, top_k=1, cached_generation=True, verbose=0, device=dev)
    n_gen = len(prompts) * args.tokens

    def grouped(threshold):
        by_len = {}
        for i, p in enumerate(prompts):
            by_len.setdefault(len(p), []).append(i)
        texts = [None] * len(prompts)
        for idx in by_len.values():
            out, _ = evo_b200.generate([prompts[i] for i in idx], model, tok, force_prompt_threshold=threshold, **kw)
            for i, t in zip(idx, out):
                texts[i] = t
        return texts

    arms = {"a_one_at_a_time": lambda thr: evo_b200.generate(prompts, model, tok, force_prompt_threshold=thr, **kw)[0],
            "b_exact_length_groups": grouped,
            "c_ragged": lambda thr: evo_b200.generate(prompts, model, tok, force_prompt_threshold=thr, ragged=True, **kw)[0]}
    result = {"model": "evo-1.5-8k-base (random init)", "prompts": len(prompts), "prompt_lengths": lengths,
              "distinct_lengths": len(set(lengths)), "new_tokens": args.tokens, "greedy": True, "card": card(0), "thresholds": {}}
    for thr in args.thresholds:
        arms["c_ragged"](thr)                             # warm-up: graph captures, rope tables, workspaces
        times = {k: [] for k in arms}
        texts = {}
        for _ in range(args.repeats):
            for name, fn in arms.items():
                sec, texts[name] = timed(lambda: fn(thr))
                times[name].append(sec)
        a, c = texts["a_one_at_a_time"], texts["c_ragged"]
        same = [x == y for x, y in zip(a, c)]
        first_diff = [next((k for k, (u, v) in enumerate(zip(x, y)) if u != v), None) for x, y in zip(a, c)]
        result["thresholds"][str(thr)] = {
            "seconds": {k: v for k, v in times.items()},
            "generated_nt_per_s": {k: n_gen / min(v) for k, v in times.items()},
            "ragged_speedup_over_a": min(times["a_one_at_a_time"]) / min(times["c_ragged"]),
            "ragged_speedup_over_b": min(times["b_exact_length_groups"]) / min(times["c_ragged"]),
            "greedy_rows_identical_c_vs_a": int(sum(same)), "first_differing_token_per_row": first_diff,
        }
        print(json.dumps({"threshold": thr, **result["thresholds"][str(thr)]}), file=sys.stderr, flush=True)

    # decode-step time: uniform loop vs ragged loop at the same batch, and batch 1
    g = torch.Generator().manual_seed(args.seed)
    acgt = torch.tensor([65, 67, 71, 84])
    ids = [acgt[torch.randint(0, 4, (n,), generator=g)].to(dev) for n in lengths]
    common = int(np.median(lengths))
    uniform = [p.repeat(-(-common // p.numel()))[:common] for p in ids]
    steps = {"uniform_B%d" % len(ids): [], "ragged_B%d" % len(ids): [], "uniform_B1": []}
    for _ in range(3):
        steps["uniform_B%d" % len(ids)].append(step_ms(model, uniform, False, args.step_iters))
        steps["ragged_B%d" % len(ids)].append(step_ms(model, ids, True, args.step_iters))
        steps["uniform_B1"].append(step_ms(model, uniform[:1], False, args.step_iters))
    result["decode_step_ms"] = {k: {"min": min(v), "all": v} for k, v in steps.items()}
    result["decode_step_prompt_length_uniform"] = common
    result["card_after"] = card(0)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
