"""bench.py — nucleotides/sec of the Evo-1 7B forward on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload 8k|131k|1k|32k|gen] [--impl ours|reference] [--dump-outputs DIR]

Workload "8k" (default, BASELINE.json configs[1]): evo-1-8k-base scoring forward, batch 8 x
8192 nt of synthetic uniform ACGT (+BOS => L = 8193), bf16, random-init weights of the 7B
architecture (no network for checkpoints).  One "step" = one forward over one batch.
  value : whole-job nt/s with the token ids already resident in HBM (model(input_ids)).
  e2e   : the same through the public API evo_b200.score_sequences(list[str]) -> list[float]:
          host strings -> pinned H2D -> forward -> fused log-softmax/gather -> D2H, per step.
N > 1 (torchrun, one rank per GPU): independent replicas of the workload, no data-path
collective (weak scaling); "131k" runs the sequence-parallel forward instead.
--impl reference: the reference's own CPU implementation of the path.  stripedhyena==0.2.2 is
not installable offline, so this arm times the oracle restatement (kind "port") on the host
cores, rank 0 only, on a bounded sample of the same workload.
--dump-outputs DIR: after the timed steps, rank 0 writes what the timed path returned in its last step as DIR/<name>.npy
(see dump_outputs), so that two builds can be compared output for output on the same seeded inputs and weights.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries ONE JSON line: NCCL's banner ("NCCL version ..." when the pod sets NCCL_DEBUG=VERSION) goes to stderr
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

WORKLOADS = {
    "8k": dict(model="evo-1-8k-base", batch=8, nt=8192, desc="evo-1-8k-base 7B scoring forward, batch 8 x 8192 nt (+BOS), bf16"),
    "1k": dict(model="evo-1-8k-base", batch=64, nt=1024, desc="evo-1-8k-base 7B scoring forward, batch 64 x 1024 nt (+BOS), bf16"),
    "32k": dict(model="evo-1-131k-base", batch=2, nt=32768, desc="evo-1-131k-base 7B forward, batch 2 x 32768 nt (+BOS), bf16"),
    "131k": dict(model="evo-1-131k-base", batch=1, nt=131072, desc="evo-1-131k-base 7B forward, batch 1 x 131072 nt, bf16"),
    # BASELINE configs[3] (secondary line, not the headline): cached generation, one step = one new nucleotide per sequence
    "gen": dict(model="evo-1.5-8k-base", batch=16, nt=4096, desc="evo-1.5-8k-base 7B cached generation, batch 16, prompt 4096 nt, greedy decode steps, bf16"),
}


def synthetic_seqs(batch, nt, seed=0):
    import numpy as np
    rng = np.random.default_rng(seed)
    return ["".join(rng.choice(list("ACGT"), size=nt)) for _ in range(batch)]


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"], "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


DUMP_ARRAY_BYTES = 16 << 20        # per array; a path returns at most two arrays, so a dump stays well under 64 MB


def dump_outputs(path, arrays):
    """Writes each array as `path`/<name>.npy: float32, or float64 for values the API hands back as host floats.  An array
    over DUMP_ARRAY_BYTES keeps a fixed sample of its rows (rows = all but the last dimension, chosen with seed 0, kept in
    row order), so the same shape always yields the same rows."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        a = a.detach().float().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a, dtype=np.float64)
        if a.nbytes > DUMP_ARRAY_BYTES:
            rows = a.reshape(-1, a.shape[-1])
            keep = DUMP_ARRAY_BYTES // (rows.shape[1] * a.itemsize)
            a = rows[np.sort(np.random.default_rng(0).choice(rows.shape[0], size=keep, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


def ncu_traffic(pattern, workload):
    """Average DRAM bytes per launch of the kernels matching `pattern`, from the committed ncu --set full
    capture of this workload (profiles/ncu_traffic_<workload>.json, made by tools/ncu_traffic.py); None if absent."""
    path = os.path.join(ROOT, "profiles", f"ncu_traffic_{workload}.json")
    if not os.path.exists(path):
        return None
    rows = [r for r in json.load(open(path))["launches"] if pattern in r["kernel"]]
    return sum(r["dram_bytes"] for r in rows) / len(rows) if rows else None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()

    def summary(self):
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(len(r) >= 6 and r[2 + j] == "Active" for r in self.rows)]
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons, "samples": len(sm)}


def cpu_baseline(model_name, target_seconds=15.0, threads=None):
    """Oracle (restatement of the reference, kind 'port') timed on the host cores on a bounded
    sample: batch 1 x L_s tokens of the same 7B forward, L_s sized for ~target_seconds.
    The reference keeps bf16 parameters on CPU too (evo/models.py:148), but host CPUs without
    AMX / AVX512-BF16 run bf16 GEMMs through a slow path (measured: 0.7 nt/s on a 128-core GPU
    host), so the arm first times one projection-sized GEMM in bf16 and fp32 and runs the forward
    in the faster dtype, with the thread count that GEMM prefers; both choices are reported."""
    import torch
    from oracle import stripedhyena_oracle as O
    import numpy as np
    ncpu = os.cpu_count() or 1

    def gemm_time(dtype, nthreads):
        torch.set_num_threads(nthreads)
        a, w = torch.randn(128, 4096).to(dtype), torch.randn(12288, 4096).to(dtype)
        torch.nn.functional.linear(a, w)
        t0 = time.perf_counter()
        torch.nn.functional.linear(a, w)
        return time.perf_counter() - t0

    cands = [(dt, nt) for dt in (torch.bfloat16, torch.float32) for nt in sorted({threads or ncpu, min(ncpu, 32)})]
    timed = sorted((gemm_time(dt, nt), str(dt), dt, nt) for dt, nt in cands)
    t_gemm, _, dtype, threads = timed[0]
    torch.set_num_threads(threads)
    cfg = O.evo_config(model_name)
    # the reference's own implementation when its package is importable (kind "reference"), else the oracle port (kind "port").
    # stripedhyena has not been importable on any box this ran on, so the first branch is exercised against a stand-in only
    # (oracle/real_reference.py, tests/test_oracle.py); any failure inside it falls back to the port and says why.
    kind, what, m = "port", "oracle (stripedhyena 0.2.2 restatement)", None
    try:
        from oracle import real_reference as RR
        ver = RR.available()
        if ver is not None:
            real = RR.build(cfg, None, dtype, share_blocks=True)
            m = lambda ids: RR._run(real, ids)
            kind, what = "reference", f"stripedhyena {ver} (torch branches: flash kernels off, rotary through apply_rotary_emb_torch)"
    except Exception as ex:          # noqa: BLE001
        what += f" [stripedhyena importable but unusable on CPU: {type(ex).__name__}: {str(ex)[:80]}]"
        m = None
    if m is None:
        sd = O.random_state_dict(cfg, seed=0, share_blocks=True)   # blocks alias one set of weights: same arithmetic, small RAM
        m = O.OracleStripedHyena(cfg, sd, dtype)
    rng = np.random.default_rng(0)

    def run(L):
        ids = torch.from_numpy(rng.choice(np.array([65, 67, 71, 84]), size=(1, L)))
        t0 = time.perf_counter()
        with torch.inference_mode():
            m(ids)
        return time.perf_counter() - t0

    run(16)                      # warm-up (thread pools, oneDNN primitives)
    t16 = run(16)                # measured probe: size the sample from a real forward, not from a model
    if t16 >= target_seconds / 2:
        L, t = 16, t16
    else:
        L = int(min(2048, 16 * target_seconds / t16))
        L = max(32, (L // 32) * 32)
        t = run(L)
        if t < 0.6 * target_seconds and L < 2048:          # throughput grows with L (weights amortised): resize once from the real run
            L = max(32, (int(min(2048, L * target_seconds / t)) // 32) * 32)
            t = run(L)
    return {"value": L / t, "unit": "nt/s", "cores": threads, "kind": kind, "host_cpus": ncpu, "cpu_dtype": str(dtype).replace("torch.", ""),
            "sample": f"{what} {str(dtype).replace('torch.', '')} on CPU, 7B shape, batch 1 x {L} nt, {t:.1f} s"}, m, run


def bench_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = args.steps if args.steps is not None else 3
    # one step = one bounded sample; the sample shrinks with the step count so that the whole arm stays near two minutes
    base, m, run = cpu_baseline(wl["model"], target_seconds=max(2.0, min(8.0, 100.0 / max(steps, 1))))
    L = int(base["sample"].split(" x ")[1].split(" nt")[0])
    for _ in range(args.warmup if args.warmup is not None else 1):
        run(min(L, 128))
    t0 = time.perf_counter()
    for _ in range(steps):
        run(L)
    dt = time.perf_counter() - t0
    v = steps * L / dt
    base["value"] = v
    print(json.dumps({
        "impl": "reference", "metric": "nucleotides/sec forward, evo-1 7B", "value": v, "unit": "nt/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": args.warmup if args.warmup is not None else 1, "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic uniform ACGT, random-init weights",
        "config": {"workload": wl["desc"], "note": "CPU arm: bounded sample; " + ("the reference's own package" if base["kind"] == "reference" else "stripedhyena not installable offline -> oracle port")},
        "cpu_baseline": base, "e2e": {"value": v, "unit": "nt/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def _dist_ctx():
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    torch.cuda.set_device(f"cuda:{local}")
    return world, rank, local


def _barrier(world):
    import torch
    import torch.distributed as dist
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def _max_over_ranks(x, world, dev):
    """(max over ranks, per-rank list) of a python float; device-side all-gather."""
    import torch
    import torch.distributed as dist
    if world == 1:
        return x, [x]
    t = torch.tensor([x], device=dev, dtype=torch.float64)
    allt = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(allt, t)
    vals = [float(v.item()) for v in allt]
    return max(vals), vals


def time_steps(fwd, steps, world, dev):
    """EXACTLY `steps` calls of fwd, CUDA events on the launch stream, barrier + synchronize on both sides.
    No per-kernel instrumentation runs inside this region.  Returns (max ms over ranks, per-rank ms, last step's result)."""
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = None
    _barrier(world)
    e0.record()
    for _ in range(steps):
        out = fwd()
    e1.record()
    _barrier(world)
    return (*_max_over_ranks(e0.elapsed_time(e1), world, dev), out)


def kernel_breakdown(model, fwd, n, world):
    """Separate pass (outside the timed region): per-kernel CUDA events -> {kind: [work, ms, launches]} per step, and the pass's own ms/step."""
    import torch
    _barrier(world)
    model._prof = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fwd()
    e1.record()
    _barrier(world)
    prof, model._prof = model._prof, None
    by = {}
    for kind, work, a, b in prof:
        key = kind if kind.startswith("comm/") else kind.split("/")[0]
        d = by.setdefault(key, [0.0, 0.0, 0])
        d[0] += work / n; d[1] += a.elapsed_time(b) / n; d[2] += 1.0 / n
    return by, e0.elapsed_time(e1) / n


def rooflines(by, step_ms, workload, peaks):
    roof = {}
    if "gemm" in by:
        ach = by["gemm"][0] / (by["gemm"][1] / 1e3) / 1e12
        roof["roofline"] = {"kernel": "gemm_tcgen05_kernel (all linear layers)", "bound": "tensor", "achieved": ach, "peak": peaks["bf16_tflops_sustained"],
                            "unit": "TFLOP/s", "frac": ach / peaks["bf16_tflops_sustained"], "traffic": ncu_traffic("gemm_tcgen05", workload),
                            "algorithmic_flops_per_launch": by["gemm"][0] / by["gemm"][2],
                            "peak_source": peaks["source"] + " (sustained cuBLAS bf16)", "share_of_step": by["gemm"][1] / step_ms, "launches_per_step": by["gemm"][2]}
    if "hyena" in by:
        ach = by["hyena"][0] / (by["hyena"][1] / 1e3) / 1e9
        roof["roofline_hyena"] = {"kernel": "hyena_scan_ms_kernel (fused FIR + gate + modal long conv + gate)", "bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"],
                                  "unit": "GB/s", "frac": ach / peaks["hbm_gbs"], "traffic": ncu_traffic("hyena_scan", workload),
                                  "algorithmic_bytes_per_launch": by["hyena"][0] / by["hyena"][2], "peak_source": peaks["source"],
                                  "share_of_step": by["hyena"][1] / step_ms, "launches_per_step": by["hyena"][2]}
    if "attn" in by:
        ach = by["attn"][0] / (by["attn"][1] / 1e3) / 1e12
        roof["roofline_attn"] = {"kernel": "attn_pp_kernel (tcgen05 causal attention)", "bound": "tensor", "achieved": ach, "peak": peaks["bf16_tflops_sustained"],
                                 "unit": "TFLOP/s", "frac": ach / peaks["bf16_tflops_sustained"], "traffic": ncu_traffic("attn_", workload),
                                 "share_of_step": by["attn"][1] / step_ms, "launches_per_step": by["attn"][2]}
    return roof


def variant_of(model, model_name):
    """A second StripedHyena that SHARES every parameter and packed weight of `model` under another config (the Evo
    checkpoints have one geometry; evo-1-131k-base only adds the rotary interpolation, evo/configs/evo-1-131k-base_inference.yml:39-40)."""
    import copy
    from evo_b200.configs import get_config
    from evo_b200.stripedhyena import dotdict
    model._ensure_packed()
    m = copy.copy(model)
    m.config = dotdict(get_config(model_name))
    m._rope, m._decode, m._prof = None, None, None
    for attr in ("_peer_carry", "_peer_ulysses"):          # symmetric-memory state belongs to the (shape, config) it was built for
        if hasattr(m, attr):
            delattr(m, attr)
    return m


def sp131k_record(model8k, world, rank, dev, steps, warmup, peaks):
    """BASELINE.json configs[2]: evo-1-131k-base, batch 1 x 131072 nt, the sequence sharded over the `world` GPUs of the
    box (strong scaling; world == 1: the plain single-GPU forward).  Timed like the main line; afterwards, outside the
    timed region, one instrumented step names where the time went (kernels and every communication piece) and every
    rank compares its shard of the logits with the UNSHARDED single-GPU forward of the same ids."""
    import torch
    import torch.distributed as dist
    from evo_b200 import CharLevelTokenizer, prepare_batch
    wl = WORKLOADS["131k"]
    model = variant_of(model8k, wl["model"])
    tok = CharLevelTokenizer(512)
    seqs = synthetic_seqs(wl["batch"], wl["nt"], seed=1234)                 # same ids on every rank
    ids_full, _ = prepare_batch(seqs, tok, prepend_bos=False, device=dev)
    L = ids_full.shape[1]
    if world > 1:
        from evo_b200.parallel import sequence_parallel_forward
        shard = L // world
        ids = ids_full[:, rank * shard:(rank + 1) * shard].contiguous()
        fwd = lambda: sequence_parallel_forward(model, ids, rank, world)
    else:
        shard = L
        fwd = lambda: model(ids_full)[0]
    for _ in range(warmup):
        fwd()
    ms, per_rank, _ = time_steps(fwd, steps, world, dev)
    by, prof_ms = kernel_breakdown(model, fwd, 1, world)
    rec = {"workload": wl["desc"], "value": wl["batch"] * wl["nt"] * steps / (ms / 1e3), "unit": "nt/s", "ms_per_step": ms / steps, "steps": steps, "warmup": warmup,
           "parallelism": f"sp{world}", "scaling": "strong", "per_rank_ms_per_step": [v / steps for v in per_rank], "tokens_per_rank": shard}
    if world > 1:
        tr = getattr(model, "_peer_carry", None)
        rec["hyena_carry_transport"] = "nvlink peer stores + flags (own kernels)" if tr not in (None, False) else "nccl all-gather"
        rec["attention_reshard"] = ("nvlink peer stores fused into the Wqkv GEMM / attention epilogues + flag rounds (own kernels)"
                                    if getattr(model, "_peer_ulysses", None) is not None else "nccl all_to_all (Ulysses) + permute copies")
    # rank 0's instrumented step: kernels and communication, each as ms per step; what no event covered is host-side gaps
    comm = {k.split("/", 1)[1]: v[1] for k, v in by.items() if k.startswith("comm/")}
    kern = {k: v[1] for k, v in by.items() if not k.startswith("comm/")}
    rec["comm_ms"] = {**comm, "total": sum(comm.values())}
    rec["kernel_ms"] = kern
    rec["instrumented_step_ms"] = prof_ms
    rec["unattributed_ms"] = prof_ms - sum(comm.values()) - sum(kern.values())
    rec.update(rooflines(by, prof_ms, "131k", peaks))
    if world > 1:
        # correctness of the sharded forward on THIS run: my shard vs the unsharded forward of the same ids on my GPU
        mine = fwd()
        ref = model(ids_full)[0][:, rank * shard:(rank + 1) * shard]
        d = (mine.float() - ref.float()).abs()
        stats = [d.max().item(), d.mean().item(), (mine.argmax(-1) == ref.argmax(-1)).float().mean().item(), ref.float().abs().max().item(),
                 float(torch.isfinite(mine.float()).all().item())]
        del mine, ref, d
        allst = [None] * world
        dist.all_gather_object(allst, stats)
        rec["sp_check"] = {"reference": "unsharded forward of the same ids on each rank's own GPU",
                           "per_rank": [{"max_abs": s[0], "mean_abs": s[1], "argmax_agree": s[2], "ref_abs_max": s[3], "finite": bool(s[4])} for s in allst]}
    torch.cuda.empty_cache()
    return rec


def sweep_record(model8k, dev, steps=3, warmup=1):
    """BASELINE.json configs[4] at one GPU: the same 65 536-token budget as 1k and 32k sequences (8k is the headline `value`,
    131k the `sp131k` record).  nt/s with ids resident in HBM, CUDA events around `steps` forwards."""
    import torch
    from evo_b200 import CharLevelTokenizer, prepare_batch
    tok = CharLevelTokenizer(512)
    out = {}
    for key in ("1k", "32k"):
        wl = WORKLOADS[key]
        m = model8k if wl["model"] == "evo-1-8k-base" else variant_of(model8k, wl["model"])
        ids, _ = prepare_batch(synthetic_seqs(wl["batch"], wl["nt"], seed=7), tok, prepend_bos=True, device=dev)
        fwd = lambda: m(ids)
        for _ in range(warmup):
            fwd()
        ms, _, _ = time_steps(fwd, steps, 1, dev)
        out[key] = {"workload": wl["desc"], "value": wl["batch"] * wl["nt"] * steps / (ms / 1e3), "unit": "nt/s", "ms_per_step": ms / steps, "steps": steps, "warmup": warmup}
        del ids
        torch.cuda.empty_cache()
    return out


def bench_ours(args, wl):
    import torch
    import torch.distributed as dist
    import evo_b200
    from evo_b200 import _lib, CharLevelTokenizer, prepare_batch, score_sequences
    from evo_b200.models import load_checkpoint

    world, rank, local = _dist_ctx()
    dev = f"cuda:{local}"
    steps = args.steps if args.steps is not None else 5
    warmup = args.warmup if args.warmup is not None else 3

    model = load_checkpoint(wl["model"], device=dev, random_init=True, seed=0)
    tok = CharLevelTokenizer(512)
    seqs = synthetic_seqs(wl["batch"], wl["nt"], seed=rank)
    seqpar = args.workload == "131k" and world > 1
    if seqpar:
        from evo_b200.parallel import sequence_parallel_forward
        ids_full, _ = prepare_batch(synthetic_seqs(wl["batch"], wl["nt"], seed=0), tok, prepend_bos=False, device=dev)
        shard = ids_full.shape[1] // world
        ids = ids_full[:, rank * shard:(rank + 1) * shard].contiguous()
        fwd = lambda: sequence_parallel_forward(model, ids, rank, world)
        tokens_per_step_job = wl["batch"] * wl["nt"]
    else:
        ids, _ = prepare_batch(seqs, tok, prepend_bos=True, device=dev)
        fwd = lambda: model(ids)
        tokens_per_step_job = wl["batch"] * wl["nt"] * world

    for _ in range(warmup):
        fwd()
    _barrier(world)

    # ---- timed region 1: device-resident inputs, nothing but the forward inside
    lib = _lib.lib()
    lib.evo_reset_launch_count()
    with ClockSampler(local) as clocks:
        ms, per_rank_ms, last = time_steps(fwd, steps, world, dev)
    launches = lib.evo_launch_count()
    value = tokens_per_step_job * steps / (ms / 1e3)
    dumped = {"logits": last[0] if isinstance(last, tuple) else last}
    del last

    # ---- separate pass: per-kernel events for the rooflines (not part of `value`)
    by, prof_ms = kernel_breakdown(model, fwd, 2, world)

    # ---- timed region 2: end to end through the public API with host inputs
    e2e = None
    if not seqpar:
        for _ in range(2):
            score_sequences(seqs, model, tok, device=dev)
        _barrier(world)
        t0 = time.perf_counter()
        for _ in range(steps):
            scores = score_sequences(seqs, model, tok, device=dev)
        torch.cuda.synchronize()
        dt, _ = _max_over_ranks(time.perf_counter() - t0, world, dev)
        L1 = wl["nt"] + 1
        e2e = {"value": tokens_per_step_job * steps / dt, "unit": "nt/s",
               "h2d_bytes_per_step": wl["batch"] * L1 * 8, "d2h_bytes_per_step": wl["batch"] * wl["nt"] * 4,
               "api": "evo_b200.score_sequences(list[str]) -> list[float]"}
        dumped["e2e_scores"] = scores
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dumped)
    del dumped

    peaks = measured_peaks()
    sub = {}
    if args.workload == "8k" and not args.no_sub:
        # BASELINE.json configs[2] next to the headline, at every N (VERDICT r1 item 1)
        try:
            sub["sp131k"] = sp131k_record(model, world, rank, dev, steps=args.sub_steps, warmup=1, peaks=peaks)
        except Exception as ex:  # noqa  (a failed sub-record must not cost the headline line)
            sub["sp131k"] = {"error": repr(ex)[:300]}
        if world == 1 and not args.no_gen:
            try:
                sub["gen"] = generate_record(model, dev, peaks)
            except Exception as ex:  # noqa
                sub["gen"] = {"error": repr(ex)[:300]}
        if world == 1:
            try:
                sub["sweep"] = sweep_record(model, dev)
            except Exception as ex:  # noqa
                sub["sweep"] = {"error": repr(ex)[:300]}

    if rank == 0:
        roof = rooflines(by, prof_ms, args.workload, peaks)
        out = {
            "metric": "nucleotides/sec forward, evo-1 7B", "value": value, "unit": "nt/s", "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "strong" if seqpar else "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic uniform ACGT (np.random.default_rng), random-init weights of the 7B architecture",
            "config": {"workload": wl["desc"], "global_batch": wl["batch"] * (1 if seqpar else world), "seq_len": wl["nt"] + (0 if seqpar else 1),
                       "parallelism": (f"sp{world}" if seqpar else f"replicas x{world}"),
                       "l2": "inputs >> L2: every step streams 12.9 GB of weights and 0.5-1.6 GB activation tensors (L2 = 126 MB)",
                       "timing": "value: CUDA events around exactly `steps` forwards, no per-kernel events inside; rooflines from a separate instrumented pass"},
            "per_rank_ms_per_step": [v / steps for v in per_rank_ms],
            "clocks": clocks.summary(), "gpu_launches": int(launches), "e2e": e2e, **roof, **sub,
        }
        if world == 1 and not args.no_cpu_baseline:
            try:
                out["cpu_baseline"] = cpu_baseline(wl["model"])[0]
            except Exception as ex:  # noqa
                out["cpu_baseline"] = {"error": str(ex)[:200]}
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def generate_record(model, dev, peaks, steps=64, warmup=4, n_new=None, world=1, rank=0, outputs=None):
    """BASELINE.json configs[3]: cached generation, batch 16, prompt 4096 nt, greedy.  One step = one new nucleotide per
    sequence through the L == 1 path (recurrent Hyena state + KV cache).
    value = generated nt/s with the state resident on the GPU; e2e = evo_b200.generate() from prompt strings to generated
    strings, the 4096-nt prefill and `n_new` decode steps included.  `outputs` (a dict) receives the last timed step's
    logits and greedy next tokens."""
    import torch
    import evo_b200
    from evo_b200 import _lib, CharLevelTokenizer
    wl = WORKLOADS["gen"]
    tok = CharLevelTokenizer(512)
    B, P = wl["batch"], wl["nt"]
    n_new = n_new if n_new is not None else P          # configs[3]: prefill 4096 + decode 4096
    seqs = synthetic_seqs(B, P, seed=rank)
    ids = torch.tensor([tok.tokenize(s) for s in seqs], dtype=torch.long, device=dev)
    d = model.initialize_inference_params()
    d["mha"].max_batch_size = d["hyena"].max_batch_size = B
    logits, d = model(ids, inference_params_dict=d)
    d["mha"].seqlen_offset = d["hyena"].seqlen_offset = P
    state = {"nxt": logits[:, -1].argmax(-1, keepdim=True), "d": d}

    def step():
        state["lg"], state["d"] = model(state["nxt"], inference_params_dict=state["d"])
        state["nxt"] = state["lg"][:, -1].argmax(-1, keepdim=True)
        state["d"]["mha"].seqlen_offset += 1
        state["d"]["hyena"].seqlen_offset += 1

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    lib = _lib.lib()
    n0 = lib.evo_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    launches = lib.evo_launch_count() - n0
    if world > 1:
        ms, _ = _max_over_ranks(ms, world, dev)
    if outputs is not None:
        outputs.update(logits=state["lg"], next_token=state["nxt"])
    del state, d, logits
    torch.cuda.empty_cache()
    # end to end: prompts as strings -> generated strings through the reference-shaped API (prefill + n_new steps)
    evo_b200.generate(seqs, model, tok, n_tokens=4, top_k=1, cached_generation=True, verbose=0, device=dev, force_prompt_threshold=P)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    evo_b200.generate(seqs, model, tok, n_tokens=n_new, top_k=1, cached_generation=True, verbose=0, device=dev, force_prompt_threshold=P)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    cfg = model.config
    n_attn = len(cfg.attn_layer_idxs)
    weight_bytes = sum(p.numel() * p.element_size() for p in model.parameters())
    ctx = P + warmup + steps / 2.0
    kv_bytes = n_attn * B * ctx * 2 * cfg.hidden_size * 2
    ach = (weight_bytes + kv_bytes) / (ms / steps / 1e3) / 1e9
    torch.cuda.empty_cache()
    return {
        "metric": "generated nucleotides/sec, evo-1.5 7B cached decode", "workload": wl["desc"], "value": B * world * steps / (ms / 1e3), "unit": "nt/s",
        "steps": steps, "warmup": warmup, "ms_per_step": ms / steps, "gpu_launches": int(launches),
        "decode": {"streamk": model.decode_streamk, "pdl": model.decode_pdl, "cuda_graph": model.decode_graph},
        "e2e": {"value": B * world * n_new / dt, "unit": "nt/s", "seconds": dt, "new_tokens": n_new, "h2d_bytes": B * P * 8, "d2h_bytes": B * n_new * (8 + 512 * 4),
                "api": f"evo_b200.generate(prompts, n_tokens={n_new}, top_k=1, cached_generation=True, force_prompt_threshold={P}): {P}-nt prefill + {n_new} steps, strings in / strings out"},
        "roofline": {"kernel": "decode step (gemm_smallm_kernel weight stream + decode_attn_tma_kernel KV stream)", "bound": "hbm", "achieved": ach,
                     "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"], "traffic": None,
                     "algorithmic_bytes_per_step": weight_bytes + kv_bytes, "peak_source": peaks["source"]},
    }


def bench_generate(args, wl):
    """`--workload gen`: the generation record as its own bench line (replicas when N > 1)."""
    import torch
    import torch.distributed as dist
    from evo_b200.models import load_checkpoint
    world, rank, local = _dist_ctx()
    dev = f"cuda:{local}"
    steps = args.steps if args.steps is not None else 64
    warmup = max(3, args.warmup if args.warmup is not None else 4)
    model = load_checkpoint(wl["model"], device=dev, random_init=True, seed=0)
    dumped = {}
    with ClockSampler(local) as clocks:
        rec = generate_record(model, dev, measured_peaks(), steps=steps, warmup=warmup, n_new=args.gen_tokens, world=world, rank=rank, outputs=dumped)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dumped)
    del dumped
    if rank == 0:
        out = {"metric": rec.pop("metric"), "value": rec.pop("value"), "unit": rec.pop("unit"), "n_gpus": world, "steps": steps, "warmup": warmup,
               "ms_per_step": rec.pop("ms_per_step"), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
               "data": "synthetic uniform ACGT prompts, random-init weights of the 7B architecture",
               "config": {"workload": rec.pop("workload"), "global_batch": wl["batch"] * world, "seq_len": wl["nt"], "parallelism": f"replicas x{world}",
                          "l2": "every step streams 12.9 GB of weights and ~3.2 GB of KV cache (L2 = 126 MB)", "decode": rec.pop("decode")},
               "clocks": clocks.summary(), **rec}
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="8k", choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sub", action="store_true", help="default workload only: skip the sp131k / gen sub-records")
    ap.add_argument("--no-gen", action="store_true", help="skip the cached-generation sub-record")
    ap.add_argument("--sub-steps", type=int, default=3, help="timed steps of the 131k sub-record")
    ap.add_argument("--gen-tokens", type=int, default=None, help="new tokens of the end-to-end generate() run (default: 4096 = BASELINE configs[3])")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's outputs as DIR/<name>.npy (float32/float64, < 64 MB)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        bench_reference(args, wl)
    elif args.workload == "gen":
        bench_generate(args, wl)
    else:
        bench_ours(args, wl)


if __name__ == "__main__":
    main()
