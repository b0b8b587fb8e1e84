#!/usr/bin/env python
"""Flagship benchmark: Llama-3-8B, FSDP (ZeRO-3) + gradient checkpointing, bf16, seq 4096, synthetic tokens.

    python bench.py --gpus N --steps K --warmup W            # ours (torchrun launches N ranks for N > 1)
    python bench.py --impl reference --gpus N ...            # unmodified reference from baseline/_ref
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/*.npy

Metric (BASELINE.json): training tokens/s for the WHOLE job, device-timed with CUDA events, max over ranks.
Weak scaling: the per-GPU batch is fixed (``--mbs``, default 2 sequences of 4096 tokens).
Each timed step = forward + backward + global grad-norm clip + AdamW update (nothing skipped, full 32 layers).
One JSON line is printed by rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

A100_TOKENS_PER_S_PER_GPU = 4044.8   # BASELINE.md row 1 (8x A100-80G, TorchAcc XLA-FSDP, seq 4096)


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=5)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference", "torch_fsdp"],
                   help="ours | reference (UNMODIFIED reference, stock path) | torch_fsdp (NOT the reference: the stack "
                        "the reference's eager FSDP path would build -- torch FSDP1 + its kernel patches -- so that "
                        "N > 1 has a same-box competitor; see DESIGN.md section 4)")
    p.add_argument("--fp8", action="store_true",
                   help="ours: Config.compute.fp8 (MX-FP8 block-scaled linear layers).  Lower precision than the "
                        "reference arm: reported as its own config, never as the headline")
    p.add_argument("--hf", action="store_true",
                   help="ours: run the SAME HuggingFace LlamaForCausalLM object as the reference arm through "
                        "ta.accelerate (kernel patches + FSDP engine) instead of the native model definition")
    p.add_argument("--model", default="llama3-8b")
    p.add_argument("--seq-len", type=int, default=4096)
    p.add_argument("--mbs", type=int, default=2, help="sequences per GPU per step")
    p.add_argument("--layers", type=int, default=None, help="debug only: override the layer count (invalidates the number)")
    p.add_argument("--no-gc", action="store_true")
    p.add_argument("--attn", default=None, help="attention backend override (native|sdpa)")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--trace", default=None, help="write a kernel timeline (chrome trace) of one extra, untimed step")
    p.add_argument("--no-comm-trace", action="store_true",
                   help="skip the extra profiled step that measures exposed communication when N > 1")
    p.add_argument("--dump-outputs", default=None, metavar="DIR",
                   help="ours: after the timed steps write what the last one computed as DIR/<name>.npy (loss, "
                        "gradient norm, a fixed sample of the updated weights) to compare two builds output for output")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        p.error("--dump-outputs is only implemented for --impl ours")
    return a


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self._stop = index, [], threading.Event()
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self.t.start()
        return self

    def stop(self) -> dict:
        self._stop.set()
        self.t.join(timeout=3)
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


def bench_config(a, world, layers):
    """The ``config`` object of the JSON line: identical in every arm (the driver compares them)."""
    return {"model": a.model, "global_batch": a.mbs * world, "seq_len": a.seq_len,
            "parallelism": f"fsdp{world}" + ("" if a.no_gc else "+gc"), "layers": layers,
            "l2": "no explicit flush: each step streams >16 GB of weights/activations (>> 126 MB L2)"}


METRIC = "Llama-3-8B FSDP bf16 training throughput (whole job, device-timed, max over ranks)"

PARAM_SAMPLE = 8192     # positions per parameter in --dump-outputs: 1.33M fp32 values (5.3 MB) for Llama-3-8B


def dump_outputs(out_dir, model, last, rank, world):
    """Write what the last timed step computed: its loss, its gradient norm before clipping and the updated fp32
    master weights -- of every parameter all of it, or PARAM_SAMPLE seeded positions when it is larger.  Parameters
    are taken in the order of their names, so the sample does not depend on how the engine groups them into flat
    shards; each rank contributes the positions it owns and a sum over ranks assembles the whole sample."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from torchacc_b200.parallel.state_dict_utils import get_shard_metadata
    meta = get_shard_metadata(model.engine)
    params = sorted(((um["prefix"] + "." if um["prefix"] else "") + p["fqn"], p, um["shard_numel"], shard)
                    for um, shard in zip(meta["units"], model.parameters()) for p in um["params"])
    g = torch.Generator().manual_seed(0)
    parts = []
    with torch.no_grad():
        for _, p, shard_numel, shard in params:
            n = p["numel"]
            idx = torch.arange(n) if n <= PARAM_SAMPLE else \
                torch.randint(0, n, (PARAM_SAMPLE,), generator=g).sort().values
            pos = (p["offset"] - meta["rank"] * shard_numel + idx).to(shard.device)
            own = (pos >= 0) & (pos < shard_numel)
            parts.append(torch.where(own, shard[pos.clamp(0, shard_numel - 1)], 0.0))
        weights = torch.cat(parts)
        if world > 1:
            dist.all_reduce(weights)
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        outs = {"loss": last["loss"], "grad_norm": last["grad_norm"], "weights_sample": weights}
        for name, t in outs.items():
            np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy())


def hf_llama(a, torch, device, world):
    """HuggingFace Llama-3-8B (random init, same distributions as the native arm) -- the model object the reference
    arm, the torch_fsdp arm and ``--hf`` all run."""
    from transformers import LlamaConfig, LlamaForCausalLM
    hf = LlamaConfig(vocab_size=128256, hidden_size=4096, intermediate_size=14336,
                     num_hidden_layers=a.layers or 32, num_attention_heads=32, num_key_value_heads=8,
                     max_position_embeddings=max(a.seq_len, 8192), rope_theta=500000.0, rms_norm_eps=1e-5,
                     tie_word_embeddings=False, attn_implementation="flash_attention_2", use_cache=False)
    torch.manual_seed(1234)
    with torch.device("meta"):
        model = LlamaForCausalLM(hf)
    model = model.to_empty(device="cpu" if world > 1 else device)
    with torch.no_grad():
        for p in model.parameters():
            if p.dim() == 1:
                p.fill_(1.0)            # RMSNorm weights (same initialisation as our arm)
            else:
                p.normal_(0, 0.02)
    return model, hf


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


def timed_loop(step_fn, steps, warmup, device, world):
    import torch
    import torch.distributed as dist
    for _ in range(warmup):
        step_fn()

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[device.index])
        torch.cuda.synchronize(device)

    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step_fn()
    e1.record()
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=device)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms)


# ----------------------------------------------------------------------------------------------------------------
# our implementation
# ----------------------------------------------------------------------------------------------------------------
def run_ours(a):
    import torch
    import torch.distributed as dist
    import torchacc_b200 as ta
    from torchacc_b200 import _native as nat
    from torchacc_b200.models import build_llama, llama_config

    rank, local_rank, world = dist_env()
    assert world == a.gpus, f"--gpus {a.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    if a.attn:
        ta.ops.set_attention_backend(a.attn)

    over = {}
    if a.layers is not None:
        over["num_hidden_layers"] = a.layers
    mcfg = llama_config(a.model, max_position_embeddings=max(a.seq_len, 8192), **over)
    torch.manual_seed(1234)
    if a.hf:
        if world > 1:
            ta.dist.init_process_group()
        model, _ = hf_llama(a, torch, device, 1)        # built on the device: 16 GB of bf16 per rank
        model = model.to(torch.bfloat16)
    else:
        with torch.device(device):
            model = build_llama(mcfg, dtype=torch.bfloat16)

    cfg = ta.Config()
    cfg.compute.bf16 = True
    cfg.compute.fp8 = bool(a.fp8)
    cfg.memory.gc = not a.no_gc
    cfg.memory.gc_cls = {"LlamaDecoderLayer"}
    cfg.dist.fsdp.size = world
    cfg.dist.fsdp.wrap_layer_cls = {"LlamaDecoderLayer"}

    # synthetic data: random tokens, pinned host memory (e2e loop uploads them every step through AsyncLoader)
    g = torch.Generator().manual_seed(rank)
    n_batches = a.warmup + a.steps + 2
    host = [{"input_ids": torch.randint(0, mcfg.vocab_size, (a.mbs, a.seq_len), generator=g).pin_memory()}
            for _ in range(4)]
    for b in host:
        b["labels"] = b["input_ids"]

    class Synth:
        def __len__(self):
            return n_batches

        def __iter__(self):
            for i in range(n_batches):
                yield host[i % len(host)]

    model, loader = ta.accelerate(model, Synth(), cfg)
    opt = ta.optim.FusedAdamW(model.parameters(), lr=1e-5, betas=(0.9, 0.95), weight_decay=0.1)

    dev_batch = {k: v.to(device) for k, v in host[0].items()}
    last = {}

    def step(batch=dev_batch):
        out = model(**batch)
        loss = out["loss"]
        loss.backward()
        last["grad_norm"] = model.clip_grad_norm_(1.0)
        opt.step()
        model.zero_grad()
        last["loss"] = loss
        return loss

    # ---- device-timed region --------------------------------------------------------------------------------
    sampler = None
    for _ in range(a.warmup):
        step()
    torch.cuda.synchronize(device)
    if rank == 0:
        sampler = ClockSampler(local_rank).start()
    l0 = nat.LAUNCHES
    ms = timed_loop(step, a.steps, 0, device, world)
    launches = nat.LAUNCHES - l0
    clocks = sampler.stop() if sampler else None
    tokens = a.mbs * a.seq_len * world * a.steps
    value = tokens / (ms / 1e3)
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, model, last, rank, world)     # before any further step changes the weights

    # ---- end-to-end through the public API: AsyncLoader H2D every step + loss D2H every step ---------------------
    e2e = None
    if not a.no_e2e:
        it = iter(loader)
        for _ in range(2):
            float(step(next(it)))
        if world > 1:
            dist.barrier(device_ids=[device.index])
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.steps):
            loss_val = float(step(next(it)))          # device -> host read of the step's loss
        e1.record()
        torch.cuda.synchronize(device)
        wall = (time.perf_counter() - t0) * 1e3
        ems = torch.tensor([max(e0.elapsed_time(e1), wall)], device=device)
        if world > 1:
            dist.all_reduce(ems, op=dist.ReduceOp.MAX)
        e2e = {"value": tokens / (float(ems) / 1e3), "unit": "tokens/s",
               "h2d_bytes_per_step": int(2 * a.mbs * a.seq_len * 8), "d2h_bytes_per_step": 4,
               "last_loss": loss_val}

    comm = None
    if a.trace or (world > 1 and not a.no_comm_trace):
        # one extra step under the CUPTI-based torch profiler, AFTER every timed region (never part of a number):
        # gives the exposed-communication figure of BASELINE.json's metric (communication-kernel time not hidden
        # behind compute kernels, rank 0's timeline).  tools/trace_summary.py prints the full tables for profiles/.
        # every rank runs exactly one more step whatever happens to the profiler (a rank that skipped it would
        # leave its peers waiting inside the collectives)
        prof = None
        try:
            from torch.profiler import ProfilerActivity, profile
            torch.cuda.synchronize(device)
            prof = profile(activities=[ProfilerActivity.CUDA])
            prof.__enter__()
        except Exception as e:  # noqa: BLE001
            prof, comm = None, {"error": f"profiler unavailable: {type(e).__name__}: {e}"[:200]}
        step()
        torch.cuda.synchronize(device)
        if prof is not None:
            try:
                prof.__exit__(None, None, None)
                if rank != 0 and a.trace and os.environ.get("TORCHACC_B200_TRACE_ALL", "0") == "1":
                    prof.export_chrome_trace(a.trace.replace(".json", f".rank{rank}.json"))   # skew diagnostics
                if rank == 0:
                    path = a.trace or os.path.join("/tmp", f"tb_bench_trace_{os.getpid()}.json")
                    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
                    prof.export_chrome_trace(path)
                    sys.path.insert(0, os.path.join(ROOT, "tools"))
                    from trace_summary import comm_exposure
                    comm = {k: round(v, 3) for k, v in comm_exposure(path).items()}
                    if not a.trace:
                        os.remove(path)
            except Exception as e:  # noqa: BLE001  -- diagnostics must never break the benchmark line
                comm = {"error": f"{type(e).__name__}: {e}"[:200]}

    dbg_path = os.environ.get("TORCHACC_B200_CARRY_DEBUG", "")
    if dbg_path and world > 1:
        # in-kernel timestamps of the copy warp of CTA 0 for every carrying GEMM launch of ONE extra (untimed) step
        nrec = 4096
        buf = torch.zeros(nrec * 8, dtype=torch.int64, device=device)
        L = nat.require()
        L.tb_carry_set_debug(buf.data_ptr(), nrec)
        step()
        torch.cuda.synchronize(device)
        used = L.tb_carry_set_debug(0, 0)
        rec = buf.view(nrec, 8)[:used].cpu().tolist()
        with open(dbg_path.replace(".json", f".rank{rank}.json"), "w") as f:
            json.dump({"fields": ["start", "s0_entry", "s0_done", "s1_entry", "s1_done", "chunks", "kinds", "end"],
                       "records": rec}, f)
    carry_counters = None
    try:
        from torchacc_b200.parallel.carry import CarryRuntime, available
        if world > 1 and available():
            carry_counters = CarryRuntime.counters()
    except Exception:  # noqa: BLE001
        pass
    if rank == 0:
        res = {
            "metric": METRIC,
            "value": value, "unit": "tokens/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": value / (A100_TOKENS_PER_S_PER_GPU * world),
            "dtype": "mxfp8 linears (e4m3 + ue8m0/32), bf16 elsewhere" if a.fp8 else "bf16", "data": "synthetic",
            "impl": "ours",
            "config": dict(bench_config(a, world, mcfg.num_hidden_layers), **({"fp8": True} if a.fp8 else {})),
            "detail": {"model_code": "HF LlamaForCausalLM through ta.accelerate" if a.hf else "native build_llama",
                       "optimizer": "FusedAdamW + clip_grad_norm(1.0)", "attention": ta.ops.get_attention_backend(),
                       "stack": "torchacc_b200: own FSDP engine + tcgen05 GEMM/attention + symmetric-memory collectives",
                       "engine_stats": dict(getattr(getattr(model, "engine", None), "stats", {}) or {}),
                       "carried_collectives": carry_counters},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "comm": comm,
            "mfu_model_flops": mcfg.flops_per_token(a.seq_len) * value / world / 1e12,
            "loss": float(last["loss"]),
        }
        print(json.dumps(res), flush=True)
    if world > 1:
        dist.barrier(device_ids=[device.index])
        dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------------------------
# reference arm: unmodified AlibabaPAI/torchacc from baseline/_ref, its own public API and eager code path
# ----------------------------------------------------------------------------------------------------------------
def run_reference(a):
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    rank, local_rank, world = dist_env()

    def unavailable(why):
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": why}), flush=True)
        sys.exit(0)

    if not os.path.isdir(os.path.join(ref_dir, "torchacc")):
        unavailable("baseline/_ref/torchacc not installed (see DESIGN.md: offline install outcome)")
    sys.path.insert(0, ref_dir)
    sys.path.insert(0, os.path.join(ROOT, "baseline", "shims"))   # stand-in for the missing `accelerate` dependency
    try:
        import torch
        import torch.distributed as dist
        # transformers first: importing the reference clears torch's decomposition tables at import time
        # (torchacc/__init__.py:137 -> utils/decompose.py), which breaks a later `import transformers` on torch 2.11
        from transformers import LlamaConfig, LlamaForCausalLM
        import transformers.models.llama.modeling_llama  # noqa: F401
        import transformers.modeling_flash_attention_utils  # noqa: F401
        import torchacc as ref_ta
    except Exception as e:  # noqa: BLE001
        unavailable(f"import failed: {type(e).__name__}: {e}"[:300])

    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    LAZY_MSG = ("reference eager backend cannot run on >1 rank: Config.get_mesh() asserts the XLA 'lazy' "
                "process-group backend (torchacc/config.py:396-398) after accelerate() initialised 'nccl' "
                "(dist/__init__.py:45-51); the lazy backend needs torch_xla, which cannot be installed offline")
    if world > 1:
        # the first two things reference accelerate() does for a distributed config (accelerate.py:69-71 and
        # dist/parallel_module.py -> config.get_mesh()), run BEFORE paying for an 8B-parameter model on every rank
        try:
            probe = ref_ta.Config()
            probe.backend = "eager"
            probe.dist.fsdp.size = world
            ref_ta.dist.init_process_group(probe)
            probe.get_mesh()
        except AssertionError as e:
            if dist.is_initialized():
                dist.destroy_process_group()
            unavailable(LAZY_MSG if "should be lazy" in str(e) else f"setup failed: AssertionError: {e}"[:400])
        except Exception as e:  # noqa: BLE001
            if dist.is_initialized():
                dist.destroy_process_group()
            unavailable(f"setup failed: {type(e).__name__}: {e}"[:400])
    try:
        model, hf = hf_llama(a, torch, device, world)
        # transformers 5.x builds `SiLUActivation` objects; the reference's liger MLP patch only accepts `nn.SiLU`
        # (torchacc/ops/liger.py:21-24).  Swapping the activation OBJECT on the user's model keeps the reference's
        # kernel patches active (the alternative, config.compute.disable_kernel_patches, would slow the reference).
        for m in model.modules():
            if type(getattr(m, "act_fn", None)).__name__ == "SiLUActivation":
                m.act_fn = torch.nn.SiLU()
        if not a.no_gc:
            model.gradient_checkpointing_enable()   # the reference's eager path has no working GC of its own
        cfg = ref_ta.Config()
        cfg.backend = "eager"
        cfg.compute.bf16 = True
        cfg.memory.gc = False
        cfg.dist.fsdp.size = world
        cfg.dist.fsdp.wrap_layer_cls = {"LlamaDecoderLayer"}
        model = ref_ta.accelerate(model, config=cfg)
        opt = torch.optim.AdamW(model.parameters(), lr=1e-5, betas=(0.9, 0.95), weight_decay=0.1, fused=True)
    except Exception as e:  # noqa: BLE001
        msg = f"setup failed: {type(e).__name__}: {e}"
        if world > 1 and "should be lazy" in str(e):
            # stock behaviour of the unmodified reference without torch_xla: accelerate() initialises the 'nccl'
            # process group for the eager backend (torchacc/dist/__init__.py:45-51) and Config.get_mesh() then
            # insists on the XLA 'lazy' backend (torchacc/config.py:396-398) -> no multi-rank eager run is possible
            msg = LAZY_MSG
        if world > 1 and dist.is_initialized():
            dist.destroy_process_group()
        unavailable(msg[:400])

    g = torch.Generator().manual_seed(rank)
    host = torch.randint(0, 128256, (a.mbs, a.seq_len), generator=g).pin_memory()
    ids = host.to(device)
    last = {}

    def step(x=ids):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = model(input_ids=x, labels=x)
        loss = out.loss if hasattr(out, "loss") else out["loss"]
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0) if world == 1 else model.clip_grad_norm_(1.0)
        opt.step()
        opt.zero_grad(set_to_none=True)
        last["loss"] = loss
        return loss

    try:
        for _ in range(a.warmup):
            step()
        torch.cuda.synchronize(device)
        sampler = ClockSampler(local_rank).start() if rank == 0 else None
        ms = timed_loop(step, a.steps, 0, device, world)
        clocks = sampler.stop() if sampler else None
    except Exception as e:  # noqa: BLE001
        unavailable(f"run failed: {type(e).__name__}: {e}"[:300])
    tokens = a.mbs * a.seq_len * world * a.steps
    value = tokens / (ms / 1e3)
    e2e = None
    if not a.no_e2e:
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        for _ in range(a.steps):
            loss_val = float(step(host.to(device, non_blocking=True)))
        torch.cuda.synchronize(device)
        wall = torch.tensor([(time.perf_counter() - t0) * 1e3], device=device)
        if world > 1:
            dist.all_reduce(wall, op=dist.ReduceOp.MAX)
        e2e = {"value": tokens / (float(wall) / 1e3), "unit": "tokens/s",
               "h2d_bytes_per_step": int(a.mbs * a.seq_len * 8), "d2h_bytes_per_step": 4, "last_loss": loss_val}
    if rank == 0:
        print(json.dumps({
            "metric": METRIC,
            "value": value, "unit": "tokens/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": value / (A100_TOKENS_PER_S_PER_GPU * world), "dtype": "bf16", "data": "synthetic",
            "impl": "reference",
            "config": bench_config(a, world, hf.num_hidden_layers),
            "detail": {"model_code": "HF LlamaForCausalLM", "gc": "HF gradient_checkpointing_enable()",
                       "optimizer": "torch.optim.AdamW(fused=True) + clip_grad_norm(1.0)",
                       "stack": "torchacc eager: torch FSDP1 + cuBLAS + flash-attn2 + liger"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": 0, "loss": float(last["loss"])}), flush=True)
    if world > 1:
        dist.barrier(device_ids=[device.index])
        dist.destroy_process_group()

# ----------------------------------------------------------------------------------------------------------------
# context arm (NOT the reference): what reference fsdp.py:196-216 would build if its eager path could run on N > 1
# ----------------------------------------------------------------------------------------------------------------
def run_torch_fsdp(a):
    """torch FSDP1 FULL_SHARD + MixedPrecision(bf16 params, fp32 reduce, fp32 buffers) + ModuleWrapPolicy over
    LlamaDecoderLayer, the reference's own kernel patches (its liger + flash-attn-2 patches, applied by importing the
    stock reference package and calling its ``apply_liger_kernel``), HF gradient checkpointing, fused torch AdamW.
    This is a hand-assembled stand-in, printed with ``"impl": "torch_fsdp"`` -- it never goes through
    ``--impl reference``, which stays the unmodified stock path (and is unavailable for N > 1, see DESIGN.md)."""
    rank, local_rank, world = dist_env()
    import torch
    import torch.distributed as dist
    from transformers import LlamaForCausalLM  # noqa: F401  (before the reference import, see run_reference)
    import transformers.models.llama.modeling_llama as ml
    import transformers.modeling_flash_attention_utils  # noqa: F401
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    patches = "none (baseline/_ref missing)"
    if os.path.isdir(os.path.join(ref_dir, "torchacc")):
        sys.path.insert(0, ref_dir)
        sys.path.insert(0, os.path.join(ROOT, "baseline", "shims"))
        try:
            import torchacc as ref_ta          # import-time patch_fa (torchacc/__init__.py:135)
            patches = "reference patch_fa"
        except Exception as e:  # noqa: BLE001
            ref_ta, patches = None, f"reference import failed: {type(e).__name__}"
    else:
        ref_ta = None
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29533")
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=device)
    model, hf = hf_llama(a, torch, device, 1)          # built on the GPU (32 GB fp32), FSDP shards it from there
    for m in model.modules():
        if type(getattr(m, "act_fn", None)).__name__ == "SiLUActivation":
            m.act_fn = torch.nn.SiLU()
    if ref_ta is not None:
        try:
            ref_ta.ops.apply_liger_kernel()    # what reference accelerate() does on the eager backend (accelerate.py:95-96)
            patches += " + reference apply_liger_kernel"
        except Exception as e:  # noqa: BLE001
            patches += f" (liger failed: {type(e).__name__}: {e})"[:120]
    if not a.no_gc:
        model.gradient_checkpointing_enable()
    from torch.distributed.fsdp import FullyShardedDataParallel as FSDP, MixedPrecision, ShardingStrategy
    from torch.distributed.fsdp.wrap import ModuleWrapPolicy
    model = FSDP(model, sharding_strategy=ShardingStrategy.FULL_SHARD,
                 auto_wrap_policy=ModuleWrapPolicy({ml.LlamaDecoderLayer}),
                 mixed_precision=MixedPrecision(param_dtype=torch.bfloat16, reduce_dtype=torch.float32,
                                                buffer_dtype=torch.float32),
                 device_id=torch.cuda.current_device(), sync_module_states=False)
    opt = torch.optim.AdamW(model.parameters(), lr=1e-5, betas=(0.9, 0.95), weight_decay=0.1, fused=True)
    g = torch.Generator().manual_seed(rank)
    host = torch.randint(0, 128256, (a.mbs, a.seq_len), generator=g).pin_memory()
    ids = host.to(device)
    last = {}

    def step(x=ids):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = model(input_ids=x, labels=x)
        loss = out.loss if hasattr(out, "loss") else out["loss"]
        loss.backward()
        model.clip_grad_norm_(1.0)
        opt.step()
        opt.zero_grad(set_to_none=True)
        last["loss"] = loss
        return loss

    for _ in range(a.warmup):
        step()
    torch.cuda.synchronize(device)
    sampler = ClockSampler(local_rank).start() if rank == 0 else None
    ms = timed_loop(step, a.steps, 0, device, world)
    clocks = sampler.stop() if sampler else None
    tokens = a.mbs * a.seq_len * world * a.steps
    value = tokens / (ms / 1e3)
    e2e = None
    if not a.no_e2e:
        dist.barrier(device_ids=[device.index])
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        for _ in range(a.steps):
            loss_val = float(step(host.to(device, non_blocking=True)))
        torch.cuda.synchronize(device)
        wall = torch.tensor([(time.perf_counter() - t0) * 1e3], device=device)
        dist.all_reduce(wall, op=dist.ReduceOp.MAX)
        e2e = {"value": tokens / (float(wall) / 1e3), "unit": "tokens/s",
               "h2d_bytes_per_step": int(a.mbs * a.seq_len * 8), "d2h_bytes_per_step": 4, "last_loss": loss_val}
    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": "tokens/s", "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": value / (A100_TOKENS_PER_S_PER_GPU * world), "dtype": "bf16", "data": "synthetic",
            "impl": "torch_fsdp", "config": bench_config(a, world, hf.num_hidden_layers),
            "detail": {"note": "NOT the reference arm: hand-assembled torch FSDP1 stack mirroring reference "
                               "dist/fsdp.py:196-216 so that N > 1 has a same-box competitor",
                       "model_code": "HF LlamaForCausalLM", "kernel_patches": patches,
                       "optimizer": "torch.optim.AdamW(fused=True) + FSDP.clip_grad_norm_(1.0)",
                       "stack": "torch FSDP1 FULL_SHARD + MixedPrecision(bf16/fp32 reduce) + cuBLAS + flash-attn2 + liger"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": 0, "loss": float(last["loss"])}), flush=True)
    dist.barrier(device_ids=[device.index])
    dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "torch_fsdp":
        run_torch_fsdp(args)
    else:
        run_ours(args)
