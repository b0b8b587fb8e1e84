"""End-to-end numerics of the native Llama on the sm_100a kernels vs the PyTorch fp32 reference path."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _tiny(device, dtype):
    from torchacc_b200.models import build_llama
    torch.manual_seed(0)
    with torch.device(device):
        return build_llama("tiny", hidden_size=512, intermediate_size=1408, num_hidden_layers=2, num_attention_heads=4,
                           num_key_value_heads=2, head_dim=128, vocab_size=2048, max_position_embeddings=512,
                           dtype=dtype)


def test_llama_native_matches_fp32_reference():
    dev = torch.device("cuda", 0)
    ref = _tiny("cpu", torch.float32)
    nat_model = _tiny(dev, torch.bfloat16)
    nat_model.load_state_dict({k: v.to(dev, torch.bfloat16) for k, v in ref.state_dict().items()})
    ids = torch.randint(0, 2048, (2, 256))
    out_r = ref(ids, labels=ids)
    out_n = nat_model(ids.to(dev), labels=ids.to(dev))
    assert abs(float(out_r["loss"]) - float(out_n["loss"])) < 3e-2, (float(out_r["loss"]), float(out_n["loss"]))
    out_r["loss"].backward()
    out_n["loss"].backward()
    for (n, pr), (_, pn) in zip(ref.named_parameters(), nat_model.named_parameters()):
        g_r, g_n = pr.grad.float(), pn.grad.float().cpu()
        denom = g_r.norm().item() + 1e-6
        rel = (g_r - g_n).norm().item() / denom
        assert rel < 8e-2, f"{n}: relative grad error {rel:.3f}"


def test_engine_trains_and_uses_native_kernels():
    import torchacc_b200 as ta
    from torchacc_b200 import _native as nat
    dev = torch.device("cuda", 0)
    model = _tiny(dev, torch.bfloat16)
    cfg = ta.Config()
    cfg.compute.bf16 = True
    cfg.memory.gc = True
    cfg.memory.gc_cls = {"LlamaDecoderLayer"}
    cfg.dist.fsdp.wrap_layer_cls = {"LlamaDecoderLayer"}
    model = ta.accelerate(model, config=cfg)
    opt = ta.optim.FusedAdamW(model.parameters(), lr=2e-3)
    ids = torch.randint(0, 2048, (4, 128), device=dev)
    n0 = nat.LAUNCHES
    losses = []
    for _ in range(8):
        out = model(input_ids=ids, labels=ids)
        out["loss"].backward()
        model.clip_grad_norm_(1.0)
        opt.step()
        model.zero_grad()
        losses.append(float(out["loss"]))
    assert nat.LAUNCHES > n0
    assert losses[-1] < losses[0] - 0.5, losses
    # every GEMM weight gradient was written straight into the flat buffer by the wgrad epilogue, also under
    # activation checkpointing (whose saved-tensor hooks hand back attribute-less aliases of the weights)
    assert model.engine.stats.get("wgrad_fallbacks", 0) == 0, model.engine.stats


@pytest.mark.parametrize("grad_dtype,tol", [("compute", 5e-2), ("fp32", 1e-2)])
def test_grad_accumulation_matches_single_batch(grad_dtype, tol):
    """Two micro-batches accumulated in the flat gradient buffer == one batch of both (fused mode, 1 GPU).  With
    dist.fsdp.grad_dtype='fp32' the wgrad epilogues accumulate into an fp32 buffer (the reference reduces gradients in
    fp32, dist/fsdp.py:204-208): 5x tighter tolerance than the bf16 buffer."""
    import torchacc_b200 as ta
    dev = torch.device("cuda", 0)
    ids = torch.randint(0, 2048, (4, 128), device=dev)

    def run(split):
        model = _tiny(dev, torch.bfloat16)
        cfg = ta.Config()
        cfg.compute.bf16 = True
        cfg.dist.fsdp.wrap_layer_cls = {"LlamaDecoderLayer"}
        cfg.dist.fsdp.grad_dtype = grad_dtype
        m = ta.accelerate(model, config=cfg)
        assert m.engine.grad_wire_dtype == (torch.float32 if grad_dtype == "fp32" else torch.bfloat16)
        opt = ta.optim.FusedAdamW(m.parameters(), lr=1e-3)
        if split:
            for part in ids.chunk(2):
                (m(input_ids=part, labels=part)["loss"] / 2).backward()
        else:
            m(input_ids=ids, labels=ids)["loss"].backward()
        return torch.cat([g.float().reshape(-1) for g in m.engine.grads()])

    g1, g2 = run(False), run(True)
    rel = (g1 - g2).norm() / g1.norm()
    assert rel < tol, float(rel)


def test_bench_dump_outputs_is_reproducible(tmp_path):
    """bench.py --dump-outputs: the last timed step's loss, gradient norm and weight sample come out as float32 .npy
    files within 64 MB, and a second run with the same arguments computes the same thing."""
    import json
    import os
    import subprocess
    import sys
    import numpy as np
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

    def run(d):
        cmd = [sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
               "--layers", "1", "--seq-len", "512", "--mbs", "1", "--no-e2e", "--dump-outputs", str(d)]
        p = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-3000:]
        res = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
        assert res["steps"] == 2 and res["warmup"] == 1
        return {f[:-4]: np.load(d / f) for f in sorted(os.listdir(d))}

    a, b = run(tmp_path / "a"), run(tmp_path / "b")
    assert sorted(a) == ["grad_norm", "loss", "weights_sample"]
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    np.testing.assert_allclose(a["loss"], b["loss"], rtol=1e-3)
    np.testing.assert_allclose(a["grad_norm"], b["grad_norm"], rtol=1e-2)
    # three AdamW steps at lr 1e-5 move a weight by at most a few 1e-5, whatever the order of the float sums
    np.testing.assert_allclose(a["weights_sample"], b["weights_sample"], rtol=0, atol=1e-4)


def test_hf_llama_through_accelerate_uses_native_attention_and_rope():
    """accelerate(HF LlamaForCausalLM): linears, RMSNorm, SwiGLU, RoPE, attention and the loss run on the native kernels
    (round-1 review: the HF path fell back to the flash-attn library and HF's elementwise RoPE) and the loss / its
    trajectory match the un-patched HF model."""
    import copy
    transformers = pytest.importorskip("transformers")
    import torchacc_b200 as ta
    from torchacc_b200 import _native as nat
    from torchacc_b200.utils.patch import unpatch_all
    from transformers import LlamaConfig, LlamaForCausalLM
    dev = torch.device("cuda", 0)
    cfg = LlamaConfig(vocab_size=2048, hidden_size=512, intermediate_size=1024, num_hidden_layers=2,
                      num_attention_heads=8, num_key_value_heads=2, max_position_embeddings=512, rms_norm_eps=1e-5,
                      tie_word_embeddings=False, attn_implementation="sdpa", use_cache=False)
    torch.manual_seed(0)
    ref = LlamaForCausalLM(cfg).to(dev, torch.bfloat16)
    ours = copy.deepcopy(ref)
    ids = torch.randint(0, 2048, (2, 256), device=dev)
    ref_loss = ref(input_ids=ids, labels=ids).loss
    from transformers.models.llama import modeling_llama as ml
    saved = [(c, c.forward) for c in (ml.LlamaRMSNorm, ml.LlamaMLP, ml.LlamaForCausalLM)]
    try:
        ours.config._attn_implementation = "flash_attention_2"       # HF dispatches to the patched interface
        c = ta.Config()
        c.compute.bf16 = True
        c.dist.fsdp.wrap_layer_cls = {"LlamaDecoderLayer"}
        model = ta.accelerate(ours, config=c)
        assert ml.apply_rotary_pos_emb.__name__ == "hf_apply_rotary_pos_emb"
        n0 = nat.LAUNCHES
        out = model(input_ids=ids, labels=ids)
        launches = nat.LAUNCHES - n0
        assert launches >= 2 * (4 + 2 + 2 + 1 + 1) + 2, launches       # linears + norms + rope + attention + swiglu per layer
        assert abs(float(out.loss) - float(ref_loss)) < 5e-2, (float(out.loss), float(ref_loss))
        opt = ta.optim.FusedAdamW(model.parameters(), lr=2e-3)
        losses = []
        for _ in range(6):
            l = model(input_ids=ids, labels=ids).loss
            l.backward()
            opt.step()
            opt.zero_grad()
            losses.append(float(l))
        assert losses[-1] < losses[0] - 0.5, losses
    finally:
        for cls, f in saved:
            cls.forward = f
            if hasattr(cls, "_tb_lce_patched"):
                del cls._tb_lce_patched
        unpatch_all()
