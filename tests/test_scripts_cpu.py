"""End-to-end runs of the user-facing scripts on CPU (gloo): BASELINE.json config #1 (benchmarks/transformer.py small
config, accelerate() dp_size=2), the examples and the accuracy benchmark."""
import json
import os
import subprocess
import sys

import pytest

from dist_utils import _free_port

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(cmd, timeout=600, env=None):
    e = dict(os.environ)
    e.update(env or {})
    e.setdefault("OMP_NUM_THREADS", "2")
    p = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=timeout, env=e)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-3000:]
    return p.stdout


def _torchrun(n, port, *args):
    return [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr",
            "127.0.0.1", "--master-port", str(port), *args]


def test_benchmark_transformer_dp2_gloo():
    out = _run(_torchrun(2, _free_port(), "benchmarks/transformer.py", "--model_name", "gpt2-tiny", "--max_seq_length", "64",
                         "--batch_size", "2", "--num_train_steps", "6", "--log_interval", "3", "--dp_size", "2"))
    recs = [json.loads(l) for l in out.splitlines() if l.startswith("{") and "samples_per_s" in l]
    assert len(recs) == 2 and recs[-1]["step"] == 6 and recs[-1]["samples_per_s"] > 0
    assert recs[-1]["loss"] < recs[0]["loss"] + 0.5


def test_example_parallelism_tour_pp_and_ring():
    for mode in ("pp", "ring"):
        out = _run(_torchrun(2, _free_port(), "examples/parallelism_tour.py", "--mode", mode))
        losses = [float(l.split("loss")[1]) for l in out.splitlines() if l.startswith(f"[{mode}]")]
        assert len(losses) == 10 and losses[-1] < losses[0], (mode, losses)


def test_example_train_llama_fsdp_single_process(tmp_path):
    out = _run([sys.executable, "examples/train_llama_fsdp.py", "--steps", "12", "--ckpt_dir", str(tmp_path / "ck")])
    assert "step   10" in out
    assert any(f.endswith(".pth") for f in os.listdir(tmp_path / "ck")), os.listdir(tmp_path / "ck")


def test_accuracy_benchmark_tiny(tmp_path):
    out = _run(["bash", "benchmarks/accuracy/run.sh"],
               env={"MODEL": "tiny", "LAYERS": "2", "STEPS": "12", "SEQ": "64", "BS": "2", "OUT": str(tmp_path)})
    res = json.loads(out.strip().splitlines()[-1])
    assert res["pass"] and res["abs_delta"] <= 1e-2


def test_accuracy_benchmark_tiny_hf_model(tmp_path):
    """Same protocol on the HuggingFace LlamaForCausalLM object (kernel patches + fused linear-CE through accelerate())."""
    pytest.importorskip("transformers")
    out = _run(["bash", "benchmarks/accuracy/run.sh"],
               env={"MODEL": "tiny", "LAYERS": "2", "STEPS": "12", "SEQ": "64", "BS": "2", "HF": "1",
                    "OUT": str(tmp_path)})
    res = json.loads(out.strip().splitlines()[-1])
    assert res["pass"] and res["abs_delta"] <= 1e-2


@pytest.mark.parametrize("flag", ["--tp", "--sp"])
def test_example_train_hf_model_under_tp_and_sp(flag):
    """examples/train_hf_model.py on 4 gloo ranks: an unmodified HF Llama under tp2 x fsdp2 / sp2 x fsdp2 trains (loss falls)."""
    pytest.importorskip("transformers")
    out = _run(_torchrun(4, _free_port(), "examples/train_hf_model.py", flag, "2", "--steps", "11"))
    losses = [float(l.split("loss")[1]) for l in out.splitlines() if l.startswith("step ")]
    assert len(losses) == 3 and losses[-1] < losses[0] - 1.0, losses
