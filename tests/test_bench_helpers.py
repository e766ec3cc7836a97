"""CPU checks of the harness pieces of ``bench.py`` that decide whether a run counts: token source, validity scan, config keys."""
import importlib.util
import json
import os

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_tokens_never_contain_the_padding_row_and_differ_per_rank():
    b = _bench()
    t0 = b.make_tokens(3, 2, 4, 64, 32100, rank=0, pinned=False)
    t1 = b.make_tokens(3, 2, 4, 64, 32100, rank=1, pinned=False)
    assert t0.shape == (3, 2, 4, 64) and t0.dtype == torch.long
    assert int(t0.max()) < 32099 + 1 and int(t0.max()) != 32099 and int(t0.min()) >= 0   # row V-1 is the zero padding row
    assert not torch.equal(t0, t1)
    assert torch.equal(t0, b.make_tokens(3, 2, 4, 64, 32100, rank=0, pinned=False))        # reproducible
    small = b.make_tokens(200, 1, 8, 64, 50, rank=3, pinned=False)                         # exhaustive at a tiny vocabulary
    assert int(small.max()) == 48 and int(small.min()) == 0


def test_first_nonfinite_reports_step_and_rank():
    b = _bench()
    log = torch.ones(4, 10)
    assert b.first_nonfinite(log) == (None, None)
    log[2, 7] = float("nan")
    log[1, 8] = float("inf")
    assert b.first_nonfinite(log) == (7, 2)
    log[3, 7] = float("inf")
    assert b.first_nonfinite(log) == (7, 2)   # lowest rank of the first bad step


def test_both_arms_share_config_keys_and_recipes_follow_the_baseline():
    b = _bench()
    keys = None
    for model, rec in b.RECIPES.items():
        cfg = b.case_config(model, rec["batch"], rec["ga"], 512, 128, 8, "adam", rec["reset"])
        keys = keys or set(cfg)
        assert set(cfg) == keys and cfg["parallelism"] == "dp8" and cfg["global_batch"] == rec["batch"] * rec["ga"] * 8
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert "tokens/s" in b.METRIC and "tokens/sec" in base["metric"]   # same quantity: whole-job tokens per second, device-timed
    assert "llama_250m" in base["metric"] and "llama_1b" in base["metric"] and set(b.RECIPES) == {"llama_250m", "llama_1b"}
    # llama_250m: the README recipe (batch 24, 1152 sequences per update on 8 GPUs); llama_1b: magnitude pruning 0.9 (config 4)
    assert b.RECIPES["llama_250m"]["batch"] * b.RECIPES["llama_250m"]["ga"] * 8 == 1152
    assert b.RECIPES["llama_1b"]["reset"]["optimizer_magnitude_pruning"] == 0.9
    assert b.EXIT_NONFINITE == 3


def test_dump_outputs_writes_float_arrays_at_fixed_positions(tmp_path):
    from relora_b200.models import LlamaForCausalLM, load_config

    b = _bench()
    torch.manual_seed(0)
    model = LlamaForCausalLM(load_config(os.path.join(ROOT, "configs", "llama_9m.json")))
    b.dump_outputs(str(tmp_path / "out"), "llama_9m", 10.5, torch.tensor(0.25), model)
    names = sorted(os.listdir(tmp_path / "out"))
    assert names == ["llama_9m_grad_norm.npy", "llama_9m_loss.npy", "llama_9m_params_sample.npy"]
    import numpy as np

    arrays = {n: np.load(tmp_path / "out" / n) for n in names}
    assert all(a.dtype == np.float32 for a in arrays.values())
    assert arrays["llama_9m_loss.npy"].tolist() == [10.5] and arrays["llama_9m_grad_norm.npy"].tolist() == [0.25]
    want = sum(min(p.numel(), b.DUMP_PER_PARAM) for p in model.parameters())
    sample = arrays["llama_9m_params_sample.npy"]
    assert sample.shape == (want,) and sum(a.nbytes for a in arrays.values()) <= b.DUMP_LIMIT_BYTES // 2
    assert np.array_equal(sample, b.parameter_sample(model).numpy())        # same model, same positions
    with torch.no_grad():
        model.lm_head.weight.add_(1.0)
    assert not np.array_equal(sample, b.parameter_sample(model).numpy())    # the sample sees the parameters
