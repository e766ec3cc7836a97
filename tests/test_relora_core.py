"""ReLoRA wrapping, merge/re-init, pruning and checkpoint-layout tests (SURVEY.md Appendix A)."""
import json
import os

import pytest
import torch

from relora_b200.models import LlamaForCausalLM, load_config
from relora_b200.relora import ReLoRaLinear, ReLoRaModel, magnitude_pruning_, optimizer_reset, random_pruning_
from relora_b200.relora.optim_reset import magnitude_threshold

CFG = os.path.join(os.path.dirname(os.path.dirname(__file__)), "configs", "llama_9m.json")
TARGETS = ["attn", "attention", "mlp"]


def _model():
    torch.manual_seed(0)
    return LlamaForCausalLM(load_config(CFG))


def test_magnitude_pruning_golden():
    t = (torch.arange(-10, 10) / 10).view(4, 5).clone()
    magnitude_pruning_(t, 0.5)
    want = torch.tensor([-1, -.9, -.8, -.7, -.6] + [0] * 11 + [.6, .7, .8, .9]).view(4, 5)
    assert torch.allclose(t, want)


def test_magnitude_threshold_matches_quantile():
    torch.manual_seed(1)
    x = torch.randn(1000)
    for q in (0.1, 0.5, 0.8, 0.9, 0.999):
        assert torch.allclose(magnitude_threshold(x, q), torch.quantile(x.abs(), q), atol=1e-6)


def test_pruning_keeps_dtype_and_ratio():
    x = torch.ones(100_000, dtype=torch.bfloat16)
    random_pruning_(x, 0.999)
    assert x.dtype == torch.bfloat16
    assert 20 <= int(x.sum()) <= 250
    y = torch.randn(4096, dtype=torch.bfloat16)
    magnitude_pruning_(y, 0.9)
    assert y.dtype == torch.bfloat16 and 0.85 < float((y == 0).float().mean()) < 0.95


def test_wrap_counts_and_quirks():
    m = _model()
    before = sum(p.numel() for p in m.parameters())
    assert before == 9_021_568
    w = ReLoRaModel(m, r=8, lora_alpha=32, target_modules=TARGETS)
    assert sum(p.numel() for p in w.parameters()) == 9_100_416
    mods = w.relora_modules()
    assert len(mods) == 28
    non_lora = [n for n, p in w.named_parameters() if p.requires_grad and "lora_" not in n]
    assert len(non_lora) == 11  # embed, 8 layer norms, final norm, lm_head
    for mod in mods:
        assert float(mod.lora_A.weight.abs().sum()) == 0 and float(mod.lora_B.weight.abs().sum()) == 0
        assert mod.scaling == 4.0 and not mod.weight.requires_grad
    ids = torch.randint(0, 32100, (2, 16))
    w(input_ids=ids, labels=ids).loss.backward()
    a = mods[0].lora_A.weight.grad
    b = mods[0].lora_B.weight.grad
    assert float(a.abs().sum()) == 0 and float(b.abs().sum()) == 0  # both-zero quirk: no LoRA gradient
    assert float(m.model.embed_tokens.weight.grad.abs().sum()) > 0
    w.merge_and_reinit()
    assert float(mods[0].lora_A.weight.abs().sum()) > 0 and float(mods[0].lora_B.weight.abs().sum()) == 0


def test_merge_invariance_fp32():
    m = _model()
    w = ReLoRaModel(m, r=8, lora_alpha=32, target_modules=TARGETS, init_lora_a="kaiming")
    w.eval()
    for mod in w.relora_modules():
        torch.nn.init.normal_(mod.lora_B.weight, std=0.02)
    ids = torch.randint(0, 32100, (2, 16))
    with torch.no_grad():
        before = w(input_ids=ids).logits
        w.merge_and_reinit()
        after = w(input_ids=ids).logits
    assert float((before - after).abs().max()) < 1e-4


def test_reinit_is_rank_invariant_and_kaiming_bounded():
    m1, m2 = _model(), _model()
    w1 = ReLoRaModel(m1, r=8, lora_alpha=32, target_modules=TARGETS)
    w2 = ReLoRaModel(m2, r=8, lora_alpha=32, target_modules=TARGETS)
    torch.manual_seed(123)  # different global RNG state on the "other rank"
    w1.merge_and_reinit()
    torch.manual_seed(999)
    torch.rand(17)
    w2.merge_and_reinit()
    for a, b in zip(w1.relora_modules(), w2.relora_modules()):
        assert torch.equal(a.lora_A.weight, b.lora_A.weight)
        bound = 1.0 / (a.in_features ** 0.5)
        assert float(a.lora_A.weight.abs().max()) <= bound + 1e-6
    # a second restart draws different values
    first = w1.relora_modules()[0].lora_A.weight.clone()
    w1.merge_and_reinit()
    assert not torch.equal(first, w1.relora_modules()[0].lora_A.weight)


def test_save_layout_and_roundtrip(tmp_path):
    m = _model()
    w = ReLoRaModel(m, r=8, lora_alpha=32, target_modules=TARGETS, init_lora_a="kaiming")
    d = str(tmp_path / "model_10")
    w.save_pretrained(d)
    assert sorted(os.listdir(d)) == ["config.json", "pytorch_model.bin", "relora_config.json"]
    rc = json.load(open(os.path.join(d, "relora_config.json")))
    assert set(rc) == {"r", "lora_alpha", "lora_dropout", "target_modules", "keep_original_weights", "lora_only",
                       "trainable_scaling", "quantize", "use_double_quant"}
    assert rc["lora_only"] is False and rc["trainable_scaling"] is False
    sd = torch.load(os.path.join(d, "pytorch_model.bin"), weights_only=True)
    for k in ("weight", "lora_A.weight", "lora_B.weight"):
        assert f"model.layers.0.self_attn.q_proj.{k}" in sd
    assert not any(k.startswith("wrapped_model.") for k in sd)
    w2 = ReLoRaModel.from_pretrained(d)
    for (n1, p1), (n2, p2) in zip(w.named_parameters(), w2.named_parameters()):
        assert n1 == n2 and torch.equal(p1, p2)
    # legacy key shim
    rc["keep_original"] = True
    del rc["lora_only"], rc["trainable_scaling"]
    json.dump(rc, open(os.path.join(d, "relora_config.json"), "w"))
    w3 = ReLoRaModel.from_pretrained(d)
    assert w3.lora_only is False


def test_lora_only_and_trainable_scaling():
    lin = ReLoRaLinear(16, 8, r=4, lora_alpha=8, lora_only=True, bias=False)
    assert lin.weight is None
    x = torch.randn(3, 16)
    lin.eval()
    assert lin(x).shape == (3, 8)
    lin2 = ReLoRaLinear(16, 8, r=4, lora_alpha=8, trainable_scaling=True, bias=True)
    assert isinstance(lin2.scaling, torch.nn.Parameter)
    assert torch.allclose(lin2._post_lora_scale(), torch.tanh(torch.tensor([1.0])))
    lin2.merge_and_reinit()
    assert float(lin2.scaling) == 0.0
    with pytest.raises(ValueError):
        ReLoRaLinear(4, 4, r=0)


@pytest.mark.parametrize("fmt,tol", [("mxfp8", 0.07), ("nvfp4", 0.3), ("8bit", 0.07), ("4bit", 0.3)])
def test_quantized_frozen_weight_and_merge(fmt, tol):
    torch.manual_seed(0)
    w = torch.randn(64, 96) * 0.02
    lin = ReLoRaLinear(96, 64, r=8, lora_alpha=16, bias=False, weight_data=w.clone(), quantize=fmt)
    rel = float((lin.weight - w).norm() / w.norm())
    assert rel < tol
    torch.nn.init.normal_(lin.lora_B.weight, std=0.05)
    target = lin.weight.float() + 2.0 * lin.lora_B.weight.float() @ lin.lora_A.weight.float()
    lin.merge_and_reinit()
    assert float((lin.weight.float() - target).norm() / target.norm()) < tol
    assert float(lin.lora_B.weight.abs().sum()) == 0
    # storage really is packed
    assert lin.qweight.data.dtype == torch.uint8


def test_optimizer_reset_modes():
    torch.manual_seed(0)
    p = [torch.nn.Parameter(torch.randn(64, 32)) for _ in range(3)]
    opt = torch.optim.AdamW(p, lr=1e-3)
    for q in p:
        q.grad = torch.randn_like(q)
    opt.step()
    with pytest.raises(ValueError):
        optimizer_reset(opt, reset_params=p[:2], optimizer_state_keys=["exp_avg", "exp_avg_sq"],
                        reset_optimizer_on_relora=True, optimizer_random_pruning=0.5, optimizer_magnitude_pruning=0.0)
    untouched = opt.state[p[2]]["exp_avg"].clone()
    pct = optimizer_reset(opt, reset_params=p[:2], optimizer_state_keys=["exp_avg", "exp_avg_sq"],
                          reset_optimizer_on_relora=False, optimizer_random_pruning=0.0, optimizer_magnitude_pruning=0.9)
    assert 88 < pct < 92
    assert torch.equal(untouched, opt.state[p[2]]["exp_avg"])
    pct = optimizer_reset(opt, reset_params=p[:2], optimizer_state_keys=["exp_avg", "exp_avg_sq"],
                          reset_optimizer_on_relora=True, optimizer_random_pruning=0.0, optimizer_magnitude_pruning=0.0)
    assert pct > 99


def test_reference_relora_state_dict_interchange():
    """A reference-wrapped model's weights load into ours (and produce the same logits as the reference, stored in tests/golden)."""
    import reference_golden as rg

    golden = rg.load()
    ours = ReLoRaModel(_model(), r=8, lora_alpha=32, target_modules=TARGETS)
    assert set(ours.wrapped_model.state_dict()) == set(golden["interchange:state_dict_keys"])
    rg.seed_parameters_(ours.wrapped_model)
    ours.eval()
    ids = rg.seeded_ids(**rg.INTERCHANGE_IDS)
    with torch.no_grad():
        b = ours(input_ids=ids, labels=ids)
    assert torch.allclose(rg.sampled(golden, "interchange:logits", b.logits), torch.from_numpy(golden["interchange:logits"]), atol=2e-5)
    assert abs(float(golden["interchange:loss"]) - float(b.loss)) < 1e-5
    # merge parity
    ours.merge_and_reinit()
    merged = [n for n, _ in ours.wrapped_model.named_parameters() if n.endswith("q_proj.weight") or n.endswith("down_proj.weight")]
    assert len(merged) == 8
    for n in merged:
        p2 = ours.wrapped_model.get_parameter(n)
        assert torch.allclose(rg.sampled(golden, f"interchange:merged:{n}", p2), torch.from_numpy(golden[f"interchange:merged:{n}"]), atol=1e-6), n


def test_utils_state_size_lr_alarm_and_packed_bytes():
    from relora_b200.utils import check_lr_and_alert, frozen_weight_bytes, optimizer_state_size

    torch.manual_seed(0)
    p = [torch.nn.Parameter(torch.randn(16, 8)) for _ in range(2)]
    opt = torch.optim.AdamW(p, lr=1e-3)
    for q in p:
        q.grad = torch.randn_like(q)
    opt.step()
    s = optimizer_state_size(opt)
    assert s["exp_avg_numel"] == 256 and s["exp_avg_nonzero"] == 256

    class Sink:
        def __init__(self):
            self.alerts = []

        def alert(self, title, text):
            self.alerts.append((title, text))

    sink = Sink()
    assert not check_lr_and_alert(opt, max_lr=1e-2, sink=sink)
    assert check_lr_and_alert(opt, max_lr=1e-4, sink=sink) and len(sink.alerts) == 1
    # block-scaled storage really shrinks the resident frozen weight: mxfp8 = 1 + 1/32 bytes, nvfp4 = 1/2 + 1/16 bytes per element
    for fmt, ratio in (("mxfp8", (1 + 1 / 32) / 2), ("nvfp4", (0.5 + 1 / 16) / 2)):
        lin = ReLoRaLinear(256, 128, r=8, bias=False, weight_data=torch.randn(128, 256) * 0.02, quantize=fmt)
        b = frozen_weight_bytes(torch.nn.Sequential(lin))
        assert abs(b["resident_bytes"] / b["bf16_bytes"] - ratio) < 0.01, (fmt, b)
        assert "weight" not in dict(lin.named_parameters())          # no dense copy is resident ...
        sd = lin.state_dict()
        assert sd["weight"].shape == (128, 256)                      # ... but checkpoints keep the reference key
        lin2 = ReLoRaLinear(256, 128, r=8, bias=False, quantize=fmt)
        lin2.load_state_dict(sd)
        assert float((lin2.weight - lin.weight).norm() / lin.weight.norm()) < (0.02 if fmt == "mxfp8" else 0.12)  # requantisation is near-idempotent
        x = torch.randn(4, 256, requires_grad=True)
        y = lin(x)
        y.sum().backward()
        assert x.grad is not None and torch.isfinite(x.grad).all()
