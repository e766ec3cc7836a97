"""What the original ReLoRA implementation (github.com/Guitaricet/relora, ``peft_pretraining``) computes, stored for the tests
that compare with it, so that they run without that code.

Both sides start from the same weights: ``seed_parameters_`` overwrites every parameter of a model from a seeded generator, in
name order, so the reference model and ours (same parameter names and shapes) hold identical values.  Inputs come from seeded
generators too.  ``tests/golden/reference.npz`` keeps the reference's outputs on them (large tensors as a fixed, seeded sample of
entries).  To regenerate it on a CPU (fp32), from a checkout of the original repository:

    python tests/reference_golden.py --reference <path to the original repository>
"""
from __future__ import annotations

import argparse
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden", "reference.npz")
TARGETS = ["attn", "attention", "mlp"]

# seeds and shapes of the inputs each comparison feeds both implementations
WEIGHT_SEED = 0
LLAMA_IDS = dict(seed=1, high=32000, shape=(2, 33))
INTERCHANGE_IDS = dict(seed=3, high=32000, shape=(2, 24))
PADDING_IDS = dict(seed=2, shape=(2, 48))
PADDING_LAYERS = 12
LOSS_CURVE = dict(steps=7, relora_every=3, ga=2, B=2, T=32, data_seed=1)


def seed_parameters_(module: torch.nn.Module, seed: int = WEIGHT_SEED) -> None:
    """Matrices ~ N(0, 0.02), vectors (norm gains) 1 + N(0, 0.02); the embedding's padding row stays zero, as at init."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for _, p in sorted(module.named_parameters(), key=lambda kv: kv[0]):
            v = torch.randn(p.shape, generator=g, dtype=torch.float32) * 0.02
            p.copy_(v + 1.0 if p.dim() == 1 else v)
        for m in module.modules():
            if isinstance(m, torch.nn.Embedding) and m.padding_idx is not None:
                m.weight[m.padding_idx].zero_()


def seeded_ids(seed: int, high: int, shape) -> torch.Tensor:
    return torch.randint(0, high, shape, generator=torch.Generator().manual_seed(seed))


def padding_row_ids(vocab: int, first: int) -> torch.Tensor:
    """Token ids over the real vocabulary [0, vocab - 1) whose first sequence starts with ``first``."""
    ids = seeded_ids(PADDING_IDS["seed"], vocab - 1, PADDING_IDS["shape"])
    ids[0, 0] = first
    return ids


def embedding_grad_norms(model, vocab: int) -> dict:
    """Gradient norm at the first position for an ordinary first token (5) and for the padding row (vocab - 1)."""
    norms = {}
    for first in (5, vocab - 1):
        ids = padding_row_ids(vocab, first)
        emb = model.model.embed_tokens(ids).detach().requires_grad_()
        model(inputs_embeds=emb, labels=ids).loss.backward()
        norms[first] = float(emb.grad[0, 0].norm())
    return norms


def loss_curve_batches(vocab: int):
    c = LOSS_CURVE
    g = torch.Generator().manual_seed(c["data_seed"])
    return [torch.randint(0, vocab, (c["ga"], c["B"], c["T"]), generator=g) for _ in range(c["steps"])]


def load() -> dict:
    with np.load(GOLDEN) as z:
        return {k: z[k] for k in z.files}


def sampled(golden: dict, key: str, t: torch.Tensor) -> torch.Tensor:
    """The entries of ``t`` (flattened) at the positions stored with ``key``."""
    return t.detach().reshape(-1)[torch.from_numpy(golden[key + ":idx"]).long()]


# ------------------------------------------------------------------------------------------------- generation
def _sample(out: dict, key: str, t: torch.Tensor, n: int, seed: int, prefer_nonzero: bool = False) -> None:
    flat = t.detach().reshape(-1).float()
    pool = flat.nonzero().flatten() if prefer_nonzero and bool((flat != 0).any()) else torch.arange(flat.numel())
    pick = pool[torch.randperm(pool.numel(), generator=torch.Generator().manual_seed(seed))[:n]].sort().values
    out[key + ":idx"] = pick.numpy().astype(np.int32)
    out[key] = flat[pick].numpy()


def _import_reference(path: str):
    # the reference imports bitsandbytes at module level; its non-quantised code never uses it
    for name in ("bitsandbytes", "bitsandbytes.nn", "bitsandbytes.functional"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["bitsandbytes"].nn = sys.modules["bitsandbytes.nn"]
    sys.modules["bitsandbytes"].functional = sys.modules["bitsandbytes.functional"]
    sys.path.append(path)
    import importlib

    return types.SimpleNamespace(llama=importlib.import_module("peft_pretraining.modeling_llama"),
                                 relora=importlib.import_module("peft_pretraining.relora"),
                                 training_utils=importlib.import_module("peft_pretraining.training_utils"))


def generate(reference: str) -> dict:
    from transformers import AutoConfig

    ref = _import_reference(reference)
    cfg_path = lambda name: os.path.join(reference, "configs", f"{name}.json")  # noqa: E731
    out = {}

    # Llama forward / backward (llama_9m)
    model = ref.llama.LlamaForCausalLM(AutoConfig.from_pretrained(cfg_path("llama_9m")))
    seed_parameters_(model)
    out["llama:state_dict_keys"] = np.array(sorted(model.state_dict()))
    ids = seeded_ids(**LLAMA_IDS)
    res = model(input_ids=ids, labels=ids)
    out["llama:loss"] = np.float64(res.loss.item())
    _sample(out, "llama:logits", res.logits, 8192, seed=10)
    res.loss.backward()
    for i, (name, p) in enumerate(model.named_parameters()):
        _sample(out, f"llama:grad:{name}", p.grad, 256, seed=100 + i, prefer_nonzero=True)
        out[f"llama:grad_norm:{name}"] = np.float64(p.grad.norm().item())

    # a sequence starting with the zero padding row overflows the gradient (llama_35m, 12 layers)
    cfg = AutoConfig.from_pretrained(cfg_path("llama_35m"))
    cfg.num_hidden_layers = PADDING_LAYERS
    model = ref.llama.LlamaForCausalLM(cfg)
    seed_parameters_(model)
    norms = embedding_grad_norms(model, cfg.vocab_size)
    out["padding:vocab"] = np.int64(cfg.vocab_size)
    out["padding:norm_ordinary"] = np.float64(norms[5])
    out["padding:norm_padding_row"] = np.float64(norms[cfg.vocab_size - 1])

    # ReLoRA-wrapped state dict: logits, loss and merged weights (llama_9m, r = 8)
    ref_w = ref.relora.ReLoRaModel(ref.llama.LlamaForCausalLM(AutoConfig.from_pretrained(cfg_path("llama_9m"))), r=8,
                                   lora_alpha=32, target_modules=TARGETS, lora_dropout=0.1, keep_original_weights=True)
    seed_parameters_(ref_w.wrapped_model)
    out["interchange:state_dict_keys"] = np.array(sorted(ref_w.wrapped_model.state_dict()))
    ref_w.eval()
    ids = seeded_ids(**INTERCHANGE_IDS)
    with torch.no_grad():
        res = ref_w(input_ids=ids, labels=ids)
    out["interchange:loss"] = np.float64(res.loss.item())
    _sample(out, "interchange:logits", res.logits, 8192, seed=20)
    ref_w.merge_and_reinit()
    for i, (name, p) in enumerate(ref_w.wrapped_model.named_parameters()):
        if name.endswith("q_proj.weight") or name.endswith("down_proj.weight"):
            _sample(out, f"interchange:merged:{name}", p, 1024, seed=200 + i)

    # training losses through a ReLoRA reset (the loop of the reference's torchrun_main.py, llama_9m, fp32)
    c = LOSS_CURVE
    cfg = AutoConfig.from_pretrained(cfg_path("llama_9m"))
    ref_w = ref.relora.ReLoRaModel(ref.llama.LlamaForCausalLM(cfg), r=8, lora_alpha=32, target_modules=TARGETS, lora_dropout=0.0,
                                   keep_original_weights=True)
    seed_parameters_(ref_w.wrapped_model)
    trainable = [p for p in ref_w.parameters() if p.requires_grad]
    lora_params = [p for n, p in ref_w.named_parameters() if p.requires_grad and "lora_" in n]
    opt = torch.optim.AdamW(trainable, lr=1e-3, betas=(0.9, 0.999), weight_decay=0.0)
    sch = ref.training_utils.get_scheculer(opt, scheduler_type="cosine_restarts", num_training_steps=9, warmup_steps=1,
                                           min_lr_ratio=0.1, cycle_length=c["relora_every"], restart_warmup_steps=1)
    torch.manual_seed(0)  # the reference re-initialises LoRA A from the global generator
    losses = []
    ref_w.train()
    for step, batch in enumerate(loss_curve_batches(cfg.vocab_size), start=1):
        tot = 0.0
        for i in range(c["ga"]):
            loss = ref_w(input_ids=batch[i], labels=batch[i].clone()).loss
            (loss / c["ga"]).backward()
            tot += float(loss.detach())
        torch.nn.utils.clip_grad_norm_(trainable, 1.0, error_if_nonfinite=True)
        opt.step()
        sch.step()
        opt.zero_grad()
        losses.append(tot / c["ga"])
        # the reference resets at update_step % relora == 1: merge, then prune the LoRA moments
        if step % c["relora_every"] == 1 and step > 1:
            ref_w.merge_and_reinit()
            ref.training_utils.optimizer_reset(opt, reset_params=lora_params, optimizer_state_keys=["exp_avg", "exp_avg_sq"],
                                               reset_optimizer_on_relora=False, optimizer_random_pruning=0.0,
                                               optimizer_magnitude_pruning=0.9)
    out["loss_curve:losses"] = np.array(losses, dtype=np.float64)

    # LR multipliers of both schedules at every step
    tu = ref.training_utils
    for adjust in (0, 5):
        out[f"scheduler:cosine_restarts:adjust{adjust}"] = np.array([tu._get_cosine_schedule_with_multiple_warmups_lambda(
            s, num_training_steps=200, first_warmup_steps=20, restart_warmup_steps=7, restart_every=50, min_lr_ratio=0.05,
            adjust_step=adjust) for s in range(200)], dtype=np.float64)
    out["scheduler:cosine"] = np.array([tu._get_cyclical_cosine_schedule_with_min_lr_lambda(
        s, num_warmup_steps=10, cycle_length=40, min_lr_ratio=0.1) for s in range(200)], dtype=np.float64)
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser(description="regenerate tests/golden/reference.npz from the original implementation")
    ap.add_argument("--reference", required=True, help="checkout of the original ReLoRA repository")
    args = ap.parse_args()
    golden = generate(os.path.abspath(args.reference))
    os.makedirs(os.path.dirname(GOLDEN), exist_ok=True)
    np.savez_compressed(GOLDEN, **golden)
    print(f"wrote {GOLDEN} ({os.path.getsize(GOLDEN)} bytes, {len(golden)} arrays)")
