"""Loss-curve parity with the unmodified reference on synthetic tokens (CPU, fp32, llama_9m): same initial weights, same
batches, the reference's own model / ReLoRaModel / scheduler / optimizer-reset code driven by the loop of
``torchrun_main.py:768-826`` versus this repo's TrainingEngine (SURVEY.md §4: "reference-vs-new loss-curve parity").
The reference's losses are stored in tests/golden (``tests/reference_golden.py`` regenerates them)."""
import os

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_training_losses_match_the_reference_through_a_relora_reset():
    import reference_golden as rg

    from relora_b200.engine.api import TrainingEngine
    from relora_b200.models import load_config

    c = rg.LOSS_CURVE
    steps, relora_every, ga, B, T = c["steps"], c["relora_every"], c["ga"], c["B"], c["T"]
    ref_losses = [float(x) for x in rg.load()["loss_curve:losses"]]
    assert len(ref_losses) == steps
    cfg_path = os.path.join(ROOT, "configs", "llama_9m.json")
    eng = TrainingEngine.build(
        model_config=cfg_path, batch_size=B, gradient_accumulation=ga, total_batch_size=B * ga,
        max_length=T, use_peft=True, lora_r=8, lora_alpha=32, lora_dropout=0.0, relora=relora_every, cycle_length=relora_every,
        scheduler="cosine_restarts", warmup_steps=1, restart_warmup_steps=1, lr=1e-3, num_training_steps=9, dtype="float32", device="cpu",
        reset_optimizer_on_relora=False, optimizer_magnitude_pruning=0.9, clip_grad_norm=1.0, min_lr_ratio=0.1)
    # the reference's weights, with the LoRA branch live from the start (upstream starts with A = B = 0)
    rg.seed_parameters_(eng.model.wrapped_model)
    our_losses = [float(eng.train_step(batch)) for batch in rg.loss_curve_batches(load_config(cfg_path).vocab_size)]
    # identical until (and including) the first update after the merge: the merged weights agree and B = 0 on both sides;
    # afterwards the re-initialised A differs by construction (upstream draws it from the torch generator, we hash)
    n_exact = relora_every + 2
    for a, b in zip(ref_losses[:n_exact], our_losses[:n_exact]):
        assert abs(a - b) < 2e-4, (ref_losses, our_losses)
    assert eng.n_lora_restarts >= 1
    # later steps: same trajectory up to the different (but equally distributed) re-initialisation
    for a, b in zip(ref_losses[n_exact:], our_losses[n_exact:]):
        assert abs(a - b) < 0.05, (ref_losses, our_losses)
