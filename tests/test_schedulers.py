"""Golden values captured from the reference schedulers (SURVEY.md Appendix A)."""
import math

import pytest
import torch

from relora_b200.relora.schedulers import build_multiplier, get_scheduler, get_scheculer


def _close(a, b, tol=2e-5):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert abs(x - y) < tol, (a, b)


def test_jagged_cosine_golden():
    m = build_multiplier("cosine_restarts", num_training_steps=100, warmup_steps=10, min_lr_ratio=0.1,
                         cycle_length=25, restart_warmup_steps=5)
    steps = [0, 1, 5, 9, 10, 11, 24, 25, 26, 27, 29, 30, 31, 49, 50, 51, 55, 75, 76, 80, 99]
    want = [0.0, 0.1, 0.5, 0.9, 1.0, 0.99973, 0.94733, 0.0, 0.17894, 0.35789, 0.71578, 0.89472, 0.88442, 0.64356,
            0.0, 0.11, 0.55, 0.0, 0.04106, 0.20528, 0.10027]
    _close([m(s) for s in steps], want)


def test_jagged_cosine_adjust_step_golden():
    m = build_multiplier("cosine_restarts", num_training_steps=100, warmup_steps=10, min_lr_ratio=0.1,
                         cycle_length=25, restart_warmup_steps=5, adjust_step=5)
    steps = [0, 9, 10, 19, 20, 21, 24, 25, 26, 44, 45, 46, 50]
    want = [0.0, 0.9, 0.99316, 0.94733, 0.93971, 0.93162, 0.9046, 0.89472, 0.88442, 0.64356, 0.0, 0.11, 0.55]
    _close([m(s) for s in steps], want)


def test_cyclical_cosine_golden():
    m = build_multiplier("cosine", num_training_steps=100, warmup_steps=10, min_lr_ratio=0.1, cycle_length=50)
    steps = [0, 1, 5, 10, 30, 49, 50, 51, 52, 55, 60, 99]
    want = [0.0, 0.1, 0.5, 1.0, 0.55, 0.1013872, 1e-07, 1e-07, 0.2, 0.5, 1.0, 0.1013872]
    _close([m(s) for s in steps], want, tol=1e-6)


def test_linear_schedule():
    m = build_multiplier("linear", num_training_steps=100, warmup_steps=10)
    assert m(0) == 0 and m(5) == 0.5 and m(10) == 1.0 and abs(m(55) - 0.5) < 1e-9 and m(100) == 0.0


def test_lr_used_by_each_update():
    p = torch.nn.Parameter(torch.zeros(1))
    opt = torch.optim.AdamW([p], lr=1e-3)
    sch = get_scheculer(opt, scheduler_type="cosine_restarts", num_training_steps=100, warmup_steps=10,
                        min_lr_ratio=0.1, cycle_length=25, restart_warmup_steps=5)
    used = []
    for _ in range(30):
        used.append(opt.param_groups[0]["lr"] * 1e3)
        opt.step()
        sch.step()
    want_head = [0, .1, .2, .3, .4, .5, .6, .7, .8, .9, 1.0, .9997, .9989, .9975, .9956, .9932, .9902, .9866, .9826,
                 .978, .9729, .9672, .9611, .9545, .9473, 0.0, .1789, .3579, .5368, .7158]
    _close(used, want_head, tol=1e-4)


def test_validation_errors():
    with pytest.raises(ValueError):
        build_multiplier("cosine_restarts", num_training_steps=101, warmup_steps=10, cycle_length=25, restart_warmup_steps=5)
    with pytest.raises(ValueError):
        build_multiplier("cosine", num_training_steps=101, warmup_steps=10, cycle_length=50)
    with pytest.raises(ValueError):
        build_multiplier("cosine_restarts", num_training_steps=100, warmup_steps=10, cycle_length=None, restart_warmup_steps=5)
    with pytest.raises(ValueError):  # adjust + warmup > restart_every
        build_multiplier("cosine_restarts", num_training_steps=100, warmup_steps=24, cycle_length=25, restart_warmup_steps=5, adjust_step=5)
    with pytest.raises(ValueError):
        build_multiplier("cosine", num_training_steps=100, warmup_steps=10, adjust_step=3)
    with pytest.raises(NotImplementedError):
        build_multiplier("nope", num_training_steps=100, warmup_steps=10)


def test_matches_reference_everywhere():
    """Every step of both schedules against the reference's lambdas (their values are stored in tests/golden)."""
    import reference_golden as rg

    golden = rg.load()
    for adjust in (0, 5):
        mine = build_multiplier("cosine_restarts", num_training_steps=200, warmup_steps=20, min_lr_ratio=0.05,
                                cycle_length=50, restart_warmup_steps=7, adjust_step=adjust)
        want = golden[f"scheduler:cosine_restarts:adjust{adjust}"]
        assert len(want) == 200
        for s in range(200):
            assert math.isclose(mine(s), float(want[s]), rel_tol=1e-12, abs_tol=1e-12), (s, adjust)
    mine = build_multiplier("cosine", num_training_steps=200, warmup_steps=10, min_lr_ratio=0.1, cycle_length=40)
    want = golden["scheduler:cosine"]
    assert len(want) == 200
    for s in range(200):
        assert math.isclose(mine(s), float(want[s]), rel_tol=1e-12, abs_tol=1e-12)
