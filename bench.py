"""Headline benchmark: ReLoRA training throughput (tokens/s, whole job) on synthetic tokens.

    python bench.py --gpus 1 --steps 8 --warmup 3                    # this engine
    python bench.py --impl reference --gpus 1 --steps 8 --warmup 3   # unmodified reference (baseline/_ref)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus 8 --steps 8 --warmup 3

Headline config (BASELINE.json / reference README.md:52-88): llama_250m, ReLoRA r=128, bf16, seq 512, per-GPU
micro-batch 24, gradient accumulation 6 (=> the README's total batch 1152 at 8 GPUs; weak scaling:
global batch 144·N sequences).  One *step* = one optimizer update = 6 micro-batches per GPU, incl.
gradient reduction, clipping, AdamW and the LR schedule.  Random-init weights, synthetic token ids.

The same line carries a ``"llama_1b"`` block (BASELINE.json config 4: llama_1b ReLoRA r=128, seq 512, micro-batch 16 x
accumulation 4, ``optimizer_magnitude_pruning 0.9``), measured the same way with fewer steps so that both models fit
in one driver invocation; ``--no-1b`` drops it, ``--model X`` benchmarks X alone.

Timing: W >= 3 untimed steps, then exactly K steps bracketed by barrier + cuda synchronize, CUDA events on
the launching stream, max over ranks.  The working set of a step (0.5 GB of weights + >1 GB of activations)
exceeds the 126 MB L2, so no explicit flush is needed.  `value` is measured with device-resident inputs;
`e2e.value` goes through the public API (`TrainingEngine.train_step`): pinned-host token ids are copied to
the device every step and the loss is read back to the host every step.

Validity: every step's loss (per rank, before the cross-rank mean) and gradient norm is kept on the device and checked
after the timed regions, together with the parameters.  A run that saw a non-finite value prints the line with
``"valid": false`` and ``"nonfinite_at_step"`` / ``"nonfinite_rank"`` and exits with status 3 — a throughput of a run that
trained garbage is not a result.  The reference arm does the same when its ``clip_grad_norm_(error_if_nonfinite=True)``
raises (torchrun_main.py:805-808).
"""
from __future__ import annotations

import argparse
import gc
import json
import math
import os
import subprocess
import sys
import threading
import time
import types

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
os.environ.setdefault("RELORA_B200_NO_WANDB", "1")
os.environ.setdefault("WANDB_MODE", "disabled")
os.environ.setdefault("TOKENIZERS_PARALLELISM", "false")

METRIC = "training throughput, llama ReLoRA (tokens/s, whole job, device-timed, max over ranks)"
# per-model recipe: per-GPU micro-batch, accumulation, optimizer-reset flavour (BASELINE.json configs 3 and 4)
RECIPES = {
    "llama_250m": dict(batch=24, ga=6, reset=dict(reset_optimizer_on_relora=True)),
    "llama_1b": dict(batch=16, ga=4, reset=dict(reset_optimizer_on_relora=False, optimizer_magnitude_pruning=0.9)),
}
EXIT_NONFINITE = 3


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", type=str, default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", type=str, default=None, help="benchmark this model only (default: llama_250m headline + llama_1b block)")
    ap.add_argument("--batch", type=int, default=None, help="per-GPU micro-batch (README.md:55; default from the model's recipe)")
    ap.add_argument("--ga", type=int, default=None, help="gradient accumulation (1152 / (24*8), README.md:56)")
    ap.add_argument("--seq", type=int, default=512)
    ap.add_argument("--lora_r", type=int, default=128)
    ap.add_argument("--engine", type=str, default="auto")
    ap.add_argument("--comm", type=str, default="auto")
    ap.add_argument("--optimizer", type=str, default="adam")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-1b", action="store_true", help="skip the llama_1b block")
    ap.add_argument("--steps-1b", type=int, default=6, help="timed steps of the llama_1b block (capped by --steps)")
    ap.add_argument("--frozen_dtype", type=str, default=None, help="fp8: E4M3 tensor-core path for the frozen weights (opt-in)")
    ap.add_argument("--attention", type=str, default="auto", choices=["auto", "native", "sdpa"])
    ap.add_argument("--cuda_graphs", type=str, default="true")
    ap.add_argument("--dump-outputs", type=str, default=None, metavar="DIR",
                    help="after the timed steps, write what the last step computed (loss, gradient norm, a fixed sample of the "
                         "parameters) as DIR/<model>_<name>.npy, so that two builds can be compared output for output")
    return ap.parse_args()


# --------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples `nvidia-smi` clocks / throttle reasons during the timed region (rank 0, GPU 0)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int = 0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------- shared
def setup_dist(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device")
    torch.cuda.set_device(local)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29517")
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
    if world != args.gpus and rank == 0:
        print(f"[bench] warning: --gpus {args.gpus} but WORLD_SIZE={world}; using {world}", file=sys.stderr)
    return rank, local, world


def timed(fn_step, steps, world, device):
    """barrier + sync | K steps between CUDA events | sync + barrier; returns max-over-ranks seconds."""
    import torch
    import torch.distributed as dist

    dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn_step(i)
    e1.record()
    torch.cuda.synchronize()
    dist.barrier()
    t = torch.tensor([e0.elapsed_time(e1) / 1e3], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def make_tokens(steps, ga, batch, seq, vocab, rank, pinned):
    """Synthetic ids uniform over the *real* vocabulary [0, vocab - 1): the configs' ``pad_token_id = -1`` makes row vocab - 1 the
    embedding's padding row (all zeros, never trained; ``modeling_llama.py:433-436``) and real text never contains that id.
    A sequence that *starts* with it keeps an exactly-zero residual row through every layer (v = 0, no biases, LoRA B = 0), where
    RMSNorm's backward has gain 1/sqrt(eps) = 1000 per norm; the gradient overflows after ~17 layers.  That is what turned both arms
    non-finite at 4 and 8 GPUs in round 1 (P = 1/32100 per sequence: ~55 % of 45-step runs at N = 4); see DESIGN.md "root cause"."""
    import torch

    g = torch.Generator().manual_seed(1234 + rank)
    t = torch.randint(0, vocab - 1, (steps, ga, batch, seq), generator=g, dtype=torch.long)
    return t.pin_memory() if pinned else t


def case_config(model, batch, ga, seq, lora_r, world, optimizer, reset):
    """The `config` object of the result line: the SAME keys for both arms (the driver compares them)."""
    return {"model": model, "global_batch": batch * ga * world, "micro_batch_per_gpu": batch, "grad_accumulation": ga,
            "seq_len": seq, "lora_r": lora_r, "lora_dropout": 0.1, "parallelism": f"dp{world}", "optimizer": optimizer,
            "optimizer_reset": "magnitude_pruning 0.9" if reset.get("optimizer_magnitude_pruning") else "reset (0.999 random pruning)",
            "l2": "per-step working set (weights + activations, >1.5 GB) exceeds the 126 MB L2; no flush"}


def first_nonfinite(per_rank_log):
    """per_rank_log: [world, n_steps] float tensor (host).  -> (step, rank) of the first non-finite entry, or (None, None)."""
    import torch

    bad = ~torch.isfinite(per_rank_log)
    if not bool(bad.any()):
        return None, None
    steps = bad.any(0).nonzero().flatten()
    s = int(steps[0])
    r = int(bad[:, s].nonzero().flatten()[0])
    return s, r


DUMP_PER_PARAM = 4096  # sampled entries per parameter tensor
DUMP_LIMIT_BYTES = 64 << 20


def parameter_sample(model, per_param=DUMP_PER_PARAM, seed=0):
    """float32 [sum of min(numel, per_param)]: every parameter (module order) at positions drawn from a fixed seed, so the same
    model configuration always yields the same positions."""
    import torch

    g = torch.Generator().manual_seed(seed)
    parts = []
    for _, p in model.named_parameters():
        n = p.numel()
        idx = torch.randint(0, n, (per_param,), generator=g) if n > per_param else torch.arange(n)
        parts.append(p.detach().flatten()[idx.to(p.device)].float().cpu())
    return torch.cat(parts)


def dump_outputs(out_dir, model_name, loss, grad_norm, model):
    """The arrays a caller of the training step holds after the last timed step: its loss, the gradient norm of that update and
    (sampled) the parameters it produced."""
    import numpy as np

    arrays = {"loss": np.array([float(loss)], dtype=np.float32),
              "grad_norm": grad_norm.detach().float().reshape(-1).cpu().numpy(),
              "params_sample": parameter_sample(model).numpy()}
    nbytes = sum(a.nbytes for a in arrays.values())
    if nbytes > DUMP_LIMIT_BYTES // 2:  # one half each for the headline model and the llama_1b block
        raise SystemExit(f"--dump-outputs: {model_name} outputs take {nbytes} bytes, more than {DUMP_LIMIT_BYTES // 2}")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{model_name}_{name}.npy"), a)


def gather_rows(t):
    """all_gather a 1-D device tensor -> [world, n] on the host."""
    import torch
    import torch.distributed as dist

    world = dist.get_world_size()
    out = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(out, t)
    return torch.stack(out).float().cpu()


# --------------------------------------------------------------------------------------------- our arm
def run_ours_case(args, info, model, steps, warmup, rank, local, world):
    import torch

    from relora_b200.engine.api import TrainingEngine
    from relora_b200.models import load_config
    from relora_b200.ops import native

    rec = RECIPES.get(model, RECIPES["llama_250m"])
    batch, ga = args.batch or rec["batch"], args.ga or rec["ga"]
    cfg_path = os.path.join(ROOT, "configs", f"{model}.json")
    vocab = load_config(cfg_path).vocab_size
    eng = TrainingEngine.build(
        info, model_config=cfg_path, batch_size=batch, gradient_accumulation=ga,
        total_batch_size=batch * ga * world, max_length=args.seq, use_peft=True, lora_r=args.lora_r,
        relora=5000, cycle_length=5000, scheduler="cosine_restarts", warmup_steps=500, restart_warmup_steps=100,
        lr=1e-3, num_training_steps=20000, dtype="bfloat16", device="cuda",
        engine=args.engine, comm=args.comm, optimizer=args.optimizer, cuda_graphs=args.cuda_graphs.lower() == "true",
        frozen_dtype=args.frozen_dtype, attention=args.attention, **rec["reset"],
    )
    dev = info.device
    n_total = warmup + steps
    host = make_tokens(n_total, ga, batch, args.seq, vocab, rank, pinned=True)
    dev_tokens = host.to(dev)
    C = native.require()
    n_log = warmup + 2 * steps
    loss_log = torch.full((n_log,), float("nan"), dtype=torch.float32, device=dev)   # this rank's loss, before the mean
    norm_log = torch.zeros(n_log, dtype=torch.float32, device=dev)
    cursor = [0]
    last = {}  # what the most recent step returned to its caller

    def record():
        i = cursor[0]
        loss_log[i].copy_(eng.last_local_loss)
        norm_log[i].copy_(eng.last_grad_norm.reshape(()))
        cursor[0] = i + 1

    def dev_step(i):
        last["loss"] = eng.train_step_device(dev_tokens[i])
        record()

    for i in range(warmup):
        dev_step(i)
    if hasattr(eng.stepper, "mark_launch_window"):
        eng.stepper.mark_launch_window()
    else:
        C.reset_launch_count()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    secs = timed(lambda i: dev_step(warmup + i), steps, world, dev)
    clocks = sampler.stop() if sampler else None
    launches = int(getattr(eng.stepper, "launches_in_window", lambda n: C.launch_count())(steps))
    tokens = eng.tokens_per_step * steps
    value = tokens / secs

    e2e = None
    if not args.no_e2e:
        losses = []

        def e2e_step(i):
            last["loss"] = eng.train_step(host[warmup + i])
            losses.append(last["loss"])
            record()

        secs2 = timed(e2e_step, steps, world, dev)
        bi = host[0].numel() * host.element_size()
        e2e = {"value": tokens / secs2, "unit": "tokens/s", "h2d_bytes_per_step": bi, "d2h_bytes_per_step": 4,
               "ms_per_step": secs2 / steps * 1e3, "last_loss": losses[-1]}
    # ---- validity: per-rank losses, gradient norms, parameters
    n_done = cursor[0]
    losses_all = gather_rows(loss_log[:n_done])
    norms_all = gather_rows(norm_log[:n_done])
    s_loss, r_loss = first_nonfinite(losses_all)
    s_norm, r_norm = first_nonfinite(norms_all)
    p_bad = torch.tensor([float((~torch.isfinite(eng.stepper.store.params.float())).sum())], device=dev)
    p_bad_all = gather_rows(p_bad).flatten()
    bad_step = min([s for s in (s_loss, s_norm) if s is not None], default=None)
    valid = bad_step is None and float(p_bad_all.sum()) == 0
    out = {
        "value": value, "unit": "tokens/s", "ms_per_step": secs / steps * 1e3, "steps": steps, "warmup": warmup,
        "config": case_config(model, batch, ga, args.seq, args.lora_r, world, args.optimizer, rec["reset"]),
        "impl_details": {"executor": type(eng.stepper).__name__, "comm": getattr(eng.stepper.sync, "transport", "none"),
                         "attention": "tcgen05 (this repo)" if getattr(eng.stepper, "native_attn", False) else "torch SDPA (cuDNN)",
                         "cuda_graphs": bool(getattr(eng.stepper, "use_graphs", False))},
        "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "valid": valid,
        "final_loss": float(losses_all[:, n_done - 1].mean()), "final_grad_norm": float(norms_all[0, n_done - 1]),
    }
    if not valid:
        out["nonfinite_at_step"] = bad_step
        out["nonfinite_rank"] = r_loss if (s_loss is not None and s_loss == bad_step) else r_norm
        out["nonfinite_params_per_rank"] = [int(x) for x in p_bad_all]
        if rank == 0:
            print(f"[bench] NON-FINITE training state ({model}): first bad step {bad_step}, per-rank losses at that step "
                  f"{losses_all[:, bad_step].tolist() if bad_step is not None else None}, norms "
                  f"{norms_all[:, bad_step].tolist() if bad_step is not None else None}", file=sys.stderr)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model, last["loss"], eng.last_grad_norm, eng.model)
    # ---- free everything before the next case (graphs, symmetric buffers, activations)
    del eng, dev_tokens, host
    gc.collect()
    torch.cuda.empty_cache()
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist

    rank, local, world = setup_dist(args)
    from relora_b200.ops import native
    from relora_b200.parallel.dist import init_distributed

    info = init_distributed("cuda", "nccl")
    head_model = args.model or "llama_250m"
    head = run_ours_case(args, info, head_model, args.steps, args.warmup, rank, local, world)
    extra = None
    if args.model is None and not args.no_1b:
        extra = run_ours_case(args, info, "llama_1b", max(1, min(args.steps, args.steps_1b)), max(3, min(args.warmup, 3)), rank, local, world)
    valid = head["valid"] and (extra is None or extra["valid"])
    if rank == 0:
        out = {
            "metric": METRIC, "value": head["value"], "unit": "tokens/s", "n_gpus": world, "steps": head["steps"], "warmup": head["warmup"],
            "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if args.frozen_dtype not in ("fp8", "fp8_full") else f"bf16 ({args.frozen_dtype}: fp8 tensor-core GEMMs for the frozen weights)",
            "data": "synthetic token ids (uniform over the vocabulary without the padding row), random-init weights", "impl": "ours", "config": head["config"],
            "impl_details": head["impl_details"], "clocks": head["clocks"], "e2e": head["e2e"], "gpu_launches": head["gpu_launches"],
            "valid": valid, "final_loss": head["final_loss"], "final_grad_norm": head["final_grad_norm"],
            "native_so": native.so_path(),
        }
        for k in ("nonfinite_at_step", "nonfinite_rank", "nonfinite_params_per_rank"):
            if k in head:
                out[k] = head[k]
        if extra is not None:
            out["llama_1b"] = extra
        print(json.dumps(out))
    dist.barrier()
    dist.destroy_process_group()
    return 0 if valid else EXIT_NONFINITE


# --------------------------------------------------------------------------------------------- reference arm
def _stub_missing_modules():
    """The reference imports bitsandbytes at module level (relora.py:10-11); the package is not in this image.
    A stub satisfies the import — the non-quantised code path never touches it.  Nothing in baseline/_ref is edited."""
    for name in ("bitsandbytes", "bitsandbytes.nn", "bitsandbytes.functional"):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules["bitsandbytes"].nn = sys.modules["bitsandbytes.nn"]
    sys.modules["bitsandbytes"].functional = sys.modules["bitsandbytes.functional"]


def run_reference_case(args, mods, model_name, steps, warmup, rank, local, world):
    import torch
    import torch.distributed as dist

    training_utils, LlamaForCausalLM, ReLoRaModel, AutoConfig = mods
    rec = RECIPES.get(model_name, RECIPES["llama_250m"])
    batch, ga = args.batch or rec["batch"], args.ga or rec["ga"]
    # same steps as the reference's torchrun_main.main (:477-492, 531-553, 598-622, 631-691, 768-826)
    torch.manual_seed(0)
    device = f"cuda:{local}"
    cfg = AutoConfig.from_pretrained(os.path.join(ROOT, "configs", f"{model_name}.json"))
    model = LlamaForCausalLM(cfg)
    model = ReLoRaModel(model, r=args.lora_r, lora_alpha=32, lora_dropout=0.1, target_modules=["attn", "attention", "mlp"],
                        trainable_scaling=False, keep_original_weights=True, lora_only=False, quantize=None, use_double_quant=True)
    model = model.to(device=device, dtype=torch.bfloat16)
    model = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local], output_device=local)
    trainable = [p for p in model.parameters() if p.requires_grad]
    optimizer = torch.optim.AdamW(trainable, lr=1e-3, weight_decay=0.0, betas=(0.9, 0.999))
    scheduler = training_utils.get_scheculer(optimizer=optimizer, scheduler_type="cosine_restarts", num_training_steps=20000,
                                             warmup_steps=500, min_lr_ratio=0.1, cycle_length=5000, restart_warmup_steps=100,
                                             adjust_step=0)
    n_total = warmup + steps
    host = make_tokens(n_total, ga, batch, args.seq, cfg.vocab_size, rank, pinned=True)
    dev_tokens = host.to(device)
    state = {"loss": 0.0, "done": 0, "failed": None}

    def step(src_tokens):
        loss_info = torch.tensor([0.0, 0.0, 0.0], device=device)
        for mb in range(ga):
            batch_ = {"input_ids": src_tokens[mb].to(device)}  # no-op for device-resident tokens
            loss = model(**batch_, labels=batch_["input_ids"]).loss
            loss_info[0] += loss.detach()
            loss_info[1] += 1
            loss_info[2] += torch.isnan(loss).float()
            (loss / ga).backward()
        grad_norm = torch.nn.utils.clip_grad_norm_(trainable, 1.0, error_if_nonfinite=True)
        if rank == 0:
            grad_norm.item()  # the reference logs it to wandb every update (torchrun_main.py:807-808)
        dist.all_reduce(loss_info, op=dist.ReduceOp.SUM)
        _loss = loss_info[0] / loss_info[1]
        if loss_info[2] == 0:
            optimizer.step()
            scheduler.step()
        optimizer.zero_grad()
        state["done"] += 1
        return _loss

    secs = secs2 = None
    clocks = None
    try:
        for i in range(warmup):
            step(dev_tokens[i])
        sampler = ClockSampler(local) if rank == 0 else None
        if sampler:
            sampler.start()
        try:
            secs = timed(lambda i: step(dev_tokens[warmup + i]), steps, world, torch.device(device))
        finally:
            clocks = sampler.stop() if sampler else None
        if not args.no_e2e:
            def e2e_step(i):
                state["loss"] = float(step(host[warmup + i]).item())
            secs2 = timed(e2e_step, steps, world, torch.device(device))
    except RuntimeError as e:  # clip_grad_norm_(error_if_nonfinite=True): every rank sees the same all-reduced gradients and raises
        state["failed"] = f"{type(e).__name__}: {e}"[:300]
    tokens = batch * ga * args.seq * world * steps
    out = {
        "value": tokens / secs if secs else None, "unit": "tokens/s", "ms_per_step": secs / steps * 1e3 if secs else None,
        "steps": steps, "warmup": warmup,
        "config": case_config(model_name, batch, ga, args.seq, args.lora_r, world, "adam", rec["reset"]),
        "impl_details": {"executor": "reference torch eager + DDP", "comm": "nccl (DDP buckets, every micro-batch)",
                         "attention": "torch SDPA", "cuda_graphs": False},
        "clocks": clocks, "gpu_launches": 0, "valid": state["failed"] is None and math.isfinite(state["loss"]),
        "e2e": ({"value": tokens / secs2, "unit": "tokens/s", "h2d_bytes_per_step": host[0].numel() * host.element_size(),
                 "d2h_bytes_per_step": 4, "ms_per_step": secs2 / steps * 1e3, "last_loss": state["loss"]} if secs2 else None),
    }
    if not out["valid"]:
        out["nonfinite_at_step"] = state["done"]
        out["failed"] = state["failed"] or "non-finite loss"
    del model, optimizer, scheduler, trainable, dev_tokens, host
    gc.collect()
    torch.cuda.empty_cache()
    return out


def run_reference(args):
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "peft_pretraining")):
        print(json.dumps({"impl": "reference", "unavailable": "baseline/_ref is not installed (pip --target baseline/_ref /root/reference)"}))
        return 0
    import torch  # noqa: F401

    rank, local, world = setup_dist(args)
    import torch.distributed as dist

    _stub_missing_modules()
    sys.path.insert(0, ref_dir)
    try:
        from peft_pretraining import training_utils
        from peft_pretraining.modeling_llama import LlamaForCausalLM
        from peft_pretraining.relora import ReLoRaModel
        from transformers import AutoConfig
    except Exception as e:
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": f"reference import failed: {type(e).__name__}: {e}"[:300]}))
        dist.destroy_process_group()
        return 0
    mods = (training_utils, LlamaForCausalLM, ReLoRaModel, AutoConfig)
    head = run_reference_case(args, mods, args.model or "llama_250m", args.steps, args.warmup, rank, local, world)
    extra = None
    if args.model is None and not args.no_1b and head["valid"]:
        extra = run_reference_case(args, mods, "llama_1b", max(1, min(args.steps, args.steps_1b)), max(3, min(args.warmup, 3)), rank, local, world)
    valid = head["valid"] and (extra is None or extra["valid"])
    if rank == 0:
        out = {
            "metric": METRIC, "value": head["value"], "unit": "tokens/s", "n_gpus": world, "steps": head["steps"], "warmup": head["warmup"],
            "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic token ids (uniform over the vocabulary without the padding row), random-init weights", "impl": "reference", "config": head["config"],
            "impl_details": head["impl_details"], "clocks": head["clocks"], "e2e": head["e2e"], "gpu_launches": 0, "valid": valid,
        }
        for k in ("nonfinite_at_step", "failed"):
            if k in head:
                out[k] = head[k]
        if extra is not None:
            out["llama_1b"] = extra
        print(json.dumps(out))
    dist.barrier()
    dist.destroy_process_group()
    return 0 if valid else EXIT_NONFINITE


class _QuietStdout:
    """Route everything libraries write to fd 1 (e.g. NCCL's version banner) to stderr so that stdout carries exactly
    the one JSON line of the bench contract."""

    def __enter__(self):
        sys.stdout.flush()
        self._saved = os.dup(1)
        os.dup2(2, 1)
        real = os.fdopen(os.dup(self._saved), "w")
        builtins_print = print

        def emit(*a, **k):
            if k.get("file") is not None:
                builtins_print(*a, **k)
            else:
                builtins_print(*a, **dict(k, file=real, flush=True))

        globals()["print"] = emit
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self._saved, 1)
        os.close(self._saved)
        globals().pop("print", None)
        return False


if __name__ == "__main__":
    a = parse()
    with _QuietStdout():
        rc = run_reference(a) if a.impl == "reference" else run_ours(a)
    sys.exit(rc)
