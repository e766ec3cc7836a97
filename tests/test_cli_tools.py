"""pretokenize.py -> trainer (--dataset_path) -> run_glue.py, fully offline with a tiny local tokenizer."""
import json
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CFG = os.path.join(ROOT, "configs", "llama_9m.json")


@pytest.fixture(scope="module")
def tiny_tokenizer(tmp_path_factory):
    from tokenizers import Tokenizer, models, pre_tokenizers
    from transformers import PreTrainedTokenizerFast

    words = ["<pad>", "</s>", "<unk>"] + [f"w{i}" for i in range(200)]
    tok = Tokenizer(models.WordLevel({w: i for i, w in enumerate(words)}, unk_token="<unk>"))
    tok.pre_tokenizer = pre_tokenizers.Whitespace()
    d = str(tmp_path_factory.mktemp("tok"))
    fast = PreTrainedTokenizerFast(tokenizer_object=tok, pad_token="<pad>", eos_token="</s>", unk_token="<unk>")
    fast.save_pretrained(d)
    return d


@pytest.fixture
def datasets_cache(tmp_path, monkeypatch):
    """``datasets.load_dataset`` caches under the user's Hugging Face home, which need not exist or be writable: keep it in
    the test's own directory."""
    from datasets import config

    cache = tmp_path / "hf_datasets"
    monkeypatch.setattr(config, "HF_DATASETS_CACHE", cache)
    monkeypatch.setattr(config, "DOWNLOADED_DATASETS_PATH", cache / "downloads")
    monkeypatch.setattr(config, "EXTRACTED_DATASETS_PATH", cache / "downloads" / "extracted")
    monkeypatch.setattr(config, "HF_MODULES_CACHE", cache / "modules")


def _corpus(path, n_lines=400, seed=0):
    import random

    rng = random.Random(seed)
    with open(path, "w") as f:
        for _ in range(n_lines):
            f.write(" ".join(f"w{rng.randrange(200)}" for _ in range(rng.randrange(5, 40))) + "\n")


def test_pretokenize_then_train(tiny_tokenizer, datasets_cache, tmp_path):
    import pretokenize
    from torchrun_main import main as train_main

    txt = str(tmp_path / "corpus.txt")
    _corpus(txt)
    out = pretokenize.main(pretokenize.parse_args(["--tokenizer", tiny_tokenizer, "--dataset", txt, "--sequence_length", "32",
                                                   "--save_dir", str(tmp_path / "pre"), "--num_cpu", "1"]))
    meta = json.load(open(os.path.join(out, "args.json")))
    assert meta["sequence_length"] == 32 and meta["vocab_size"] == 203
    with pytest.raises(ValueError):  # refuses to overwrite
        pretokenize.main(pretokenize.parse_args(["--tokenizer", tiny_tokenizer, "--dataset", txt, "--sequence_length", "32",
                                                 "--save_dir", str(tmp_path / "pre"), "--num_cpu", "1"]))
    import datasets

    dd = datasets.load_from_disk(out)
    assert all(len(r) == 32 for r in dd["train"]["input_ids"][:5])
    # the trainer needs a validation split: reuse train
    dd2 = datasets.DatasetDict({"train": dd["train"], "validation": dd["train"].select(range(8))})
    data_dir = str(tmp_path / "data")
    dd2.save_to_disk(data_dir)
    json.dump(meta, open(os.path.join(data_dir, "args.json"), "w"))
    res = train_main(["--model_config", CFG, "--dataset_path", data_dir, "--batch_size", "2", "--total_batch_size", "2",
                      "--max_length", "32", "--lr", "1e-3", "--scheduler", "cosine", "--warmup_steps", "1", "--num_training_steps", "3",
                      "--save_every", "3", "--eval_every", "100", "--save_dir", str(tmp_path / "run"), "--device", "cpu",
                      "--dtype", "float32", "--workers", "0", "--use_peft", "--lora_r", "4"])
    assert res["update_step"] == 3
    with pytest.raises(AssertionError):  # dataset sequence length must match --max_length
        train_main(["--model_config", CFG, "--dataset_path", data_dir, "--batch_size", "2", "--max_length", "64", "--num_training_steps", "1",
                    "--save_dir", str(tmp_path / "run2"), "--device", "cpu", "--dtype", "float32", "--workers", "0"])


def test_run_glue_on_local_files(tiny_tokenizer, datasets_cache, tmp_path):
    import random

    import run_glue
    from torchrun_main import main as train_main

    # a ReLoRA checkpoint to start from (exercises the LoRA-merge on load)
    ck = str(tmp_path / "pre")
    train_main(["--model_config", CFG, "--synthetic_data", "64", "--batch_size", "2", "--total_batch_size", "2", "--max_length", "16",
                "--lr", "1e-3", "--scheduler", "cosine", "--warmup_steps", "1", "--num_training_steps", "2", "--save_every", "2",
                "--eval_every", "100", "--save_dir", ck, "--device", "cpu", "--dtype", "float32", "--workers", "0", "--use_peft",
                "--lora_r", "4", "--init_lora_a", "kaiming"])
    rng = random.Random(0)

    def rows(n):
        out = []
        for _ in range(n):
            lab = rng.randrange(2)
            toks = [f"w{rng.randrange(0, 100) if lab == 0 else rng.randrange(100, 200)}" for _ in range(8)]
            out.append({"sentence1": " ".join(toks), "label": lab})
        return out

    tr, va = str(tmp_path / "train.json"), str(tmp_path / "val.json")
    for p, r in ((tr, rows(128)), (va, rows(32))):
        with open(p, "w") as f:
            for x in r:
                f.write(json.dumps(x) + "\n")
    res = run_glue.main(["--model_name_or_path", os.path.join(ck, "model_2"), "--tokenizer_name", tiny_tokenizer, "--train_file", tr,
                         "--validation_file", va, "--do_train", "--do_eval", "--max_seq_length", "16", "--per_device_train_batch_size", "16",
                         "--learning_rate", "1e-3", "--num_train_epochs", "2", "--output_dir", str(tmp_path / "glue"), "--device", "cpu"])
    assert "eval_accuracy" in res and 0.0 <= res["eval_accuracy"] <= 1.0
    assert os.path.exists(str(tmp_path / "glue" / "all_results.json"))


def test_glue_metrics():
    import numpy as np

    import run_glue

    p, l = np.array([1, 0, 1, 1]), np.array([1, 0, 0, 1])
    assert run_glue.glue_metrics("sst2", p, l) == {"accuracy": 0.75}
    m = run_glue.glue_metrics("mrpc", p, l)
    assert abs(m["f1"] - 0.8) < 1e-9
    assert abs(run_glue.glue_metrics("cola", p, l)["matthews_correlation"] - 0.5773502691896258) < 1e-9
    s = run_glue.glue_metrics("stsb", np.array([0.1, 0.4, 0.9]), np.array([0.0, 0.5, 1.0]))
    assert s["spearmanr"] == 1.0 and s["pearson"] > 0.98


def test_engine_only_flags_parse_and_do_not_alias_quantize():
    """--frozen_dtype fp8 / fp8_full are compute paths of the fused executor (not storage quantisation); --attention picks
    the attention kernels."""
    from relora_b200.config import parse_args

    base = ["--model_config", "configs/llama_9m.json", "--synthetic_data", "64", "--batch_size", "2", "--total_batch_size", "2",
            "--num_training_steps", "2", "--device", "cpu"]
    a = parse_args(base + ["--frozen_dtype", "fp8_full", "--attention", "native"])
    assert a.frozen_dtype == "fp8_full" and a.quantize is None and a.attention == "native"
    b = parse_args(base + ["--frozen_dtype", "nvfp4"])
    assert b.quantize == "nvfp4"
    c = parse_args(base)
    assert c.attention == "auto" and c.frozen_dtype is None
