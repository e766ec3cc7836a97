"""Model parity: Llama vs the reference implementation, Pythia vs HF transformers, generation, seq-classification."""
import os

import pytest
import torch

from relora_b200.models import GPTNeoXForCausalLM, LlamaForCausalLM, LlamaForSequenceClassification, SimpleConfig, load_config

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CFG = os.path.join(ROOT, "configs", "llama_9m.json")


def test_llama_matches_reference_logits_and_grads():
    import reference_golden as rg

    golden = rg.load()
    ours = LlamaForCausalLM(load_config(CFG))
    assert set(ours.state_dict()) == set(golden["llama:state_dict_keys"])  # identical key set incl. rotary inv_freq buffers
    rg.seed_parameters_(ours)
    ids = rg.seeded_ids(**rg.LLAMA_IDS)
    b = ours(input_ids=ids, labels=ids)
    assert torch.allclose(rg.sampled(golden, "llama:logits", b.logits), torch.from_numpy(golden["llama:logits"]), atol=1e-5)
    assert abs(float(golden["llama:loss"]) - float(b.loss)) < 1e-6
    b.loss.backward()
    for n, q in ours.named_parameters():
        assert torch.allclose(rg.sampled(golden, f"llama:grad:{n}", q.grad), torch.from_numpy(golden[f"llama:grad:{n}"]), atol=1e-5), n
        assert abs(float(q.grad.norm()) - float(golden[f"llama:grad_norm:{n}"])) <= 1e-5 + 1e-4 * float(golden[f"llama:grad_norm:{n}"]), n
    # chunked LM-head loss == materialised-logits loss
    c = ours(input_ids=ids, labels=ids, return_logits=False)
    assert c.logits is None and abs(float(c.loss) - float(b.loss)) < 1e-5


def test_llama_generate_uses_cache_consistently():
    torch.manual_seed(0)
    m = LlamaForCausalLM(load_config(CFG)).eval()
    ids = torch.randint(0, 32000, (1, 7))
    out = m.generate(ids, max_new_tokens=5)
    assert out.shape == (1, 12)
    # greedy continuation without cache gives the same tokens
    cur = ids
    for _ in range(5):
        nxt = m(input_ids=cur).logits[:, -1].argmax(-1, keepdim=True)
        cur = torch.cat([cur, nxt], 1)
    assert torch.equal(out, cur)


def test_param_counts_match_reference_table():
    # SURVEY.md §2.4: llama_9m 9.02 M; llama_100m 100.117 M (reference notebooks/02 cell 0)
    assert LlamaForCausalLM(load_config(CFG)).num_parameters() == 9_021_568
    cfg = load_config(os.path.join(ROOT, "configs", "llama_100m.json"))
    with torch.device("meta"):
        m = LlamaForCausalLM.__new__(LlamaForCausalLM)
        torch.nn.Module.__init__(m)
        from relora_b200.models.llama import LlamaModel

        m.config = cfg
        m.model = LlamaModel(cfg)
        m.lm_head = torch.nn.Linear(cfg.hidden_size, cfg.vocab_size, bias=False)
    assert sum(p.numel() for p in m.parameters()) == 100_117_120


def test_sequence_classification_head():
    cfg = load_config(CFG)
    cfg.num_labels = 3
    cfg.pad_token_id = 0
    m = LlamaForSequenceClassification(cfg)
    ids = torch.tensor([[5, 6, 7, 0, 0], [8, 9, 10, 11, 12]])
    out = m(input_ids=ids, labels=torch.tensor([1, 2]))
    assert out.logits.shape == (2, 3) and out.loss.ndim == 0
    full = m.score(m.model(input_ids=ids)[0])
    assert torch.allclose(out.logits[0], full[0, 2]) and torch.allclose(out.logits[1], full[1, 4])


@pytest.mark.parametrize("parallel", [True, False])
def test_pythia_matches_hf(parallel):
    transformers = pytest.importorskip("transformers")
    kw = dict(vocab_size=512, hidden_size=64, num_hidden_layers=2, num_attention_heads=4, intermediate_size=256, rotary_pct=0.25,
              max_position_embeddings=128, use_parallel_residual=parallel, hidden_act="gelu", layer_norm_eps=1e-5)
    try:
        hf_cfg = transformers.GPTNeoXConfig(**kw)
        torch.manual_seed(0)
        hf = transformers.GPTNeoXForCausalLM(hf_cfg).eval()
    except Exception as e:  # API drift
        pytest.skip(f"HF GPTNeoX unavailable: {e}")
    ours = GPTNeoXForCausalLM(SimpleConfig(model_type="gpt_neox", **kw)).eval()
    missing, unexpected = ours.load_hf_state_dict(hf.state_dict(), strict=True)
    ids = torch.randint(0, 512, (1, 17))
    with torch.no_grad():
        a = hf(input_ids=ids).logits
        b = ours(input_ids=ids).logits
    assert torch.allclose(a, b, atol=2e-5), float((a - b).abs().max())
    # batch > 1 in eval takes the explicit-mask branch
    ids2 = torch.randint(0, 512, (3, 9))
    with torch.no_grad():
        assert torch.allclose(hf(input_ids=ids2).logits, ours(input_ids=ids2).logits, atol=2e-5)
    # cache consistency
    g = ours.generate(ids[:, :5], max_new_tokens=4)
    cur = ids[:, :5]
    for _ in range(4):
        cur = torch.cat([cur, ours(input_ids=cur).logits[:, -1].argmax(-1, keepdim=True)], 1)
    assert torch.equal(g, cur)


def test_pythia_relora_wrap_targets():
    from relora_b200.relora import ReLoRaLinear, ReLoRaModel

    m = GPTNeoXForCausalLM(SimpleConfig(model_type="gpt_neox", vocab_size=128, hidden_size=32, num_hidden_layers=1,
                                        num_attention_heads=2, intermediate_size=64, max_position_embeddings=64))
    w = ReLoRaModel(m, r=4, lora_alpha=8, target_modules=["attn", "attention", "mlp"])
    names = sorted(n for n, mod in w.named_modules() if isinstance(mod, ReLoRaLinear))
    assert names == ["wrapped_model.gpt_neox.layers.0.attention.dense", "wrapped_model.gpt_neox.layers.0.attention.query_key_value",
                     "wrapped_model.gpt_neox.layers.0.mlp.dense_4h_to_h", "wrapped_model.gpt_neox.layers.0.mlp.dense_h_to_4h"]
    assert all(mod.bias is not None for mod in w.relora_modules())  # biases carried over
    ids = torch.randint(0, 128, (2, 8))
    w(input_ids=ids, labels=ids).loss.backward()


def test_rope_scaling_variants():
    from relora_b200.models.pythia import (GPTNeoXDynamicNTKScalingRotaryEmbedding, GPTNeoXLinearScalingRotaryEmbedding,
                                           GPTNeoXRotaryEmbedding)

    base = GPTNeoXRotaryEmbedding(16, 32)
    lin = GPTNeoXLinearScalingRotaryEmbedding(16, 32, scaling_factor=2.0)
    x = torch.zeros(1)
    c0, _ = base(x, 32)
    c1, _ = lin(x, 32)
    assert torch.allclose(c1[0, 0, 2], c0[0, 0, 1])  # position 2 / factor 2 == position 1
    dyn = GPTNeoXDynamicNTKScalingRotaryEmbedding(16, 32, scaling_factor=2.0)
    inv_before = dyn.inv_freq.clone()
    dyn(x, 64)  # beyond the trained context: base grows
    assert not torch.equal(inv_before, dyn.inv_freq) and dyn.cos_cached.shape[2] == 64


def test_sequence_starting_with_the_padding_row_overflows_the_reference_gradient():
    """Root cause of round 1's non-finite 4-/8-GPU benchmark runs (both arms).  The configs' ``pad_token_id = -1`` makes row V-1
    the embedding's zero padding row; a sequence that *starts* with it keeps an exactly-zero residual row through every layer
    (v = 0, no biases), and RMSNorm's backward at x = 0 multiplies the gradient by 1/sqrt(eps) = 1000 per norm: it overflows
    fp32 within ~12 layers of the *unmodified reference model* (stored in tests/golden), and of ours on the same weights.
    Synthetic token generators therefore never emit that id (real tokenised text does not contain it either)."""
    import reference_golden as rg

    from relora_b200.data.synthetic import SyntheticTokens

    golden = rg.load()
    cfg = load_config(os.path.join(ROOT, "configs", "llama_35m.json"))
    cfg.num_hidden_layers = rg.PADDING_LAYERS
    V = cfg.vocab_size
    assert V == int(golden["padding:vocab"])
    ref_ordinary, ref_padding_row = float(golden["padding:norm_ordinary"]), float(golden["padding:norm_padding_row"])
    assert ref_ordinary < 1e3                   # reference, ordinary token: ordinary gradient
    assert not (ref_padding_row < 1e30)         # reference, padding row first: overflow (inf / nan)
    model = LlamaForCausalLM(cfg)
    rg.seed_parameters_(model)
    norms = rg.embedding_grad_norms(model, V)
    assert abs(norms[5] - ref_ordinary) < 1e-4 * ref_ordinary
    assert not (norms[V - 1] < 1e30)
    # ... which is why the synthetic sources draw from [0, V - 1)
    ds = SyntheticTokens(64, 128, V, seed=3)
    assert max(int(ds[i]["input_ids"].max()) for i in range(64)) < V - 1
