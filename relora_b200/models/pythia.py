"""Pythia / GPT-NeoX causal LM with HF-compatible parameter names.

Parity target: reference ``peft_pretraining/modeling_pythia.py``:

* fused ``query_key_value`` ``Linear(h, 3h)`` *with bias*, stored head-interleaved
  ``[nh, (q|k|v), hd]`` (``:108, :172-183``);
* partial rotary embedding on the first ``rotary_pct·hd`` dims (``:97, :185-197``) with base,
  linear-scaled and dynamic-NTK tables (``:303-375``);
* SDPA attention: causal without mask when training or batch 1, additive padding+causal mask
  otherwise (``:262-288``);
* GELU MLP ``4h`` with biases (``:395-406``), ``nn.LayerNorm`` pre-norms, hidden dropouts,
  parallel-residual option (``:409-463``);
* untied ``embed_out`` head, shifted cross-entropy (``:701-857``).

Module / parameter names match HF (``gpt_neox.layers.N.attention.query_key_value.weight`` …) so HF
Pythia checkpoints load; ``ReLoRaModel`` wraps ``attention.query_key_value``, ``attention.dense``,
``mlp.dense_h_to_4h`` and ``mlp.dense_4h_to_h`` (their names contain "attention" / "mlp").
"""
from __future__ import annotations

import os
from typing import List, Optional, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

from .llama import CausalLMOutput, _PretrainedMixin, rotate_half

__all__ = [
    "GPTNeoXRotaryEmbedding",
    "GPTNeoXLinearScalingRotaryEmbedding",
    "GPTNeoXDynamicNTKScalingRotaryEmbedding",
    "GPTNeoXAttention",
    "GPTNeoXMLP",
    "GPTNeoXLayer",
    "GPTNeoXModel",
    "GPTNeoXForCausalLM",
]


class GPTNeoXRotaryEmbedding(nn.Module):
    def __init__(self, dim: int, max_position_embeddings: int, base: float = 10000, device=None):
        super().__init__()
        self.dim = dim
        self.max_position_embeddings = max_position_embeddings
        self.base = base
        self.register_buffer("inv_freq", self._inv_freq(base, device))
        self._set_cos_sin_cache(max_position_embeddings, self.inv_freq.device)

    def _inv_freq(self, base, device):
        return 1.0 / (base ** (torch.arange(0, self.dim, 2, dtype=torch.float32, device=device) / self.dim))

    def _positions(self, seq_len, device):
        return torch.arange(seq_len, device=device, dtype=self.inv_freq.dtype)

    def _set_cos_sin_cache(self, seq_len: int, device):
        self.max_seq_len_cached = seq_len
        freqs = torch.outer(self._positions(seq_len, device), self.inv_freq.to(device))
        emb = torch.cat((freqs, freqs), dim=-1)
        # plain attributes (not buffers) upstream: they do not follow ``.to(dtype)``
        self.cos_cached = emb.cos()[None, None]
        self.sin_cached = emb.sin()[None, None]

    def forward(self, x, seq_len: int):
        if seq_len > self.max_seq_len_cached:
            self._set_cos_sin_cache(seq_len, x.device)
        return self.cos_cached[:, :, :seq_len].to(x.device), self.sin_cached[:, :, :seq_len].to(x.device)


class GPTNeoXLinearScalingRotaryEmbedding(GPTNeoXRotaryEmbedding):
    """Positions divided by ``scaling_factor`` (position interpolation)."""

    def __init__(self, dim, max_position_embeddings, base=10000, device=None, scaling_factor: float = 1.0):
        self.scaling_factor = scaling_factor
        super().__init__(dim, max_position_embeddings, base, device)

    def _positions(self, seq_len, device):
        return super()._positions(seq_len, device) / self.scaling_factor


class GPTNeoXDynamicNTKScalingRotaryEmbedding(GPTNeoXRotaryEmbedding):
    """Base grows with the sequence length once it exceeds the trained context (dynamic NTK)."""

    def __init__(self, dim, max_position_embeddings, base=10000, device=None, scaling_factor: float = 1.0):
        self.scaling_factor = scaling_factor
        super().__init__(dim, max_position_embeddings, base, device)

    def _set_cos_sin_cache(self, seq_len, device):
        if seq_len > self.max_position_embeddings:
            grow = (self.scaling_factor * seq_len / self.max_position_embeddings) - (self.scaling_factor - 1)
            base = self.base * grow ** (self.dim / (self.dim - 2))
            self.register_buffer("inv_freq", self._inv_freq(base, device))
        super()._set_cos_sin_cache(seq_len, device)


def apply_partial_rotary(q, k, cos, sin, position_ids):
    """Rotate ``q``/``k`` (already sliced to the rotary dims) at ``position_ids``."""
    cos = cos[0, 0][position_ids].unsqueeze(1)
    sin = sin[0, 0][position_ids].unsqueeze(1)
    return (q * cos) + (rotate_half(q) * sin), (k * cos) + (rotate_half(k) * sin)


def _rope_settings(config):
    """(rotary fraction, base, scaling dict) from either config dialect: the classic GPT-NeoX fields ``rotary_pct`` /
    ``rotary_emb_base`` / ``rope_scaling`` (modeling_pythia.py:95-106 of the reference, checkpoints' ``config.json``) or the
    ``rope_parameters`` dict that transformers >= 5 folds them into (``partial_rotary_factor``, ``rope_theta``, ``rope_type``, ``factor``)."""
    rp = getattr(config, "rope_parameters", None) or {}
    pct = getattr(config, "rotary_pct", None)
    if pct is None:
        pct = rp.get("partial_rotary_factor", getattr(config, "partial_rotary_factor", 0.25))
    base = getattr(config, "rotary_emb_base", None)
    if base is None:
        base = rp.get("rope_theta", getattr(config, "rope_theta", 10000))
    scaling = getattr(config, "rope_scaling", None)
    if (scaling is None or not scaling.get("type", scaling.get("rope_type"))) and rp.get("rope_type") not in (None, "default"):
        scaling = {"type": rp["rope_type"], "factor": rp.get("factor", 1.0)}
    return float(pct), base, scaling


def _make_rope(config, rotary_ndims):
    _, base, scaling = _rope_settings(config)
    if scaling is None or scaling.get("type", scaling.get("rope_type")) in (None, "default"):
        return GPTNeoXRotaryEmbedding(rotary_ndims, config.max_position_embeddings, base=base)
    kind = scaling.get("type", scaling.get("rope_type"))
    factor = scaling["factor"]
    if kind == "linear":
        return GPTNeoXLinearScalingRotaryEmbedding(rotary_ndims, config.max_position_embeddings, base=base, scaling_factor=factor)
    if kind == "dynamic":
        return GPTNeoXDynamicNTKScalingRotaryEmbedding(rotary_ndims, config.max_position_embeddings, base=base, scaling_factor=factor)
    raise ValueError(f"Unknown RoPE scaling type {kind}")


class GPTNeoXAttention(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.num_attention_heads = config.num_attention_heads
        self.hidden_size = config.hidden_size
        if self.hidden_size % self.num_attention_heads != 0:
            raise ValueError("The hidden size is not divisble by the number of attention heads! Make sure to update them")
        self.head_size = self.hidden_size // self.num_attention_heads
        self.rotary_ndims = int(self.head_size * _rope_settings(config)[0])
        self.rotary_emb = _make_rope(config, self.rotary_ndims)
        bias = getattr(config, "attention_bias", True)
        self.query_key_value = nn.Linear(config.hidden_size, 3 * config.hidden_size, bias=bias)
        self.dense = nn.Linear(config.hidden_size, config.hidden_size, bias=bias)
        self.dropout_prob_attn = float(getattr(config, "attention_dropout", 0.0))

    def forward(self, hidden_states, attention_mask, position_ids, layer_past=None, use_cache=False):
        B, T, _ = hidden_states.shape
        qkv = self.query_key_value(hidden_states).view(B, T, self.num_attention_heads, 3 * self.head_size)
        # the native path is plain causal attention: it takes no padding mask, so batched eval with a mask stays on the masked
        # SDPA branch below (same condition as that branch's unmasked case)
        if (layer_past is None and not use_cache and getattr(position_ids, "_rb_default", False) and _native(qkv)
                and self.rotary_ndims % 2 == 0 and not self.training_dropout_active()
                and (attention_mask is None or B == 1 or self.training)):
            return self._forward_native(qkv, B, T)
        q = qkv[..., : self.head_size].permute(0, 2, 1, 3)
        k = qkv[..., self.head_size : 2 * self.head_size].permute(0, 2, 1, 3)
        v = qkv[..., 2 * self.head_size :].permute(0, 2, 1, 3)

        rd = self.rotary_ndims
        kv_len = T + (layer_past[0].shape[-2] if layer_past is not None else 0)
        cos, sin = self.rotary_emb(v, seq_len=kv_len)
        q_rot, k_rot = apply_partial_rotary(q[..., :rd], k[..., :rd], cos, sin, position_ids)
        # rotary tables stay fp32 upstream, so q/k are promoted and cast back ("downcast_qk")
        q = torch.cat((q_rot, q[..., rd:]), dim=-1).to(v.dtype)
        k = torch.cat((k_rot, k[..., rd:]), dim=-1).to(v.dtype)
        if layer_past is not None:
            k = torch.cat((layer_past[0], k), dim=-2)
            v = torch.cat((layer_past[1], v), dim=-2)
        present = (k, v) if use_cache else None

        p = self.dropout_prob_attn if self.training else 0.0
        if B == 1 or self.training:
            out = F.scaled_dot_product_attention(q, k, v, attn_mask=None, dropout_p=p, is_causal=q.shape[2] > 1)
        else:
            mask = attention_mask
            if T > 1:
                causal = torch.ones(T, kv_len, dtype=torch.bool, device=q.device).tril(diagonal=kv_len - T)
                cm = torch.zeros(T, kv_len, dtype=v.dtype, device=q.device).masked_fill(~causal, torch.finfo(v.dtype).min)
                cm = cm[None, None].expand(B, -1, -1, -1)
                mask = cm + attention_mask if attention_mask is not None else cm
            out = F.scaled_dot_product_attention(q, k, v, attn_mask=mask, dropout_p=p, is_causal=False)
        out = out.to(v.dtype).permute(0, 2, 1, 3).reshape(B, T, self.hidden_size)
        return self.dense(out), present


    def training_dropout_active(self) -> bool:
        return self.training and self.dropout_prob_attn > 0.0

    def _forward_native(self, qkv, B, T):
        """CUDA / bf16 training path: partial rotary in place on the fused projection output (csrc/neox.cu), then causal attention
        on the tcgen05 kernels when the head size allows (<= 64), torch SDPA otherwise.  Positions are 0..T-1 (no cache)."""
        from ..ops import fused

        nh, hd, rd = self.num_attention_heads, self.head_size, self.rotary_ndims
        cos, sin = self.rotary_emb(qkv, seq_len=T)
        qkv = fused.neox_rope(qkv, cos[0, 0].float().contiguous(), sin[0, 0].float().contiguous(), nh, hd, rd)
        q = qkv[..., :hd].permute(0, 2, 1, 3)
        k = qkv[..., hd : 2 * hd].permute(0, 2, 1, 3)
        v = qkv[..., 2 * hd :].permute(0, 2, 1, 3)
        if fused.native_attention_supported(q, hd) and os.environ.get("RELORA_B200_ATTENTION", "auto") != "sdpa":
            out = fused.causal_attention(q, k, v)
        else:
            out = F.scaled_dot_product_attention(q, k, v, attn_mask=None, dropout_p=0.0, is_causal=T > 1)
        out = out.permute(0, 2, 1, 3).reshape(B, T, self.hidden_size)
        return self.dense(out), None


def _native(x: torch.Tensor) -> bool:
    """CUDA + bf16 (and the extension present): the leaf ops of this file dispatch to csrc/neox.cu."""
    if not x.is_cuda:
        return False
    from ..ops import dispatch

    return dispatch.use_fused(x)


def _layer_norm(mod: nn.LayerNorm, x: torch.Tensor) -> torch.Tensor:
    if _native(x) and mod.elementwise_affine:
        from ..ops import fused

        if fused.layernorm_supported(x):
            return fused.layernorm(x, mod.weight, mod.bias, mod.eps)
    return mod(x)


class GPTNeoXMLP(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.dense_h_to_4h = nn.Linear(config.hidden_size, config.intermediate_size)
        self.dense_4h_to_h = nn.Linear(config.intermediate_size, config.hidden_size)
        act = getattr(config, "hidden_act", "gelu")
        if act in ("gelu",):
            self.act = nn.GELU()
        elif act in ("gelu_new", "gelu_fast", "gelu_pytorch_tanh"):
            self.act = nn.GELU(approximate="tanh")
        elif act == "relu":
            self.act = nn.ReLU()
        elif act == "silu":
            self.act = nn.SiLU()
        else:
            raise NotImplementedError(f"hidden_act={act}")

    def forward(self, x):
        z = self.dense_h_to_4h(x)
        if isinstance(self.act, nn.GELU) and _native(z) and z.numel() % 8 == 0:
            from ..ops import fused

            a = fused.gelu(z, tanh_approx=self.act.approximate == "tanh")
        else:
            a = self.act(z)
        return self.dense_4h_to_h(a)


class GPTNeoXLayer(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.use_parallel_residual = getattr(config, "use_parallel_residual", True)
        self.input_layernorm = nn.LayerNorm(config.hidden_size, eps=config.layer_norm_eps)
        self.post_attention_layernorm = nn.LayerNorm(config.hidden_size, eps=config.layer_norm_eps)
        hd = float(getattr(config, "hidden_dropout", 0.0))
        self.post_attention_dropout = nn.Dropout(hd)
        self.post_mlp_dropout = nn.Dropout(hd)
        self.attention = GPTNeoXAttention(config)
        self.mlp = GPTNeoXMLP(config)

    def forward(self, hidden_states, attention_mask=None, position_ids=None, layer_past=None, use_cache=False):
        attn, present = self.attention(_layer_norm(self.input_layernorm, hidden_states), attention_mask, position_ids, layer_past, use_cache)
        attn = self.post_attention_dropout(attn)
        if self.use_parallel_residual:
            # x = x + attn(ln1(x)) + mlp(ln2(x))
            mlp = self.post_mlp_dropout(self.mlp(_layer_norm(self.post_attention_layernorm, hidden_states)))
            hidden_states = mlp + attn + hidden_states
        else:
            attn = attn + hidden_states
            mlp = self.post_mlp_dropout(self.mlp(_layer_norm(self.post_attention_layernorm, attn)))
            hidden_states = mlp + attn
        return hidden_states, present


class _NeoXMixin(_PretrainedMixin):
    config_class_name = "GPTNeoXConfig"

    def _init_weights(self, module):
        std = getattr(self.config, "initializer_range", 0.02)
        if isinstance(module, nn.Linear):
            module.weight.data.normal_(mean=0.0, std=std)
            if module.bias is not None:
                module.bias.data.zero_()
        elif isinstance(module, nn.Embedding):
            module.weight.data.normal_(mean=0.0, std=std)
            if module.padding_idx is not None:
                module.weight.data[module.padding_idx].zero_()
        elif isinstance(module, nn.LayerNorm):
            module.bias.data.zero_()
            module.weight.data.fill_(1.0)

    # HF hub checkpoints differ in which non-parameter buffers they carry; load tolerantly
    _IGNORED_SUFFIXES = ("attention.bias", "attention.masked_bias", "rotary_emb.inv_freq")

    def load_hf_state_dict(self, state, strict: bool = True):
        own = self.state_dict()
        filtered = {k: v for k, v in state.items() if not (k.endswith(self._IGNORED_SUFFIXES) and k not in own)}
        missing, unexpected = self.load_state_dict(filtered, strict=False)
        missing = [k for k in missing if not k.endswith(self._IGNORED_SUFFIXES)]
        if strict and (missing or unexpected):
            raise RuntimeError(f"Error(s) loading state_dict: missing={missing} unexpected={list(unexpected)}")
        return missing, list(unexpected)

    @classmethod
    def from_pretrained(cls, path: str, revision: Optional[str] = None, **kwargs):
        """Load from a local directory (``config.json`` + weights).  Hub names need network access,
        which this engine does not assume; pre-download and pass the directory."""
        from .configs import load_config

        if not os.path.isdir(path):
            raise FileNotFoundError(
                f"{path!r} is not a local directory. Download the checkpoint "
                f"(revision={revision}) and pass its path via --model_name_or_path."
            )
        config = load_config(path)
        model = cls(config, **kwargs)
        bin_path = os.path.join(path, "pytorch_model.bin")
        if os.path.exists(bin_path):
            state = torch.load(bin_path, map_location="cpu", weights_only=True)
        else:
            from safetensors.torch import load_file

            state = load_file(os.path.join(path, "model.safetensors"))
        model.load_hf_state_dict(state, strict=True)
        return model


class GPTNeoXModel(nn.Module, _NeoXMixin):
    def __init__(self, config):
        super().__init__()
        self.config = config
        self.embed_in = nn.Embedding(config.vocab_size, config.hidden_size)
        self.emb_dropout = nn.Dropout(float(getattr(config, "hidden_dropout", 0.0)))
        self.layers = nn.ModuleList([GPTNeoXLayer(config) for _ in range(config.num_hidden_layers)])
        self.final_layer_norm = nn.LayerNorm(config.hidden_size, eps=config.layer_norm_eps)
        self.gradient_checkpointing = False

    def get_input_embeddings(self):
        return self.embed_in

    def set_input_embeddings(self, value):
        self.embed_in = value

    def forward(self, input_ids=None, attention_mask=None, position_ids=None, inputs_embeds=None,
                past_key_values=None, use_cache=None, output_hidden_states=False):
        if (input_ids is None) == (inputs_embeds is None):
            raise ValueError("You have to specify exactly one of input_ids or inputs_embeds")
        if inputs_embeds is None:
            inputs_embeds = self.embed_in(input_ids)
        B, T, _ = inputs_embeds.shape
        past_len = past_key_values[0][0].size(-2) if past_key_values is not None else 0
        default_positions = position_ids is None and past_len == 0
        if position_ids is None:
            position_ids = torch.arange(past_len, T + past_len, dtype=torch.long, device=inputs_embeds.device).unsqueeze(0).expand(B, T)
        else:
            position_ids = position_ids.view(-1, T).long()
        if default_positions:
            position_ids._rb_default = True  # positions 0..T-1: lets the attention take the in-place rotary kernel
        if attention_mask is not None:
            am = attention_mask.view(B, -1)[:, None, None, :].to(dtype=inputs_embeds.dtype)
            attention_mask = (1.0 - am) * torch.finfo(inputs_embeds.dtype).min
        use_cache = bool(use_cache) and not (self.gradient_checkpointing and self.training)

        h = self.emb_dropout(inputs_embeds)
        cache = [] if use_cache else None
        all_h = [] if output_hidden_states else None
        for i, layer in enumerate(self.layers):
            if all_h is not None:
                all_h.append(h)
            past = past_key_values[i] if past_key_values is not None else None
            if self.gradient_checkpointing and self.training:
                h, present = torch.utils.checkpoint.checkpoint(layer, h, attention_mask, position_ids, None, False, use_reentrant=False)
            else:
                h, present = layer(h, attention_mask, position_ids, past, use_cache)
            if cache is not None:
                cache.append(present)
        h = _layer_norm(self.final_layer_norm, h)
        if all_h is not None:
            all_h.append(h)
        return h, cache, all_h


class GPTNeoXForCausalLM(nn.Module, _NeoXMixin):
    def __init__(self, config):
        super().__init__()
        self.config = config
        self.gpt_neox = GPTNeoXModel(config)
        self.embed_out = nn.Linear(config.hidden_size, config.vocab_size, bias=False)
        self.post_init()

    def get_input_embeddings(self):
        return self.gpt_neox.embed_in

    def get_output_embeddings(self):
        return self.embed_out

    def set_output_embeddings(self, new):
        self.embed_out = new

    def forward(self, input_ids=None, attention_mask=None, position_ids=None, inputs_embeds=None,
                head_mask=None, past_key_values=None, labels=None, use_cache=None,
                output_attentions=None, output_hidden_states=None, return_dict=None):
        if head_mask is not None:
            raise ValueError("head_mask is not supported (attention runs as one fused kernel)")
        h, cache, all_h = self.gpt_neox(
            input_ids=input_ids, attention_mask=attention_mask, position_ids=position_ids,
            inputs_embeds=inputs_embeds, past_key_values=past_key_values, use_cache=use_cache,
            output_hidden_states=bool(output_hidden_states),
        )
        logits = self.embed_out(h)
        loss = None
        if labels is not None:
            labels = labels.to(logits.device)
            shift_logits = logits[:, :-1, :].contiguous()
            shift_labels = labels[:, 1:].contiguous()
            loss = F.cross_entropy(shift_logits.view(-1, shift_logits.size(-1)), shift_labels.view(-1))
        return CausalLMOutput(loss=loss, logits=logits, past_key_values=cache, hidden_states=all_h, attentions=None)

    @torch.no_grad()
    def generate(self, input_ids, max_new_tokens: int = 20, eos_token_id: Optional[int] = None):
        was_training = self.training
        self.eval()
        out = self(input_ids=input_ids, use_cache=True)
        cache, tokens, nxt_logits = out.past_key_values, input_ids, out.logits[:, -1]
        for _ in range(max_new_tokens):
            nxt = nxt_logits.argmax(-1, keepdim=True)
            tokens = torch.cat([tokens, nxt], dim=1)
            if eos_token_id is not None and bool((nxt == eos_token_id).all()):
                break
            out = self(input_ids=nxt, past_key_values=cache, use_cache=True)
            cache, nxt_logits = out.past_key_values, out.logits[:, -1]
        self.train(was_training)
        return tokens
