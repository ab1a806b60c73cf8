"""Llama architecture description + the model-size presets the reference ships (reference: open_diloco/configs/*.json)."""
from __future__ import annotations

import json
import os
from dataclasses import asdict, dataclass, field
from pathlib import Path

_PRESET_DIR = Path(__file__).resolve().parent.parent / "configs"


@dataclass
class LlamaConfig:
    hidden_size: int = 1024
    intermediate_size: int = 2688
    num_hidden_layers: int = 12
    num_attention_heads: int = 16
    num_key_value_heads: int | None = None
    vocab_size: int = 32000
    rms_norm_eps: float = 1e-5
    rope_theta: float = 10000.0
    max_position_embeddings: int = 2048
    initializer_range: float = 0.02
    tie_word_embeddings: bool = False
    use_cache: bool = False
    model_type: str = "llama"
    architectures: list = field(default_factory=lambda: ["LlamaForCausalLM"])
    hidden_act: str = "silu"
    attention_bias: bool = False
    mlp_bias: bool = False
    bos_token_id: int = 1
    eos_token_id: int = 2

    def __post_init__(self):
        if self.num_key_value_heads is None:
            self.num_key_value_heads = self.num_attention_heads
        assert self.hidden_size % self.num_attention_heads == 0
        assert self.num_attention_heads % self.num_key_value_heads == 0
        if self.tie_word_embeddings or self.attention_bias or self.mlp_bias or self.hidden_act != "silu":
            raise NotImplementedError("only untied, bias-free, SiLU Llama is supported (the reference's model family)")

    @property
    def head_dim(self) -> int:
        return self.hidden_size // self.num_attention_heads

    @property
    def q_dim(self) -> int:
        return self.num_attention_heads * self.head_dim

    @property
    def kv_dim(self) -> int:
        return self.num_key_value_heads * self.head_dim

    @property
    def qkv_dim(self) -> int:
        return self.q_dim + 2 * self.kv_dim

    # -------------------------------------------------------------- io
    @classmethod
    def from_dict(cls, d: dict) -> "LlamaConfig":
        known = {f for f in cls.__dataclass_fields__}
        cfg = cls(**{k: v for k, v in d.items() if k in known})
        # head_dim is derived (hidden_size / num_attention_heads: the engine's q projection is hidden_size wide); a config
        # that asks for another head size would otherwise build a different model without a word
        if d.get("head_dim") is not None and int(d["head_dim"]) != cfg.head_dim:
            raise ValueError(f"head_dim {d['head_dim']} differs from hidden_size / num_attention_heads = {cfg.hidden_size} / "
                             f"{cfg.num_attention_heads} = {cfg.head_dim}; only head_dim == hidden_size / "
                             f"num_attention_heads is supported")
        return cfg

    @classmethod
    def from_pretrained(cls, name_or_path: str) -> "LlamaConfig":
        """Accepts a preset name (``150m``, ``llama-150m``, ``PrimeIntellect/llama-150m-fresh``), a config JSON, or a
        HF-style model directory containing ``config.json``."""
        p = Path(name_or_path)
        if p.is_dir():
            p = p / "config.json"
        if p.is_file():
            return cls.from_dict(json.loads(p.read_text()))
        key = os.path.basename(str(name_or_path)).lower().replace("llama-", "").replace("-fresh", "").replace("config_", "")
        key = key.replace(".json", "")
        preset = _PRESET_DIR / f"config_{key}.json"
        if preset.is_file():
            return cls.from_dict(json.loads(preset.read_text()))
        raise FileNotFoundError(f"no model config at {name_or_path!r} and no preset named {key!r} in {_PRESET_DIR}")

    def to_dict(self) -> dict:
        return asdict(self)

    def save_pretrained(self, directory: str) -> None:
        os.makedirs(directory, exist_ok=True)
        d = self.to_dict()
        d["torch_dtype"] = "float32"
        Path(directory, "config.json").write_text(json.dumps(d, indent=2))

    # -------------------------------------------------------------- derived numbers
    def num_parameters(self) -> int:
        h, i, L, V = self.hidden_size, self.intermediate_size, self.num_hidden_layers, self.vocab_size
        per_layer = 2 * h + h * self.q_dim + 2 * h * self.kv_dim + self.q_dim * h + 3 * h * i
        return 2 * V * h + L * per_layer + h

    def flops_per_token(self, seq_len: int) -> float:
        """fwd+bwd FLOPs per token: 6 x matmul parameters + causal attention (SURVEY.md §6)."""
        h, i, L, V = self.hidden_size, self.intermediate_size, self.num_hidden_layers, self.vocab_size
        mm_params = L * (h * self.q_dim + 2 * h * self.kv_dim + self.q_dim * h + 3 * h * i) + V * h
        attn = L * 2 * 2 * seq_len * self.q_dim * 0.5  # QK^T and PV, causal half, forward
        return 6.0 * mm_params + 3.0 * attn
