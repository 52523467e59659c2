"""Builds a tiny model (GPT2LLM variants, CoCa, ViT) with the REFERENCE implementation (``ref``: baseline/_ref) or with THIS
framework (``ours``), sets every parameter from a generator seeded by its name (the FQNs are the checkpoint contract),
runs forward + backward on CPU in fp32. ``ref`` writes the state-dict layout and a record of its outputs, loss and
gradients (exact values at fixed, seeded positions plus sum and norm of every tensor) to <file.json.gz>; ``ours`` reads
that record and reports the differences. Usage: reference_model_forward.py {ref|ours} <file.json.gz> <variant>"""

import gzip
import json
import math
import sys
import zlib
from pathlib import Path

import torch

REPO = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(REPO))
which, path, variant = sys.argv[1], sys.argv[2], sys.argv[3]
N_SAMPLES = 4  # recorded elements per gradient tensor (model outputs: 128)


def seeded_init(model):
    """Every floating parameter from a generator seeded by its state-dict name: matrices ~ N(0, 0.05), vectors 1 + N(0, 0.05)
    (weights: norm scales) or N(0, 0.05) (biases). Tied tensors take the value of their last name in sorted order."""
    with torch.no_grad():
        for name, t in sorted(model.state_dict(keep_vars=True).items()):
            if not isinstance(t, torch.nn.Parameter) or not t.is_floating_point():
                continue
            noise = 0.05 * torch.randn(t.shape, generator=torch.Generator().manual_seed(zlib.crc32(name.encode())))
            t.copy_(noise if t.dim() > 1 else noise + (1.0 if name.endswith("weight") else 0.0))


def positions(n, n_samples):
    return torch.randperm(n, generator=torch.Generator().manual_seed(0))[:n_samples].sort().values


def record(t, n_samples):
    flat = t.detach().double().reshape(-1)
    return {"shape": list(t.shape), "sum": float(f"{flat.sum().item():.12g}"), "sumsq": float(f"{flat.square().sum().item():.12g}"),
            "val": [float(f"{v:.9g}") for v in flat[positions(flat.numel(), n_samples)].tolist()]}  # fmt: skip


def deviation(t, rec):
    """A lower bound of max |t - recorded tensor|: at the recorded positions, of the means and of the norms."""
    assert list(t.shape) == rec["shape"], (list(t.shape), rec["shape"])
    flat = t.detach().double().reshape(-1)
    n = flat.numel()
    at = (flat[positions(n, len(rec["val"]))] - torch.tensor(rec["val"], dtype=torch.float64)).abs().max().item()
    return max(at, abs(flat.sum().item() - rec["sum"]) / n, abs(flat.square().sum().item() ** 0.5 - rec["sumsq"] ** 0.5) / math.sqrt(n))


def layout(model):
    sd = model.state_dict()
    buffers = {n for n, _ in model.named_buffers()}
    return {n: list(t.shape) for n, t in sd.items()}, {n: t for n, t in sd.items() if n in buffers}


def finish(model, outputs: dict, loss):
    grads = {n: p.grad for n, p in model.named_parameters() if p.grad is not None}
    state, buffers = layout(model)
    if which == "ref":
        Path(path).write_bytes(gzip.compress(json.dumps({
            "state": state, "buffers": {n: record(b, N_SAMPLES) for n, b in buffers.items()}, "loss": None if loss is None else loss.item(),
            "out": {k: record(v, 128) for k, v in outputs.items()}, "grads": {n: record(g, N_SAMPLES) for n, g in grads.items()},
        }).encode(), mtime=0))  # fmt: skip
        print(json.dumps({"saved": True, "n_params": sum(p.numel() for p in model.parameters())}))
        return
    assert set(grads) == set(blob["grads"]), sorted(set(grads) ^ set(blob["grads"]))
    print(json.dumps({
        "logit_diff": max(deviation(v, blob["out"][k]) for k, v in outputs.items()),
        "loss_diff": 0.0 if loss is None else abs(loss.item() - blob["loss"]),
        "grad_diff": max(deviation(grads[n], rec) for n, rec in blob["grads"].items()), "n_tensors": len(state),
    }))  # fmt: skip


def prepare(model):
    """ours: the state-dict layout (what a strict load of the reference's checkpoint checks) and the buffers in it must be
    the reference's."""
    seeded_init(model)
    if which == "ours":
        state, buffers = layout(model)
        assert state == blob["state"], sorted(k for k in set(state) | set(blob["state"]) if state.get(k) != blob["state"].get(k))[:10]
        for n, rec in blob["buffers"].items():
            assert deviation(buffers[n].float(), rec) < 1e-6, n
    return model


if which == "ref":
    sys.path.insert(0, str(REPO / "baseline"))
    import ref_env

    ref_env.prepare()
else:
    import modalities_b200  # noqa: F401
    from modalities_b200 import compat

    compat.install_modalities_alias()
    blob = json.loads(gzip.decompress(Path(path).read_bytes()))
if variant in ("coca", "vit"):
    torch.manual_seed(0)
    if variant == "coca":
        from modalities.models.coca.coca_model import CoCa, CoCaConfig

        c = CoCaConfig(
            prediction_key="logits", vision_embd_prediction_key="vision_embeddings", text_embd_prediction_key="text_embeddings",
            vision_cls_prediction_key="vision_cls", text_cls_prediction_key="text_cls",
            vision_encoder_config=dict(sample_key="images", prediction_key="vision_embeddings", img_size=32, n_classes=None, n_layer=2,
                                       attention_config={"attention_engine_type": "default_attention"}, n_head=4, n_embd=64,
                                       dropout=0.0, patch_size=8, patch_stride=8, n_img_channels=3, add_cls_token=False, bias=True),
            # (no ffn_hidden for the vision encoder: the reference's config has no such field — its blocks always use 3072)
            text_decoder_config=dict(sample_key="input_ids", prediction_key="logits", block_size=17, vocab_size=97, n_layer_text=2,
                                     n_layer_multimodal_text=2, n_head=4, n_embd=64, ffn_hidden=128, dropout=0.0, bias=True,
                                     attention_config={"attention_engine_type": "default_attention"}, activation="swiglu", epsilon=1e-5),
            n_pool_head=4, n_vision_queries=8, bias_attn_pool=False, epsilon_attn_pool=1e-5,
        )  # fmt: skip
        model = CoCa(**{k: getattr(c, k) for k in type(c).model_fields}).float()
        keys = ["logits", "vision_cls", "text_cls"]
    else:
        from modalities.models.vision_transformer.vision_transformer_model import VisionTransformer

        model = VisionTransformer(sample_key="images", prediction_key="logits", img_size=32, n_classes=10, n_layer=2, n_head=4, n_embd=64,
                                  ffn_hidden=128, dropout=0.0, patch_size=8, patch_stride=8, n_img_channels=3, add_cls_token=True,
                                  bias=True, attention_config=None).float()  # fmt: skip
        keys = ["logits"]
    g = torch.Generator().manual_seed(1)
    batch = {"images": torch.randn(3, 3, 32, 32, generator=g), "input_ids": torch.randint(0, 97, (3, 16), generator=g)}
    model = prepare(model)
    out = model(batch)
    sum(out[k].float().pow(2).mean() for k in keys).backward()
    finish(model, {k: out[k] for k in keys}, None)
    sys.exit(0)
d = 128
norm_type, act, n_kv, poe, bias, tie = {
    "swiglu_gqa_rope_layernorm": ("layer_norm", "swiglu", 2, "NOPE", False, False),
    "gelu_mha_abs_rmsnorm_bias_tied": ("pytorch_rms_norm", "gelu", 4, "ABSOLUTE", True, True),
}[variant]
norm = {"norm_type": norm_type, "config": {"normalized_shape": d, "eps": 1e-5}}
rope = [{"type_hint": "RotaryTransform", "config": {"n_embd": d, "n_head": 4, "seq_length_dim": -2, "base_freq": 10000}}]
cfg = dict(
    sample_key="input_ids", prediction_key="logits", poe_type=poe, sequence_length=64, vocab_size=256, n_layer=2, n_head_q=4,
    n_head_kv=n_kv, n_embd=d, ffn_hidden=128, dropout=0.0, bias=bias,
    attention_config={"qkv_transforms": rope if poe == "NOPE" else []}, attention_implementation="pytorch_flash",
    activation_type=act, attention_norm_config=norm, ffn_norm_config=norm, lm_head_norm_config=norm, use_weight_tying=tie,
)  # fmt: skip
from modalities.models.gpt2.gpt2_model import GPT2LLM, GPT2LLMConfig  # noqa: E402

c = GPT2LLMConfig(**cfg)
torch.manual_seed(0)
model = prepare(GPT2LLM(**{k: getattr(c, k) for k in type(c).model_fields if k != "use_meta_device"}).float())
ids = torch.randint(0, 256, (2, 65), generator=torch.Generator().manual_seed(1))
logits = model({"input_ids": ids[:, :-1]})["logits"]
loss = torch.nn.functional.cross_entropy(logits.reshape(-1, 256), ids[:, 1:].reshape(-1))
loss.backward()
finish(model, {"logits": logits}, loss)
