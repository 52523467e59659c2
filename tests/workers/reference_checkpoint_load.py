"""Loads a sharded (DCP) checkpoint written by THIS framework's training run into a plain single-process GPT2LLM + AdamW +
LR scheduler through ``AppState`` + ``torch.distributed.checkpoint.load`` — with the REFERENCE's classes (``ref``) or with
this framework's (``ours``) — and prints what was restored. Usage:
    reference_checkpoint_load.py {ref|ours|ours_sharded} <checkpoint_dir> [save] [tiny]
(``save``: train three steps with this arm's classes and WRITE the checkpoint instead — for the opposite direction;
``tiny``: a 2-layer GELU model of ~2k parameters instead of the model of configs/config_lorem_ipsum_fsdp2.yaml.)
    reference_checkpoint_load.py layout <checkpoint_dir>
prints the checkpoint's entries {key: [shape, dtype] of a tensor, or null for a pickled value}."""

import hashlib
import json
import sys
from pathlib import Path

import torch
import torch.distributed.checkpoint as dcp

REPO = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(REPO))
which, ckpt = sys.argv[1], sys.argv[2]
if which == "layout":
    meta = dcp.FileSystemReader(ckpt).read_metadata().state_dict_metadata
    print(json.dumps({k: [list(m.size), str(m.properties.dtype)] if hasattr(m, "size") else None for k, m in sorted(meta.items())}))
    sys.exit(0)
tiny = "tiny" in sys.argv[3:]
sharded = which == "ours_sharded"  # this framework's sharded runtime (one rank) + FusedAdamW instead of plain torch objects
which = "ours" if sharded else which
if which == "ref":
    sys.path.insert(0, str(REPO / "baseline"))
    import ref_env

    ref_env.prepare()
else:
    import modalities_b200  # noqa: F401
    from modalities_b200 import compat

    compat.install_modalities_alias()
from modalities.checkpointing.stateful.app_state import AppState  # noqa: E402
from modalities.models.gpt2.gpt2_model import GPT2LLM, GPT2LLMConfig  # noqa: E402

# the model of configs/config_lorem_ipsum_fsdp2.yaml, or a tiny one whose checkpoint is small enough to store
d, V, n_head_q, n_head_kv, ffn, act = (8, 64, 2, 1, 16, "gelu") if tiny else (128, 50304, 8, 4, 128, "swiglu")
sizes = {"n_embd": d, "vocab_size": V, "ffn_hidden": ffn}
norm = {"norm_type": "pytorch_rms_norm", "config": {"normalized_shape": d, "eps": 1e-5}}
c = GPT2LLMConfig(sample_key="input_ids", prediction_key="logits", poe_type="NOPE", sequence_length=256, n_layer=2,
                  n_head_q=n_head_q, n_head_kv=n_head_kv, dropout=0.0, bias=False,
                  attention_config={"qkv_transforms": [{"type_hint": "RotaryTransform", "config": {"n_embd": d, "n_head": n_head_q, "seq_length_dim": -2, "base_freq": 10000}}]},
                  attention_implementation="pytorch_flash", activation_type=act, attention_norm_config=norm, ffn_norm_config=norm,
                  lm_head_norm_config=norm, use_weight_tying=False, **({k: 128 for k in sizes} if tiny else sizes))  # fmt: skip
c = c.model_copy(update=sizes)  # (the config validation refuses sizes that are not multiples of 128)
torch.manual_seed(123)  # different from the training run: everything that matters must come from the checkpoint
model = GPT2LLM(**{k: getattr(c, k) for k in type(c).model_fields if k != "use_meta_device"}).float()
if sharded:
    from modalities_b200.optim.fused_adam import FusedAdamW
    from modalities_b200.parallel.sharded import MixedPrecisionPolicy, shard_model_

    model = shard_model_(model, ["GPT2Block"], None, MixedPrecisionPolicy(torch.float32, torch.float32), device=torch.device("cpu"))
    opt = FusedAdamW(model.parameters(), lr=1.0, betas=(0.9, 0.95), eps=1e-8, weight_decay=0.1)
else:
    opt = torch.optim.AdamW(model.parameters(), lr=1.0, betas=(0.9, 0.95), eps=1e-8, weight_decay=0.1)
sched = torch.optim.lr_scheduler.OneCycleLR(opt, max_lr=6e-4, div_factor=10, final_div_factor=1, total_steps=8, pct_start=0.25, anneal_strategy="cos", cycle_momentum=False)
app = AppState(model=model, optimizer=opt, lr_scheduler=sched)
if "save" in sys.argv[3:]:
    # the other direction: train three plain AdamW steps with THIS arm's classes and write a checkpoint for the other arm
    for g in opt.param_groups:
        g["lr"] = 1e-3
    gen = torch.Generator().manual_seed(4)
    for _ in range(3):
        batch = torch.randint(0, V, (2, 33), generator=gen)
        out = model({"input_ids": batch[:, :-1]})["logits"]
        torch.nn.functional.cross_entropy(out.reshape(-1, V), batch[:, 1:].reshape(-1)).backward()
        opt.step()
        sched.step()
        opt.zero_grad()
    dcp.save({"app": app}, checkpoint_id=ckpt)
else:
    dcp.load({"app": app}, checkpoint_id=ckpt)
    if sharded:
        model._sdp.sync_compute_params()
ids = torch.randint(0, V, (2, 65), generator=torch.Generator().manual_seed(9))
with torch.no_grad():
    logits = model({"input_ids": ids[:, :-1]})["logits"]
loss = torch.nn.functional.cross_entropy(logits.reshape(-1, V), ids[:, 1:].reshape(-1)).item()
name = {id(p): n for n, p in model.named_parameters()}
st = opt.state_dict()["state"]
pid = {i: p for i, p in enumerate(p for g in opt.param_groups for p in g["params"])}
h = hashlib.md5()
for n, p in sorted(model.named_parameters()):
    h.update(p.detach().numpy().tobytes())
mom = hashlib.md5()
steps = set()
for i in sorted(st):
    mom.update(st[i]["exp_avg"].detach().float().contiguous().numpy().tobytes())
    mom.update(st[i]["exp_avg_sq"].detach().float().contiguous().numpy().tobytes())
    steps.add(float(st[i]["step"]))
print(json.dumps({"loss": round(loss, 6), "weights_md5": h.hexdigest(), "moments_md5": mom.hexdigest(), "adam_steps": sorted(steps),
                  "n_state": len(st), "lr": [round(g["lr"], 10) for g in opt.param_groups], "sched_last_epoch": sched.last_epoch}))  # fmt: skip
