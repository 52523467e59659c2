"""Headline benchmark: training throughput (tokens/s, whole job) of GPT-2.7B, sharded data parallel (FSDP2 semantics),
bf16, sequence length 4096, synthetic packed tokens, random-init weights — BASELINE.json's metric and config.

    python bench.py --gpus N --steps K --warmup W                 # this framework
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # ... and write the last timed step's results
    python bench.py --impl reference --gpus N --steps K --warmup W   # the unmodified reference from baseline/_ref
    (N > 1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py ...)

Both arms build the same model through their own public API from the same kind of YAML (``configs/bench/*.yaml``): model
→ sharding wrapper → weight init → AdamW (weight-decay groups) → LR scheduler → gradient clipper → CLM loss, and run
the same training step (forward, loss, backward, clip, optimizer step, scheduler step, zero grad).

Timing protocol: W untimed warm-up steps, then EXACTLY K steps bracketed by barrier + ``torch.cuda.synchronize()``,
timed with CUDA events on the compute stream, max over ranks. Two passes:
  * ``value``  – device-timed steps on a device-resident batch (kernel-side number),
  * ``e2e``    – every step copies its inputs host→device from pinned memory and reads the loss back to the host.
Working set per step (5.6 GB bf16 weights + activations) is far larger than the 126 MB L2, so no explicit L2 flush is
needed between iterations (stated in ``config.l2``). SM clocks / throttle reasons are sampled with nvidia-smi during
the timed region.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))

BASELINE_TOK_S = 134_799.0  # best published 8-GPU 2.7B row of the reference (8x H100, scaling_mn5.md:15), BASELINE.md
# --config: the BASELINE.json configurations. gpt2_2p7b (#2 / #4 with --dtype fp8) is the default the driver runs;
# llama3_8b_tp2 (#3) = Llama-3-8B architecture, sharded DP x tensor parallel 2 (Colwise/Rowwise attention + MLP, sequence
# parallel norms); llama3_8b_instruct_ac (#5) = the same architecture, warm start from a DCP checkpoint written by this
# run's own initial state, full activation checkpointing per block, instruction-tuning style loss masking (the prompt half
# of every sample carries ignore_index targets), seq 8192 / micro batch 2 like the reference's instruction-tuning tutorial.
CONFIGS = {
    "gpt2_2p7b": dict(n_layer=32, n_embd=2560, n_head_q=32, n_head_kv=32, ffn_hidden=10240, vocab_size=50304,
                      sequence_length=4096, norm="layer_norm", rope_base=10000, tp=1, ac=False, mbs=4, masked=False, warmstart=False,
                      label="GPT-2.7B (L32 d2560 H32 hd80, SwiGLU ffn 10240->6912, LayerNorm, RoPE, vocab 50304, untied, no bias)",
                      published=BASELINE_TOK_S),
    "llama3_8b_tp2": dict(n_layer=32, n_embd=4096, n_head_q=32, n_head_kv=8, ffn_hidden=21504, vocab_size=128256,
                          sequence_length=4096, norm="pytorch_rms_norm", rope_base=500000, tp=2, ac=False, mbs=2, masked=False,
                          warmstart=False, published=None,
                          label="Llama-3-8B architecture (L32 d4096 32q/8kv hd128, SwiGLU 14336, RMSNorm, RoPE 5e5, vocab 128256, untied)"),
    "llama3_8b_instruct_ac": dict(n_layer=32, n_embd=4096, n_head_q=32, n_head_kv=8, ffn_hidden=21504, vocab_size=128256,
                                  sequence_length=8192, norm="pytorch_rms_norm", rope_base=500000, tp=1, ac=True, mbs=2, masked=True,
                                  warmstart=True, published=None,
                                  label="Llama-3-8B architecture, instruction-tuning step: DCP warm start, full activation "
                                        "checkpointing per block, prompt tokens masked (ignore_index)"),
}
MODEL = dict(CONFIGS["gpt2_2p7b"])

TP_STAGE = """tp_model:
  component_key: model
  variant_key: gpt2_tp
  config:
    model:
      instance_key: model_raw
      pass_type: BY_REFERENCE
    device_mesh:
      instance_key: device_mesh
      pass_type: BY_REFERENCE
"""
AC_STAGE = """ac_model:
  component_key: model
  variant_key: activation_checkpointed
  config:
    ac_variant: full_activation_checkpointing
    layers_fqn: transformer.h
    model:
      instance_key: @AC_INPUT@
      pass_type: BY_REFERENCE
    ac_fun_params: {}
"""


# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clocks and throttle reasons of this rank's GPU while the timed region runs."""

    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")  # fmt: skip

    def __init__(self, gpu_index: int, period_s: float = 0.2):
        self.gpu_index = gpu_index
        self.period_s = period_s
        self.samples: list[list[str]] = []
        self._stop = threading.Event()
        self._thread = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(
                    ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-i", str(self.gpu_index)],
                    capture_output=True, text=True, timeout=5,
                ).stdout.strip()  # fmt: skip
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(self.period_s)

    def __enter__(self):
        self._thread.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._thread.join(timeout=10)

    def summary(self) -> dict:
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(s) > 3 + i and s[3 + i].lower().startswith("active") for s in self.samples)]
        return {
            "sm_mhz": sm[len(sm) // 2] if sm else None,
            "sm_max_mhz": float(self.samples[0][1]) if self.samples[0][1].replace(".", "").isdigit() else None,
            "power_w_max": max((float(s[2]) for s in self.samples if s[2].replace(".", "").isdigit()), default=None),
            "reasons": reasons,
            "samples": len(self.samples),
        }


def write_config(impl: str, mbs: int, world: int, steps_total: int, out_dir: Path) -> Path:
    """Instantiate the YAML template of the chosen arm."""
    text = (REPO / "configs" / "bench" / "train_step.yaml").read_text()
    stages, last = "", "model_raw"
    if MODEL["tp"] > 1:
        stages, last = stages + TP_STAGE + "\n", "tp_model"
    if MODEL["ac"]:
        stages, last = stages + AC_STAGE.replace("@AC_INPUT@", last) + "\n", "ac_model"
    fields = {"MBS": mbs, "SEQ": MODEL["sequence_length"], "TP": MODEL["tp"], "DP_REPLICATE": int(os.environ.get("MB200_BENCH_DP_REPLICATE", 1)), "FSDP_INPUT": last, "VOCAB": MODEL["vocab_size"],
              "LAYERS": MODEL["n_layer"], "HQ": MODEL["n_head_q"], "HKV": MODEL["n_head_kv"], "FFN": MODEL["ffn_hidden"],
              "EMBD": MODEL["n_embd"], "ROPE": MODEL["rope_base"], "NORM": MODEL["norm"], "EXTRA_MODEL_STAGES": stages}  # fmt: skip
    for k, v in fields.items():
        text = text.replace(f"@{k}@", str(v))
    out_dir.mkdir(parents=True, exist_ok=True)
    path = out_dir / f"bench_{MODEL['name']}_{impl}_r{os.environ.get('RANK', '0')}.yaml"
    path.write_text(text)
    return path


# ----------------------------------------------------------------------------------------------------------------------
def run(args) -> dict:
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    for k, v in (("RANK", rank), ("LOCAL_RANK", local_rank), ("WORLD_SIZE", world)):
        os.environ.setdefault(k, str(v))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29533")
    if args.gpus != world:
        raise SystemExit(f"--gpus {args.gpus} does not match WORLD_SIZE {world}: launch with torch.distributed.run for N > 1")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    dist.init_process_group("nccl", device_id=device)

    MODEL.clear()
    MODEL.update(CONFIGS[args.config], name=args.config)
    if args.mbs is None:
        args.mbs = MODEL["mbs"]
    if world % MODEL["tp"]:
        raise SystemExit(f"--config {args.config} needs a multiple of {MODEL['tp']} GPUs (tensor parallel degree)")
    dp = world // MODEL["tp"]
    mbs, T, V = args.mbs, MODEL["sequence_length"], MODEL["vocab_size"]
    # configs and the warm-start checkpoint: outside the tree, one directory per user shared by the ranks of a run
    tmp = Path(os.environ.get("MB200_BENCH_TMP") or Path(tempfile.gettempdir()) / f"mb200_bench_{os.getuid()}")
    cfg_path = write_config(args.impl, mbs, world, args.steps * 2 + args.warmup * 2 + 4, tmp)

    if args.impl == "reference":
        from baseline.ref_env import prepare

        prepare()
        from modalities.batch import DatasetBatch  # noqa: I001
        from modalities.main import Main
        from modalities.trainer import Trainer
        from bench_models import make_bench_components_model

        model_type = make_bench_components_model("modalities")
    else:
        from modalities_b200.batch import DatasetBatch
        from modalities_b200.main import Main
        from modalities_b200.trainer import Trainer
        from bench_models import make_bench_components_model

        model_type = make_bench_components_model("modalities_b200")

    if args.dtype == "fp8" and args.impl != "reference":
        from modalities_b200.ops import functional as OF

        OF.set_fp8(True)
    torch.manual_seed(0)  # the same random-init weights in every run (--dump-outputs compares runs output for output)
    main = Main(cfg_path, experiments_root_path=tmp / "experiments", experiment_id=f"bench_{args.impl}")
    components = main.build_components(components_model_type=model_type)
    model = components.app_state.model_parts[0]
    optimizer, scheduler = components.app_state.optimizer, components.app_state.lr_scheduler
    d_, L_, hd_ = MODEL["n_embd"], MODEL["n_layer"], MODEL["n_embd"] // MODEL["n_head_q"]
    f_ = (2 * MODEL["ffn_hidden"] // 3 + 255) // 256 * 256  # SwiGLU hidden size rule of the model (multiple of 256)
    n_norm = (2 if MODEL["norm"] == "layer_norm" else 1) * d_
    n_params = (2 * V * d_ + L_ * (d_ * d_ * 2 + 2 * d_ * hd_ * MODEL["n_head_kv"] + 3 * d_ * f_ + 2 * n_norm) + n_norm)
    if MODEL["tp"] == 1:
        counted = sum(int(getattr(p, "full_numel", p.numel())) for p in model.parameters())
        assert counted == n_params, f"parameter count mismatch: model {counted} vs formula {n_params}"

    class _NullPublisher:
        def publish_message(self, *a, **k):
            pass

    trainer = Trainer(
        global_rank=rank, progress_publisher=_NullPublisher(), evaluation_result_publisher=_NullPublisher(),
        gradient_acc_steps=1, global_num_tokens_per_train_step=mbs * T * dp, device_mesh=components.device_mesh,
        num_seen_train_steps=0, global_num_seen_tokens=0, num_target_steps=10**9, num_target_tokens=10**15,
        gradient_clipper=components.gradient_clipper, profiler=None if args.impl != "reference" else _ref_no_profiler(),
    )  # fmt: skip
    model.train()
    if args.impl != "reference":
        if hasattr(components.gradient_clipper, "attach_optimizer"):
            components.gradient_clipper.attach_optimizer(optimizer)
        trainer.prepare_fused_loss([model], components.loss_fn)  # what Trainer.train() sets up for its loop

    gen = torch.Generator().manual_seed(1234 + rank // MODEL["tp"])  # the ranks of one tensor-parallel group share their data

    def host_batch():
        ids = torch.randint(0, V, (mbs, T + 1), generator=gen, dtype=torch.int64)
        x, y = ids[:, :-1].contiguous(), ids[:, 1:].contiguous()
        if MODEL["masked"]:
            y[:, : T // 2] = -100  # instruction tuning: the prompt half of every sample does not contribute to the loss
        return x.pin_memory(), y.pin_memory()

    warmstart = None
    if MODEL["warmstart"]:
        warmstart = _warmstart_roundtrip(args.impl, components, tmp / f"warmstart_{args.impl}", rank)
        optimizer, scheduler = components.app_state.optimizer, components.app_state.lr_scheduler

    pool = [host_batch() for _ in range(4)]
    h2d_bytes = sum(t.numel() * t.element_size() for t in pool[0])
    counter = _LaunchCounter(args.impl)
    last_step = {}  # what the latest training step returned: loss and gradient norm (device tensors)

    def step(i: int, from_host: bool, dev_batch=None):
        if from_host:
            x, y = pool[i % len(pool)]
            if args.impl == "reference":
                batch = DatasetBatch(samples={"input_ids": x}, targets={"target_ids": y})  # moved by the reference itself
            else:
                batch = DatasetBatch(samples={"input_ids": x}, targets={"target_ids": y})
                batch.to(device, non_blocking=True)
        else:
            batch = DatasetBatch(samples={"input_ids": dev_batch[0]}, targets={"target_ids": dev_batch[1]})
        _, _, loss, grad_norm = trainer._train_batch(batch=batch, model_parts=[model], optimizer=optimizer, scheduler=scheduler,
                                                     loss_fun=components.loss_fn, micro_batch_id=i)  # fmt: skip
        last_step.update(loss=loss, grad_norm=grad_norm)
        if from_host:
            return float(loss.detach().float().item())  # device→host read of the step result
        return loss

    def mem(tag: str) -> None:
        if os.environ.get("MB200_BENCH_MEMDEBUG") == "1" and rank == 0:
            print(f"[mem] {tag}: allocated {torch.cuda.memory_allocated(device) / 2**30:.2f} GB, peak "
                  f"{torch.cuda.max_memory_allocated(device) / 2**30:.2f} GB, reserved {torch.cuda.memory_reserved(device) / 2**30:.2f} GB",
                  file=sys.stderr, flush=True)  # fmt: skip

    mem("after build")

    def timed(from_host: bool):
        dev_batch = tuple(t.to(device) for t in pool[0]) if not from_host else None
        for i in range(args.warmup):
            step(i, from_host, dev_batch)
            mem(f"after warm-up step {i}")
        dist.barrier()
        torch.cuda.synchronize()
        counter.reset()
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        wall0 = time.perf_counter()
        with ClockSampler(local_rank) as clocks:
            start.record()
            last = None
            for i in range(args.steps):
                last = step(i, from_host, dev_batch)
            end.record()
            dist.barrier()
            torch.cuda.synchronize()
        wall = time.perf_counter() - wall0
        ms = start.elapsed_time(end)
        t = torch.tensor([ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        launches = counter.count()
        loss_val = last if isinstance(last, float) else float(last.detach().float().item())
        return t.item(), wall, clocks.summary(), launches, loss_val

    rt = None
    comm_verify = None
    if args.impl != "reference" and world > 1:
        from modalities_b200.comm.symmetric import verify_transport
        from modalities_b200.parallel.sharded import get_runtime

        rt = get_runtime(model)
        if rt is not None:
            # multi-GPU correctness visible in the result line: the NVLink collectives of this very model's buffers are
            # compared with NCCL on rank-dependent data before anything is timed
            comm_verify = verify_transport(rt)
            rt.comm_meter = True
    ms_dev, _, clocks, launches, loss_dev = timed(from_host=False)
    exposed_ms = busy_ms = None
    if rt is not None:
        # events accumulated over warm-up + timed steps of the device pass; report the per-step mean
        exposed_ms = rt.exposed_comm_ms() / (args.steps + args.warmup)
        # ... and how long the collectives ran on the communication stream (overlapped or not; includes peer waits)
        busy_ms = rt.comm_busy_ms() / (args.steps + args.warmup)
        rt.comm_meter = False
    ms_e2e, wall_e2e, clocks_e2e, _, loss_e2e = timed(from_host=True)
    if args.dump_outputs and rank == 0:
        dump_outputs(Path(args.dump_outputs), last_step, model)

    if args.profile:
        from torch.profiler import ProfilerActivity, profile

        dev_batch = tuple(t.to(device) for t in pool[0])
        torch.cuda.synchronize()
        dist.barrier()
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            for i in range(2):
                step(i, False, dev_batch)
            torch.cuda.synchronize()
        if rank == 0:
            Path(args.profile).parent.mkdir(parents=True, exist_ok=True)
            Path(args.profile).write_text(prof.key_averages().table(sort_by="cuda_time_total", row_limit=60, max_name_column_width=70))

    tokens = mbs * T * dp * args.steps
    value = tokens / (ms_dev / 1e3)
    e2e_value = tokens / (ms_e2e / 1e3)
    flops_per_token = 6 * n_params + 12 * MODEL["n_layer"] * T * MODEL["n_embd"]
    result = {
        "metric": "train_tokens_per_second",
        "value": value,
        "unit": "tokens/s",
        "n_gpus": world,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": ms_dev / args.steps,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": value / MODEL["published"] if MODEL["published"] and args.dtype == "bf16" else None,
        "dtype": "bf16" if args.dtype == "bf16" else "fp8 (MXFP8 e4m3 1x32 block-scaled GEMMs for QKV / attention-out / MLP; bf16 attention, LM head, norms; fp32 master + AdamW)",
        "data": "synthetic random tokens (uniform over the vocabulary), random-init weights",
        "impl": args.impl,
        "config": {
            "name": args.config,
            "model": MODEL["label"],
            "params": n_params,
            "global_batch": mbs * dp,
            "micro_batch_per_gpu": mbs,
            "seq_len": T,
            "parallelism": (f"dp{dp}" + (f" (hybrid: replicate {os.environ['MB200_BENCH_DP_REPLICATE']} x shard)"
                                         if os.environ.get("MB200_BENCH_DP_REPLICATE", "1") != "1" else "")
                            + (f" x tp{MODEL['tp']}" if MODEL["tp"] > 1 else "")
                            + " (sharded data parallel, bf16 params / bf16 reduce, fp32 master + AdamW"
                            + (", full activation checkpointing per block" if MODEL["ac"] else "") + ")"),
            "warmstart": warmstart,
            "l2": "no flush: per-step working set (>5 GB weights + activations) is far larger than the 126 MB L2",
            "optimizer": "AdamW(0.9,0.95) wd 0.1 (embedding/layernorm excluded), linear warm-up, grad clip 1.0",
            "baseline_ref": ("8xH100 2.7B seq4096 MBS4: 134799 tok/s (reference docs/scaling_experiments/scaling_mn5.md:15)"
                             if MODEL["published"] else "no published number for this configuration; compare with --impl reference"),
        },
        "clocks": {k: clocks.get(k) for k in ("sm_mhz", "sm_max_mhz", "reasons", "power_w_max", "samples")},
        "e2e": {
            "value": e2e_value,
            "unit": "tokens/s",
            "ms_per_step": ms_e2e / args.steps,
            "h2d_bytes_per_step": h2d_bytes,
            "d2h_bytes_per_step": 4,
            "wall_s": wall_e2e,
            "clocks": {k: clocks_e2e.get(k) for k in ("sm_mhz", "reasons")},
        },
        "gpu_launches": launches,
        "peak_mem_gb": round(torch.cuda.max_memory_allocated(device) / 2**30, 2),
        "exposed_comm_ms_per_step": exposed_ms,
        "comm_busy_ms_per_step": busy_ms,
        "comm_verify": comm_verify,
        "mfu_nominal_2.25PF": value * flops_per_token / (2.25e15 * world),
        "loss": {"device_pass": loss_dev, "e2e_pass": loss_e2e},
    }
    dist.barrier()
    dist.destroy_process_group()
    return result if rank == 0 else {}


def dump_outputs(out_dir: Path, last_step: dict, model, per_param: int = 4096) -> None:
    """The results of the last timed step as float32 .npy files: ``loss`` and ``grad_norm`` (what the training step returns)
    and ``params_sample``, the updated parameters of this rank at ``per_param`` seeded positions of every parameter in
    ``named_parameters`` order (a fixed sample: 2.7B parameters would not fit the 64 MB the dump may take)."""
    import numpy as np
    import torch

    out_dir.mkdir(parents=True, exist_ok=True)
    for name in ("loss", "grad_norm"):
        np.save(out_dir / f"{name}.npy", last_step[name].detach().float().reshape(1).cpu().numpy())
    gen = torch.Generator().manual_seed(0)
    samples = []
    with torch.no_grad():
        for _, p in model.named_parameters():
            flat = (p.to_local() if hasattr(p, "to_local") else p).detach().reshape(-1)
            idx = torch.randint(0, flat.numel(), (min(per_param, flat.numel()),), generator=gen)
            samples.append(flat[idx.to(flat.device)].float().cpu())
    np.save(out_dir / "params_sample.npy", torch.cat(samples).numpy())


def _warmstart_roundtrip(impl: str, components, folder: Path, rank: int):
    """Instruction-tuning runs start from pretrained weights: write this run's (sharded, DTensor) model state dict with
    torch.distributed.checkpoint and load it back into the live model through each package's own state-dict hooks
    (outside the timed region; weights only — the optimizer of a fine-tuning run starts fresh)."""
    import shutil

    import torch.distributed as dist
    import torch.distributed.checkpoint as dcp

    try:
        model = components.app_state.model_parts[0]
        if rank == 0:
            shutil.rmtree(folder, ignore_errors=True)
        dist.barrier()
        t0 = time.perf_counter()
        dcp.save({"model": model.state_dict()}, checkpoint_id=str(folder))
        dist.barrier()
        state = {"model": model.state_dict()}
        dcp.load(state, checkpoint_id=str(folder))
        model.load_state_dict(state["model"])
        dist.barrier()
        secs = time.perf_counter() - t0
        if rank == 0:
            shutil.rmtree(folder, ignore_errors=True)
        return {"ok": True, "what": "model weights, DCP sharded save + load", "save_plus_load_s": round(secs, 1)}
    except Exception as e:  # noqa: BLE001
        return {"ok": False, "error": f"{type(e).__name__}: {e}"[:200]}


def _ref_no_profiler():
    from modalities.utils.profilers.profilers import SteppableNoProfiler

    return SteppableNoProfiler()


class _LaunchCounter:
    """Number of this framework's own kernel launches (0 for the reference arm, which has none)."""

    def __init__(self, impl: str):
        self.impl = impl

    def reset(self):
        if self.impl != "reference":
            from modalities_b200.ops import native

            native.reset_launch_count()

    def count(self) -> int:
        if self.impl == "reference":
            return 0
        from modalities_b200.ops import native

        return native.launch_count()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--mbs", type=int, default=None, help="micro batch size per data-parallel rank (default: the config's)")
    ap.add_argument("--config", choices=sorted(CONFIGS), default="gpt2_2p7b", help="BASELINE.json configuration (see CONFIGS)")
    ap.add_argument("--dtype", choices=["bf16", "fp8"], default="bf16",
                    help="fp8: block-internal GEMMs (QKV, attention out, MLP) on the MXFP8 block-scaled tensor-core path "
                         "(BASELINE config 4); everything else as in the bf16 run. Own arm only.")
    ap.add_argument("--profile", type=str, default=None,
                    help="after the timed passes, run 2 more steps under torch.profiler on rank 0 and write the per-kernel table here")
    ap.add_argument("--dump-outputs", type=str, default=None, metavar="DIR",
                    help="after the timed passes, write the loss, gradient norm and a fixed sample of the updated parameters of the "
                         "last timed step to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        try:
            from baseline.ref_env import prepare

            prepare()
            import modalities  # noqa: F401
        except Exception as e:  # noqa: BLE001
            if int(os.environ.get("RANK", 0)) == 0:
                print(json.dumps({"impl": "reference", "unavailable": f"{type(e).__name__}: {e}"[:300]}))
            return
    result = run(args)
    if result:
        print(json.dumps(result))


if __name__ == "__main__":
    main()
