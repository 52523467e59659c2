"""Engine-level tests: schedulers, optimizer groups, number conversion, checkpoint strategies, MFU, sweeps, model
equivalences, pipeline stage pruning, end-to-end training + warm start through the CLI on CPU / gloo."""
import copy
import json
import math
import os
import subprocess
import sys
from pathlib import Path

import pytest
import torch
import yaml

from modalities_b200.checkpointing.checkpoint_saving_strategies import SaveEveryKStepsCheckpointingStrategy, SaveKMostRecentCheckpointsStrategy
from modalities_b200.checkpointing.fsdp.fsdp_checkpoint_saving import DCPCheckpointSaving
from modalities_b200.models.gpt2.gpt2_model import GPT2LLM, GPT2LLMConfig
from modalities_b200.models.model import SwiGLU
from modalities_b200.models.parallelism.pipeline_parallelism import prune_to_fqns
from modalities_b200.models.parallelism.stages_generator import GPT2LLMStagesGenerator
from modalities_b200.nn.model_initialization.composed_initialization import ComposedInitializationRoutines
from modalities_b200.nn.model_initialization.parameter_name_filters import SupportWeightInitModels, WeightInitTypes
from modalities_b200.optim.fused_adam import FusedAdamW
from modalities_b200.optim.lr_schedulers import DummyLRScheduler, LRSchedulerFactory
from modalities_b200.optim.optimizer_factory import get_optimizer_groups
from modalities_b200.training.training_progress import TrainingProgress
from modalities_b200.utils.benchmarking.benchmarking_utils import SweepSets, get_updated_sweep_status
from modalities_b200.utils.benchmarking.sweep_utils import SweepGenerator
from modalities_b200.utils.mfu import GPT2MFUCalculator
from modalities_b200.utils.number_conversion import NumberConversion
from modalities_b200.utils.seeding import calculate_hashed_seed

REPO = Path(__file__).resolve().parents[1]


def tiny_cfg(**over):
    d = over.pop("n_embd", 128)
    norm = {"norm_type": over.pop("norm", "layer_norm"), "config": {"normalized_shape": d, "eps": 1e-5}}
    base = dict(
        sample_key="input_ids", prediction_key="logits", poe_type="NOPE", sequence_length=32, vocab_size=128, n_layer=2,
        n_head_q=4, n_head_kv=2, n_embd=d, ffn_hidden=128, dropout=0.0, bias=False,
        attention_config={"qkv_transforms": [{"type_hint": "RotaryTransform", "config": {"n_embd": d, "n_head": 4, "seq_length_dim": -2, "base_freq": 10000}}]},
        attention_implementation="pytorch_flash", activation_type="swiglu", attention_norm_config=norm, ffn_norm_config=norm,
        lm_head_norm_config=norm, use_weight_tying=False,
    )  # fmt: skip
    base.update(over)
    return GPT2LLMConfig(**base)


def build(cfg):
    return GPT2LLM(**{k: getattr(cfg, k) for k in type(cfg).model_fields if k != "use_meta_device"})


def test_config_validators():
    with pytest.raises(ValueError):
        tiny_cfg(n_head_kv=3)
    with pytest.raises(ValueError):
        tiny_cfg(vocab_size=100)
    with pytest.raises(ValueError):
        build(tiny_cfg(poe_type="ABSOLUTE"))  # RoPE needs NOPE
    assert SwiGLU._get_hidden_dim(10240, 256) == 6912 and SwiGLU._get_hidden_dim(16384, 256) == 11008


def test_fqns_and_weight_tying():
    m = build(tiny_cfg())
    names = [n for n, _ in m.named_parameters()]
    for expected in ("transformer.wte.weight", "transformer.h.0.attention_norm.weight", "transformer.h.0.attn.q_attn.weight",
                     "transformer.h.1.attn.c_proj.weight", "transformer.h.0.mlp.W.weight", "transformer.h.0.mlp.W_2.weight",
                     "transformer.lm_head_norm.weight", "transformer.lm_head.weight"):  # fmt: skip
        assert expected in names
    assert m.transformer.h["0"].attn.k_attn.weight.shape == (64, 128)
    tied = build(tiny_cfg(use_weight_tying=True))
    assert tied.transformer.wte.weight is tied.transformer.lm_head.weight
    gelu = build(tiny_cfg(activation_type="gelu", poe_type="ABSOLUTE", attention_config={"qkv_transforms": []}))
    assert "transformer.wpe.weight" in dict(gelu.named_parameters()) and hasattr(gelu.transformer.h["0"].mlp, "c_fc")


@pytest.mark.parametrize("norm", ["layer_norm", "rms_norm", "pytorch_rms_norm"])
def test_attention_implementations_agree(norm):
    torch.manual_seed(0)
    x = torch.randint(0, 128, (2, 32))
    ref_model = build(tiny_cfg(attention_implementation="manual", norm=norm if norm != "rms_norm" else "layer_norm"))
    out_ref = ref_model(x)
    for impl in ("pytorch_flash", "dao_flash", "b200_flash"):
        m = build(tiny_cfg(attention_implementation=impl, norm=norm if norm != "rms_norm" else "layer_norm"))
        m.load_state_dict(ref_model.state_dict())
        assert torch.allclose(m(x), out_ref, atol=2e-5)
    out_dict = ref_model({"input_ids": x})
    assert torch.equal(out_dict["logits"], out_ref)


def test_pipeline_stage_pruning_equals_full_model():
    torch.manual_seed(1)
    m = build(tiny_cfg(n_layer=4))
    stages = GPT2LLMStagesGenerator(4).get_stages(num_layers_per_stage=2, pp_dims=3)
    assert stages[0][:3] == ["transformer.wte", "transformer.wpe", "transformer.drop"] and stages[-1][-1] == "transformer.lm_head"
    parts = [prune_to_fqns(copy.deepcopy(m), s) for s in stages]
    x = torch.randint(0, 128, (2, 32))
    h = x
    for p in parts:
        h = p(h)
    assert torch.allclose(h, m(x), atol=1e-6)
    assert sum(len(list(p.parameters())) for p in parts) == len(list(m.parameters()))
    with pytest.raises(ValueError):
        GPT2LLMStagesGenerator(4).get_stages(num_layers_per_stage=4, pp_dims=4)


def test_weight_init_statistics():
    m = build(tiny_cfg(n_embd=256, ffn_hidden=512))
    init = ComposedInitializationRoutines.get_composed_model_initializer(SupportWeightInitModels.GPT2, WeightInitTypes.SCALED, 0.0, 0.02, None, 2)
    init.initialize_in_place(m)
    p = dict(m.named_parameters())
    assert p["transformer.h.0.attn.q_attn.weight"].std().item() == pytest.approx(0.02, rel=0.1)
    assert p["transformer.h.0.attn.c_proj.weight"].std().item() == pytest.approx(0.02 / math.sqrt(4), rel=0.1)
    assert p["transformer.h.0.mlp.W_2.weight"].std().item() == pytest.approx(0.01, rel=0.1)
    auto = ComposedInitializationRoutines.get_composed_model_initializer(SupportWeightInitModels.GPT2, WeightInitTypes.PLAIN, 0.0, "auto", 256, None)
    auto.initialize_in_place(m)
    assert p["transformer.wte.weight"].std().item() == pytest.approx(math.sqrt(2 / (5 * 256)), rel=0.1)
    from modalities_b200.models.gpt2.llama3_like_initialization import Llama3Initializer

    m = build(tiny_cfg(n_embd=256, ffn_hidden=512, norm="pytorch_rms_norm"))  # Llama-3 style models carry no biases
    p = dict(m.named_parameters())
    Llama3Initializer(num_layers=2, n_embd=256, depth_init=True).initialize_in_place(m)
    assert p["transformer.h.1.attn.c_proj.weight"].std().item() == pytest.approx(0.02 / math.sqrt(4), rel=0.15)
    assert p["transformer.lm_head.weight"].abs().max().item() <= 3 / 16 + 1e-6


def test_optimizer_groups_and_fused_adam_matches_torch():
    torch.manual_seed(0)
    m = build(tiny_cfg())
    groups = get_optimizer_groups(m, 0.1, ["embedding", "layernorm"])
    assert groups[0]["weight_decay"] == 0.1 and groups[1]["weight_decay"] == 0.0
    no_decay = {id(p) for p in groups[1]["params"]}
    assert id(m.transformer.wte.weight) in no_decay and id(m.transformer.h["0"].attention_norm.weight) in no_decay
    assert id(m.transformer.lm_head.weight) not in no_decay
    ref = copy.deepcopy(m)
    opt = FusedAdamW(get_optimizer_groups(m, 0.1, ["embedding", "layernorm"]), lr=1e-2, betas=(0.9, 0.95))
    ropt = torch.optim.AdamW(get_optimizer_groups(ref, 0.1, ["embedding", "layernorm"]), lr=1e-2, betas=(0.9, 0.95))
    x = torch.randint(0, 128, (2, 32))
    for _ in range(3):
        for mod, o in ((m, opt), (ref, ropt)):
            mod(x).float().pow(2).mean().backward()
            o.step()
            o.zero_grad()
    for (n, a), (_, b) in zip(m.named_parameters(), ref.named_parameters()):
        assert torch.allclose(a, b, atol=1e-6), n


def test_lr_schedulers():
    p = torch.nn.Parameter(torch.zeros(1))
    opt = torch.optim.SGD([p], lr=1.0)
    sched = LRSchedulerFactory.get_linear_warmup_cosine_annealing_lr_scheduler(opt, warmup_steps=4, total_steps=12, initial_lr=0.2, final_lr=0.1, max_lr=1.0)
    lrs = []
    for _ in range(14):
        lrs.append(opt.param_groups[0]["lr"])
        opt.step()
        sched.step()
    assert lrs[0] == pytest.approx(0.2) and lrs[4] == pytest.approx(1.0) and lrs[12] == pytest.approx(0.1) and lrs[13] == pytest.approx(0.1)
    assert lrs[8] == pytest.approx(0.1 + 0.45 * (1 + math.cos(math.pi * 0.5)))
    with pytest.raises(ValueError):
        LRSchedulerFactory.get_linear_warmup_cosine_annealing_lr_scheduler(opt, 5, 5, 0.1, 0.1, 1.0)
    d = DummyLRScheduler(torch.optim.SGD([p], lr=0.3))
    d.step()
    assert d.get_last_lr() == [0.3]


def test_number_conversion_and_seeding():
    path = Path("/x/eid_2024-seen_steps_12-seen_tokens_6144-target_steps_40-target_tokens_20480")
    nc = NumberConversion
    assert nc.get_last_step_from_checkpoint_path(path) == 11 and nc.get_num_seen_steps_from_checkpoint_path(path) == 12
    assert nc.get_global_num_seen_tokens_from_checkpoint_path(path) == 6144
    assert nc.get_global_num_target_tokens_from_checkpoint_path(path) == 20480 and nc.get_num_target_steps_from_checkpoint_path(path) == 40
    assert nc.get_num_steps_from_num_tokens(dp_degree=2, local_micro_batch_size=4, global_num_tokens=8192, sequence_length=64, gradient_accumulation_steps=2) == 8
    assert nc.get_num_tokens_from_num_steps(8, 2, 4, 64, 2) == 8192
    assert nc.get_local_num_batches_from_num_tokens(num_ranks=2, global_num_tokens=8192, sequence_length=64, local_micro_batch_size=4) == 16
    with pytest.raises(ValueError):
        nc.get_num_seen_steps_from_checkpoint_path(Path("/no/match"))
    assert calculate_hashed_seed(["1", "2"]) == calculate_hashed_seed(["1", "2"]) != calculate_hashed_seed(["1", "3"])


def test_checkpoint_strategies_and_paths(tmp_path):
    tp = lambda s: TrainingProgress(num_seen_steps_current_run=s, num_seen_tokens_current_run=s * 10, num_target_steps=20, num_target_tokens=200)  # noqa: E731
    keep2 = SaveKMostRecentCheckpointsStrategy(k=2)
    i1, i2, i3 = (keep2.get_checkpoint_instruction(tp(s)) for s in (1, 2, 3))
    assert i1.save_current and not i1.checkpoints_to_delete and not i2.checkpoints_to_delete
    assert i3.save_current and i3.checkpoints_to_delete[0].num_seen_steps_total == 1
    assert not SaveKMostRecentCheckpointsStrategy(k=0).get_checkpoint_instruction(tp(1)).save_current
    assert not SaveKMostRecentCheckpointsStrategy(k=-1).get_checkpoint_instruction(tp(9)).checkpoints_to_delete
    every = SaveEveryKStepsCheckpointingStrategy(k=3)
    assert [every.get_checkpoint_instruction(tp(s)).save_current for s in (1, 3, 4, 6)] == [False, True, False, True]
    saver = DCPCheckpointSaving(tmp_path, "myexp", 0)
    folder = saver._folder_for(tp(4))
    assert folder.name == "eid_myexp-seen_steps_4-seen_tokens_40-target_steps_20-target_tokens_200"
    folder.mkdir(parents=True)
    (folder / "x.distcp").write_text("x")
    saver._delete_checkpoint(tp(4))
    assert not folder.exists()


def test_mfu_formula():
    m = build(tiny_cfg())
    calc = GPT2MFUCalculator(n_layer=2, sequence_length=32, n_embd=128, world_size=1, model_parts=m)
    n = sum(p.numel() for p in m.parameters())
    assert calc._flops_per_token == 6 * n + 12 * 2 * 32 * 128
    calc._theoretical_flops = 1e12
    assert calc.compute(10.0).item() == pytest.approx(10 * 32 * calc._flops_per_token / 1e12)


def test_sweep_generation_and_remaining_runs(tmp_path):
    sweep = tmp_path / "sweep.yaml"
    sweep.write_text(yaml.dump({"sweep": {"mbs": [1, 2], "seq": [128, 256, 512]}, "settings": {"x": "${sweep.mbs}"}}))
    written = SweepGenerator.generate_sweep_configs(sweep, tmp_path / "out", [2, 4])
    assert len(written) == 12 and all(p.parent.parent.name in ("2", "4") for p in written)
    assert yaml.safe_load(written[0].read_text())["sweep"] == {"mbs": 1, "seq": 128}
    status = get_updated_sweep_status(tmp_path / "out", expected_steps=3, world_size=2)
    assert len(status[SweepSets.UPDATED_CONFIGS.value]) == 6
    done = status[SweepSets.ALL_CONFIGS.value][0]
    (done.parent / "evaluation_results.jsonl").write_text("{}\n{}\n{}\n")
    oom = status[SweepSets.ALL_CONFIGS.value][1]
    (oom.parent / "error_logs_host_0.log").write_text(json.dumps({"error": {"type": "OutOfMemoryError"}}))
    status = get_updated_sweep_status(tmp_path / "out", expected_steps=3, world_size=2, skip_exception_types=["OutOfMemoryError"],
                                      create_new_folders_if_partially_done=False)  # fmt: skip
    assert len(status[SweepSets.REMAINING_CONFIGS.value]) == 4


# ----------------------------------------------------------------------------------------------------------------------
def _run_cli(args, nproc, port, env_extra, timeout=600):
    env = dict(os.environ, MB200_DEVICE_TYPE="cpu", MB200_PARAM_DTYPE="FP_32", CUDA_VISIBLE_DEVICES="", **env_extra)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), "-m", "modalities_b200", *args, "--backend", "gloo"]  # fmt: skip
    return subprocess.run(cmd, cwd=REPO, env=env, capture_output=True, text=True, timeout=timeout)


def _losses(exp_root: Path):
    files = sorted(exp_root.glob("*/evaluation_results.jsonl"))
    out = {}
    for f in files:
        for line in f.read_text().splitlines():
            rec = json.loads(line)
            if rec["dataloader_tag"] == "train":
                out[rec["num_train_steps_done"]] = rec["losses"]["train loss last"]
    return out


@pytest.mark.timeout(900)
def test_e2e_training_and_warmstart_across_world_sizes(tmp_path, lorem_pbin, free_port):
    """examples/warmstart/pre_train_and_warmstart.sh (the reference's tutorials/warmstart): 8 steps on 2 gloo ranks with DCP
    checkpoints after steps 4 and 8, the checkpoint layout check, then a warm start from the step-4 checkpoint on ONE rank
    (DCP reshards) with twice the micro batch — the script itself asserts that steps 5-8 continue the uninterrupted curve
    (reference: tests/end2end_tests/test_fsdp2_warmstart_pp_tp.py, rel 1e-2). On top: the experiment-folder and checkpoint
    artefacts of the first run; the step-4 checkpoint holds every entry the reference's checkpoint classes write for this
    model, with the same shape and dtype (tests/golden/reference/checkpoint_layout.json.gz), and loads into this
    framework's plain single-process AppState."""
    env = dict(os.environ, MB200_DEVICE_TYPE="cpu", MB200_PARAM_DTYPE="FP_32", CUDA_VISIBLE_DEVICES="", MB200_DATA_PATH=str(lorem_pbin),
               MASTER_PORT=str(free_port))  # fmt: skip
    r = subprocess.run(["bash", "examples/warmstart/pre_train_and_warmstart.sh", str(tmp_path / "ws"), "2", "1", "gloo"], cwd=REPO, env=env,
                       capture_output=True, text=True, timeout=800)  # fmt: skip
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "checkpoint layout OK" in r.stdout and "warm start continues the uninterrupted loss curve" in r.stdout
    full_root = tmp_path / "ws" / "pretrain"
    full = _losses(full_root)
    assert sorted(full) == list(range(1, 9)) and full[8] < full[1]
    exp = next(full_root.iterdir())
    assert (exp / "config_lorem_ipsum_fsdp2.yaml").exists() and (exp / "config_lorem_ipsum_fsdp2.yaml.resolved").exists()
    info = json.loads((exp / "checkpoints" / "last_checkpoint_info.json").read_text())
    ckpts = sorted(p.name for p in (exp / "checkpoints").iterdir() if p.is_dir())
    assert len(ckpts) == 2 and "seen_steps_4-seen_tokens_4096-target_steps_8-target_tokens_8192" in ckpts[0]
    assert sorted(p.name for p in (exp / "checkpoints" / ckpts[0]).iterdir()) == [".metadata", "__0_0.distcp", "__1_0.distcp"]
    assert info["checkpoint_folder_path"].endswith(ckpts[1])
    assert sorted(_losses(tmp_path / "ws" / "warmstart")) == [5, 6, 7, 8]
    # what the REFERENCE's AppState + torch AdamW + OneCycleLR write for this model — and request when they load it — is the
    # stored layout: the sharded checkpoint must hold each of those entries with the same shape and dtype. Then this
    # framework's AppState loads it on a plain single process (DCP reshards) and restores Adam step and scheduler position.
    from conftest import reference_golden

    def worker(*args):
        r = subprocess.run([sys.executable, "tests/workers/reference_checkpoint_load.py", *args], cwd=REPO, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        return json.loads(r.stdout.strip().splitlines()[-1])

    layout = worker("layout", str(exp / "checkpoints" / ckpts[0]))
    wanted = reference_golden("checkpoint_layout")
    assert {k: layout.get(k, "missing") for k in wanted} == wanted
    loaded = worker("ours", str(exp / "checkpoints" / ckpts[0]))
    assert loaded["adam_steps"] == [4.0] and loaded["n_state"] == 21 and loaded["sched_last_epoch"] == 4, loaded


def test_pure_components_give_the_reference_implementations_results():
    """tests/workers/reference_differential.py runs the same calls through this framework as through the reference's own code
    (its results: tests/golden/reference/differential.json.gz) and the results must be EQUAL: the warm-up / cosine LR
    schedule (40 steps), the resumable sampler's index sequences (shuffle / skip / drop_last / ranks), continuous packing
    over the shipped ``.pbin`` (lengths, first / last samples, checksum), the next-token collator and the loss-masking wrapper, nine number-conversion functions, the CLM
    cross entropy and both NCE variants, the composed and the Llama-3-like weight initialisation (per-parameter md5 of the
    bytes), seeded shuffles of tokenised / JSONL data and shuffled dataset chunks (file md5), combined and dummy datasets,
    the HF and SentencePiece tokenizer wrappers on the shipped tokenizer files, chunk ranges, and the sweep expansion of
    examples/scaling_up (sweep hash, per-world-size config hashes, md5 of every generated YAML), the checkpointing strategies'
    save / delete decisions, the DCP folder name, the ``evaluation_results.jsonl`` record and the MFU arithmetic."""
    from conftest import reference_golden, run_arms

    res = run_arms(lambda which: [sys.executable, "tests/workers/reference_differential.py", which], arms=("ours",), cwd=REPO)
    res["ref"] = reference_golden("differential")
    assert set(res["ref"]) == set(res["ours"]) and len(res["ref"]) >= 21
    for key, want in res["ref"].items():
        assert res["ours"][key] == want, key
    assert len(res["ref"]["weight_init"]) > 20 and len(res["ref"]["sampler"]) >= 13


def test_models_are_numerically_identical_to_the_reference_implementation():
    """Differential test against the reference's OWN model code: the reference built each model with weights seeded by
    parameter name and recorded its state-dict layout, buffers, outputs, loss and parameter gradients on CPU
    (tests/golden/reference/model_<variant>.json.gz); this framework's model must have the same layout (what a strict load
    checks: the FQNs and shapes are the checkpoint contract) and produce the same outputs, loss and gradients — GPT2LLM with
    SwiGLU / GQA / RoPE / LayerNorm and with GELU / MHA / absolute positions / RMSNorm / biases / tied embeddings, CoCa (ViT
    encoder + attention pooling + text and multimodal decoders, 153 tensors) and the stand-alone ViT."""
    from conftest import REFERENCE_GOLDEN

    variants = ["swiglu_gqa_rope_layernorm", "gelu_mha_abs_rmsnorm_bias_tied", "coca", "vit"]
    procs = [subprocess.Popen([sys.executable, "tests/workers/reference_model_forward.py", "ours", str(REFERENCE_GOLDEN / f"model_{v}.json.gz"), v],
                              cwd=REPO, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for v in variants]  # fmt: skip
    for v, p in zip(variants, procs):
        out, err = p.communicate(timeout=600)
        assert p.returncode == 0, (v, err[-3000:])
        rep = json.loads(out.strip().splitlines()[-1])
        assert rep["n_tensors"] > 20 and rep["logit_diff"] < 1e-5 and rep["loss_diff"] < 1e-6 and rep["grad_diff"] < 1e-5, (v, rep)


@pytest.mark.timeout(900)
def test_e2e_legacy_fsdp1_surface_trains_and_warmstarts(tmp_path, lorem_pbin, free_port):
    """Legacy FSDP1 config surface (model/fsdp1_wrapped, checkpoint_saving_execution/fsdp1 -> full-state .bin files,
    gradient_clipper/fsdp1) on 2 gloo ranks, then a warm start on ONE rank through model/fsdp1_checkpointed and
    optimizer/fsdp1_checkpointed: the loss curve continues. Reference: tests/end2end_tests/test_fsdp_warmstart.py and
    config_files/training/config_lorem_ipsum_long_fsdp1{,_warmstart}.yaml."""
    env = {"MB200_DATA_PATH": str(lorem_pbin), "MB200_MP_PRESET": "NO_MIXED_PRECISION"}
    full_root = tmp_path / "full"
    r = _run_cli(["run", "--config_file_path", "configs/config_lorem_ipsum_fsdp1.yaml", "--experiments_root_path", str(full_root)], 2, free_port, env)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    full = _losses(full_root)
    assert sorted(full) == list(range(1, 9)) and full[8] < full[1]
    exp = next(full_root.iterdir())
    ckpt_dir = exp / "checkpoints"  # <checkpoint_path>/eid_<experiment_id>-<entity>-....bin (reference layout)
    bins = sorted(p.name for p in ckpt_dir.glob("*.bin"))
    assert len(bins) == 4 and all(("-model-" in b) or ("-optimizer-" in b) for b in bins), bins
    model4 = next(p for p in ckpt_dir.glob("*-model-seen_steps_4-*.bin"))
    opt4 = next(p for p in ckpt_dir.glob("*-optimizer-seen_steps_4-*.bin"))
    assert "seen_tokens_4096-target_steps_8-target_tokens_8192" in model4.name
    last = json.loads((ckpt_dir / "last_checkpoint_info.json").read_text())
    assert set(last) == {"model_checkpoint_path", "optimizer_checkpoint_path"} and "seen_steps_8" in last["model_checkpoint_path"]

    info4 = tmp_path / "info4.json"
    info4.write_text(json.dumps({"model_checkpoint_path": str(model4), "optimizer_checkpoint_path": str(opt4)}))
    warm_root = tmp_path / "warm"
    r = _run_cli(["warmstart", "--config_file_path", "configs/config_lorem_ipsum_fsdp1_warmstart.yaml", "--experiments_root_path", str(warm_root),
                  "--last_checkpoint_info_file_path", str(info4)], 1, free_port + 1, env)  # fmt: skip
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    warm = _losses(warm_root)
    assert sorted(warm) == [5, 6, 7, 8]
    for step in (5, 6, 7, 8):
        assert warm[step] == pytest.approx(full[step], rel=1e-2), (step, warm, full)


@pytest.mark.timeout(600)
def test_e2e_coca_example_config_trains(tmp_path, free_port):
    """configs/config_coca_dummy_data.yaml: CoCa on the dummy image/text dataset through the CLI (1 gloo rank, 4 steps,
    evaluation + full-state checkpoint). Reference: config_files/training/config_example_coca.yaml."""
    env = {"MB200_MP_PRESET": "NO_MIXED_PRECISION"}
    root = tmp_path / "coca"
    r = _run_cli(["run", "--config_file_path", "configs/config_coca_dummy_data.yaml", "--experiments_root_path", str(root)], 1, free_port, env)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    losses = _losses(root)
    assert sorted(losses) == [1, 2, 3, 4] and all(0 < v < 10 for v in losses.values())
    exp = next(root.iterdir())
    assert len(list((exp / "checkpoints").rglob("*-model-seen_steps_4-*.bin"))) == 1


@pytest.mark.timeout(900)
def test_instruction_tuning_example_end_to_end(tmp_path, free_port):
    """examples/instruction_tuning: `data prepare_instruction_tuning_data` (chat template -> split -> index -> pack) and a
    loss-masked fine-tuning run on the packed training partition (1 gloo rank). Reference:
    tutorials/instruction_tuning + tests/instruction_tuning/test_e2e_instruction_tuning.py."""
    import subprocess
    import sys

    repo = Path(__file__).resolve().parents[1]
    src = tmp_path / "conversations.jsonl"
    rows = [{"id": i, "conversations": [{"role": "human_1", "content": f"What is {i} plus {i}?"},
                                        {"role": "gpt", "content": f"{i} plus {i} equals {2 * i}."}]}
            for i in range(60)]  # fmt: skip
    src.write_text("".join(json.dumps(r) + "\n" for r in rows))
    env = dict(os.environ, MB200_IT_SRC_JSONL=str(src), MB200_IT_DST_JSONL=str(tmp_path / "prepared" / "chat.jsonl"),
               RANK="0", LOCAL_RANK="0", WORLD_SIZE="1", CUDA_VISIBLE_DEVICES="")  # fmt: skip
    r = subprocess.run([sys.executable, "-m", "modalities_b200", "data", "prepare_instruction_tuning_data", "--config_file_path",
                        "examples/instruction_tuning/apply_chat_template_config.yaml"], cwd=repo, env=env, capture_output=True, text=True, timeout=600)  # fmt: skip
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    out_dirs = [d for d in (tmp_path / "prepared").iterdir() if d.is_dir()]
    assert len(out_dirs) == 1 and out_dirs[0].name.startswith("conversations_")
    train_pbin = next(out_dirs[0].glob("*train*.pbin"))
    assert next(out_dirs[0].glob("*val*.pbin")).exists() and next(out_dirs[0].glob("*train*.idx")).exists()
    first = json.loads(next(out_dirs[0].glob("*train*.jsonl")).read_text().splitlines()[0])
    assert first["chat"].startswith("You are a helpful assistant.") and "Assistant:^" in first["chat"] and "$" in first["chat"]

    root = tmp_path / "it"
    r = _run_cli(["run", "--config_file_path", "examples/instruction_tuning/train_instruct_model_fsdp2_config.yaml",
                  "--experiments_root_path", str(root)], 1, free_port, {"MB200_IT_TRAIN_PBIN": str(train_pbin)})  # fmt: skip
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    losses = _losses(root)
    assert sorted(losses) == [1, 2, 3, 4] and all(0 < v < 12 for v in losses.values())


@pytest.mark.timeout(900)
def test_scaling_up_example_sweep_is_resumable(tmp_path, lorem_pbin):
    """examples/scaling_up: `benchmark prepare_sweep_configs` on the shipped sweep config, then the resumable runner
    trains every remaining config (1 gloo rank) and a second invocation finds nothing left to do.
    Reference: tutorials/scaling_up + tests/utils/benchmarking."""
    sweep_dir = tmp_path / "sweep"
    env = dict(os.environ, MB200_DEVICE_TYPE="cpu", MB200_PARAM_DTYPE="FP_32", CUDA_VISIBLE_DEVICES="", MB200_DATA_PATH=str(lorem_pbin),
               MB200_BACKEND="gloo", RANK="0", LOCAL_RANK="0", WORLD_SIZE="1")  # fmt: skip
    r = subprocess.run([sys.executable, "-m", "modalities_b200", "benchmark", "prepare_sweep_configs", "--sweep_config_path",
                        "examples/scaling_up/gpt_throughput_sweep.yaml", "--output_dir", str(sweep_dir), "--world_sizes", "1,2"],
                       cwd=REPO, env=env, capture_output=True, text=True, timeout=300)  # fmt: skip
    assert r.returncode == 0, r.stderr[-2000:]
    (sweep_root,) = [d for d in sweep_dir.iterdir() if d.is_dir()]  # <output_dir>/<timestamp>_<hash of the sweep file>/<world size>/<hash>/
    configs = sorted(sweep_root.glob("1/*/*.yaml"))
    assert len(configs) == 4 and len(list(sweep_root.glob("2/*/*.yaml"))) == 4
    # keep the test short: only two of the four world-size-1 combinations stay
    for cfg in configs[2:]:
        for f in cfg.parent.iterdir():
            f.unlink()
        cfg.parent.rmdir()
    r = subprocess.run(["bash", "examples/scaling_up/run_sweep.sh", str(sweep_root), "1", "4"], cwd=REPO, env=env, capture_output=True, text=True, timeout=800)
    assert r.returncode == 0 and "2 configs to run" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
    for cfg in configs[:2]:
        lines = (cfg.parent / "evaluation_results.jsonl").read_text().splitlines()
        assert len(lines) == 4, r.stdout[-3000:] + r.stderr[-3000:]
    r = subprocess.run(["bash", "examples/scaling_up/run_sweep.sh", str(sweep_root), "1", "4"], cwd=REPO, env=env, capture_output=True, text=True, timeout=300)
    assert "0 configs to run" in r.stdout, r.stdout[-2000:]


@pytest.mark.timeout(900)
def test_getting_started_example_script(tmp_path):
    """examples/getting_started/run_getting_started_example.sh on CPU: index -> pack -> train (1 gloo rank) -> HF conversion
    with logit verification; the exported directory loads through transformers' trust_remote_code path and generates.
    Reference: tutorials/getting_started (tests/tests.py --include_examples)."""
    from transformers import AutoModelForCausalLM

    env = dict(os.environ, MB200_DEVICE_TYPE="cpu", MB200_PARAM_DTYPE="FP_32", MB200_MP_PRESET="NO_MIXED_PRECISION", CUDA_VISIBLE_DEVICES="",
               RANK="0", LOCAL_RANK="0", WORLD_SIZE="1")  # fmt: skip
    r = subprocess.run(["bash", "examples/getting_started/run_getting_started_example.sh", str(tmp_path), "1", "gloo"], cwd=REPO, env=env,
                       capture_output=True, text=True, timeout=850)  # fmt: skip
    assert r.returncode == 0, r.stdout[-2500:] + r.stderr[-3500:]
    assert (tmp_path / "data" / "train.idx").exists() and (tmp_path / "data" / "train.pbin").exists()
    losses = _losses(tmp_path / "experiments")
    assert sorted(losses) == [6] or sorted(losses) == list(range(1, 7))
    hf_dir = tmp_path / "hf_model"
    assert {"config.json", "modeling_gpt2.py", "configuration_gpt2.py"} <= {p.name for p in hf_dir.iterdir()}
    hf = AutoModelForCausalLM.from_pretrained(hf_dir, trust_remote_code=True).eval()
    ids = torch.randint(0, 50304, (1, 8))
    out = hf.generate(ids, max_new_tokens=4, do_sample=False, attention_mask=torch.ones_like(ids), pad_token_id=0)
    assert out.shape == (1, 12)
    # the other export path: `convert_pytorch_to_hf_checkpoint` wraps the framework model itself in an HF adapter
    from modalities_b200.models.huggingface_adapters.hf_adapter import HFModelAdapter

    ckpt = max((tmp_path / "experiments").glob("*/checkpoints/*-model-*.bin"), key=lambda p: p.stat().st_mtime)
    r = subprocess.run([sys.executable, "-m", "modalities_b200", "convert_pytorch_to_hf_checkpoint", "--config_file_path",
                        "examples/getting_started/example_conversion_config.yaml", "--output_hf_checkpoint_dir", str(tmp_path / "hf_adapter"),
                        "--prediction_key", "logits"], cwd=REPO, env=dict(env, MB200_CHECKPOINT_FILE=str(ckpt)), capture_output=True, text=True, timeout=300)  # fmt: skip
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    adapter = HFModelAdapter.from_pretrained(tmp_path / "hf_adapter", prediction_key="logits").eval()
    with torch.no_grad():
        a = adapter(input_ids=ids)  # the adapter returns the tensor under prediction_key (return_dict=True -> ModelOutput)
        assert torch.allclose(a.float(), hf(input_ids=ids).logits.float(), atol=2e-2, rtol=2e-2)  # both exports agree


@pytest.mark.timeout(600)
def test_failing_run_writes_structured_error_logs_per_rank(tmp_path, lorem_pbin, free_port):
    """A run that dies (here: a config whose dataset path does not exist) exits non-zero and leaves one JSON error file per
    rank in --error_log_folder: {environment: {rank, local_rank, world_size, hostname}, error: {error, type, stacktrace}};
    the sweep status reads `error.type` from these files (reference: __main__.py:726-749, benchmarking_utils.py:67-84)."""
    logs = tmp_path / "errors"
    r = _run_cli(["run", "--config_file_path", "configs/config_lorem_ipsum_fsdp2.yaml", "--experiments_root_path", str(tmp_path / "exp"),
                  "--error_log_folder", str(logs)], 2, free_port, {"MB200_DATA_PATH": str(tmp_path / "does_not_exist.pbin")})  # fmt: skip
    assert r.returncode != 0
    files = sorted(logs.glob("error_logs_*_*.log"))
    assert len(files) == 2 and {f.name.rsplit("_", 1)[1] for f in files} == {"0.log", "1.log"}
    rec = json.loads(files[0].read_text())
    assert set(rec) == {"environment", "error"}
    assert set(rec["environment"]) == {"rank", "local_rank", "world_size", "hostname"} and rec["environment"]["world_size"] == 2
    assert set(rec["error"]) == {"error", "type", "stacktrace"} and isinstance(rec["error"]["stacktrace"], list)
    assert rec["error"]["type"] and "does_not_exist" in (rec["error"]["error"] + "".join(rec["error"]["stacktrace"]))


@pytest.mark.timeout(1200)
@pytest.mark.parametrize("name, nproc", [("config_lorem_ipsum_long_fsdp2.yaml", 2), ("config_lorem_ipsum_long_fsdp2_pp_tp.yaml", 4)])
# ("config_lorem_ipsum_long_fsdp1.yaml", 2) passes as well; left out of the default run to keep the suite short
def test_reference_training_yaml_runs_unmodified_except_for_the_environment(name, nproc, tmp_path, free_port):
    """Drop-in check: the reference's OWN shipped training configs train here on gloo ranks — the FSDP2 object graph
    (device mesh, fsdp2_wrapped, model_initialized, gpt2 on the meta device, AdamW + OneCycle, DCP checkpoints, rich
    progress, MFU) and the full 3-D graph (PP 2 (GPipe) x TP 2 x FSDP: staged pipeline -> model part -> gpt2_tp ->
    fsdp2_wrapped -> pipeline builder -> scheduled pipeline -> selectors). Only environment-specific values are patched:
    device type / dtypes for CPU, the small corpus, output paths, the W&B subscriber (wandb is not installed), the worker
    count, the cadence — and `settings.paths.experiments_root_path`, which these files lack although the reference's
    current settings schema requires it too (SURVEY §5.6 'stale settings.paths')."""
    import re

    from conftest import REFERENCE_GOLDEN

    text = (REFERENCE_GOLDEN / name).read_text()
    fsdp1 = "fsdp1" in name  # the legacy surface has no device mesh and names its precision by preset
    patches = [
        ("    device_type: cuda", "    device_type: cpu", not fsdp1),
        ("      param_dtype: BF_16", "      param_dtype: FP_32", not fsdp1),
        ("      reduce_dtype: BF_16", "      reduce_dtype: FP_32", not fsdp1),
        ("    mixed_precision_settings: BF_16", "    mixed_precision_settings: NO_MIXED_PRECISION", fsdp1),
        ("    train_dataset_path: ./data/lorem_ipsum_long.pbin", "    train_dataset_path: ./data/lorem_ipsum.pbin", True),
        ("    checkpoint_saving_path: data/checkpoints", f"    checkpoint_saving_path: {tmp_path}/checkpoints", True),
        ("    num_workers: 2", "    num_workers: 0", True),
    ]
    for old, new, expected in patches:
        assert (old in text) or not expected, old
        text = text.replace(old, new)
    text = text.replace("    checkpointing_interval_in_steps: 32", "    checkpointing_interval_in_steps: 8")
    text = text.replace("    evaluation_interval_in_steps: 32", "    evaluation_interval_in_steps: 8")
    text = text.replace("  paths:\n", "  paths:\n    experiments_root_path: ${modalities_env:experiments_root_path}\n", 1)
    start = text.index("evaluation_subscriber:\n  component_key: results_subscriber\n  variant_key: wandb")
    nxt = re.search(r"\n\w+:\n", text[start + 10 :])
    end = start + 10 + nxt.start() + 1 if nxt else len(text)
    text = (text[:start] + "evaluation_subscriber:\n  component_key: results_subscriber\n  variant_key: to_disc\n  config:\n"
            f"    output_file_path: {tmp_path}/exp_results.jsonl\n\n" + text[end:])  # fmt: skip
    cfg = tmp_path / name
    cfg.write_text(text)
    r = _run_cli(["run", "--config_file_path", str(cfg), "--experiments_root_path", str(tmp_path / "exp")], nproc, free_port, {}, timeout=1000)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    records = [json.loads(line) for line in (tmp_path / "exp_results.jsonl").read_text().splitlines()]
    train = [rec["losses"]["train loss last"] for rec in records if rec["dataloader_tag"] == "train"]
    assert len(train) >= 3 and train[-1] < train[0] - 0.5, train
    if name == "config_lorem_ipsum_long_fsdp2.yaml":
        assert len(train) == 15  # 7 989 tokens / (256 x 2 ranks)
        assert len(list((tmp_path / "checkpoints").rglob("*.distcp"))) == 2  # the step-8 DCP checkpoint, one file per rank


def test_hf_export_matches_framework_model(tmp_path):
    """Framework GPT → stand-alone HF model: identical logits, KV-cache generation, reload through trust_remote_code.
    Reference analogue: /root/reference/tests/conversion/gpt2/test_conversion_model.py."""
    from transformers import AutoModelForCausalLM

    from modalities_b200.conversion.gpt2.conversion_code import transfer_model_code
    from modalities_b200.conversion.gpt2.conversion_model import _copy_weights_model, convert_model_config
    from modalities_b200.conversion.gpt2.modeling_gpt2 import GPT2ForCausalLM

    torch.manual_seed(0)
    cfg = tiny_cfg()
    model = build(cfg).float().eval()
    with torch.no_grad():
        for p in model.parameters():
            torch.nn.init.normal_(p, 0.0, 0.05)
    norm = {"norm_type": "layer_norm", "config": {"normalized_shape": 128, "eps": 1e-5}}
    config_dict = {"model_raw": {"config": dict(
        poe_type="NOPE", activation_type="swiglu", attention_implementation="pytorch_flash", attention_norm_config=norm,
        ffn_norm_config=norm, lm_head_norm_config=norm, vocab_size=128, n_embd=128, n_layer=2, n_head_kv=2, n_head_q=4,
        ffn_hidden=128, bias=False, sequence_length=32,
        attention_config={"qkv_transforms": [{"type_hint": "RotaryTransform", "config": {"base_freq": 10000}}]},
    )}}  # fmt: skip
    hf = GPT2ForCausalLM(convert_model_config(config_dict)).float().eval()
    _copy_weights_model(hf, model)
    ids = torch.randint(0, 128, (2, 32))
    with torch.no_grad():
        ref = model({"input_ids": ids})["logits"]
        assert torch.allclose(hf(input_ids=ids).logits, ref, atol=1e-5)
        out = hf.generate(ids[:, :8], max_new_tokens=6, do_sample=False, attention_mask=torch.ones(2, 8, dtype=torch.long), pad_token_id=0)
        greedy = hf(input_ids=out, use_cache=False).logits.argmax(-1)
    assert (greedy[:, 7:-1] == out[:, 8:]).all()  # cached decoding == full recomputation
    hf.config.auto_map = {"AutoConfig": "configuration_gpt2.GPT2Config", "AutoModelForCausalLM": "modeling_gpt2.GPT2ForCausalLM"}
    hf.save_pretrained(tmp_path)
    transfer_model_code(str(tmp_path))
    assert "modalities_b200" not in (tmp_path / "modeling_gpt2.py").read_text().split('"""', 2)[2]
    reloaded = AutoModelForCausalLM.from_pretrained(tmp_path, trust_remote_code=True).eval()
    with torch.no_grad():
        assert torch.allclose(reloaded(input_ids=ids).logits, ref, atol=1e-5)
    # cast to bf16 (inference loading with ``precision: BF16``): the rotary tables must not depend on the rounded
    # ``inv_freq`` buffer, and the export stays BIT-identical to the framework model (the reference's own criterion)
    model_bf16, hf_bf16 = model.to(torch.bfloat16), hf.to(torch.bfloat16)
    rot = next(m for m in model_bf16.modules() if type(m).__name__ == "RotaryTransform")
    cos, _ = rot._tables(32, torch.device("cpu"), torch.bfloat16)
    ang = torch.outer(torch.arange(32.0), 1.0 / (10000 ** (torch.arange(0, 32, 2).float() / 32)))
    assert torch.equal(cos[0, 0, :, :16], ang.cos())
    with torch.no_grad():
        assert torch.equal(hf_bf16(input_ids=ids).logits, model_bf16({"input_ids": ids})["logits"])
    # config criteria
    bad = {"model_raw": {"config": dict(config_dict["model_raw"]["config"], activation_type="gelu")}}
    with pytest.raises(AssertionError):
        convert_model_config(bad)


def test_hf_task_heads_of_the_exported_model():
    """Sequence / token classification and QA heads of the stand-alone HF model (reference:
    conversion/gpt2/modeling_gpt2.py GPT2ForSequenceClassification / TokenClassification / QuestionAnswering)."""
    from modalities_b200.conversion.gpt2.configuration_gpt2 import GPT2Config
    from modalities_b200.conversion.gpt2.modeling_gpt2 import (
        GPT2ForCausalLM,
        GPT2ForQuestionAnswering,
        GPT2ForSequenceClassification,
        GPT2ForTokenClassification,
    )

    torch.manual_seed(0)
    cfg = GPT2Config(vocab_size=64, hidden_size=32, num_hidden_layers=2, num_attention_heads=4, num_key_value_heads=2,
                     intermediate_size=64, max_position_embeddings=32, pad_token_id=0, num_labels=3)  # fmt: skip
    ids = torch.randint(1, 64, (2, 10))
    ids[1, 6:] = 0  # right padding
    mask = (ids != 0).long()
    seq = GPT2ForSequenceClassification(cfg).eval()
    out = seq(input_ids=ids, attention_mask=mask, labels=torch.tensor([0, 2]))
    assert out.logits.shape == (2, 3) and torch.isfinite(out.loss)
    with torch.no_grad():  # pooled at the last non-padding token: the padded tail does not matter
        assert torch.allclose(seq(input_ids=ids[1:, :6]).logits, out.logits[1:].detach(), atol=1e-5)
    tok = GPT2ForTokenClassification(cfg).eval()
    out = tok(input_ids=ids, attention_mask=mask, labels=torch.randint(0, 3, (2, 10)))
    assert out.logits.shape == (2, 10, 3) and torch.isfinite(out.loss)
    qa = GPT2ForQuestionAnswering(cfg).eval()
    out = qa(input_ids=ids, attention_mask=mask, start_positions=torch.tensor([1, 2]), end_positions=torch.tensor([3, 5]))
    assert out.start_logits.shape == (2, 10) and out.end_logits.shape == (2, 10) and torch.isfinite(out.loss)
    lm = GPT2ForCausalLM(cfg)
    assert lm.get_decoder() is lm.model
    lm.set_decoder(seq.model)
    assert lm.get_decoder() is seq.model


def test_hf_adapter_roundtrip(tmp_path):
    """HFModelAdapter wraps a config-built model; save_pretrained / from_pretrained reproduce the logits.
    Reference analogue: /root/reference/tests/checkpointing/test_checkpoint_conversion.py."""
    from modalities_b200.models.huggingface_adapters.hf_adapter import HFModelAdapter, HFModelAdapterConfig

    norm = {"norm_type": "layer_norm", "config": {"normalized_shape": 128, "eps": 1e-5}}
    config = {"model": {"component_key": "model", "variant_key": "gpt2", "config": dict(
        sample_key="input_ids", prediction_key="logits", poe_type="NOPE", sequence_length=32, vocab_size=128, n_layer=2,
        n_head_q=4, n_head_kv=2, n_embd=128, ffn_hidden=128, dropout=0.0, bias=False, use_meta_device=False,
        attention_config={"qkv_transforms": [{"type_hint": "RotaryTransform", "config": {"n_embd": 128, "n_head": 4, "seq_length_dim": -2, "base_freq": 10000}}]},
        attention_implementation="pytorch_flash", activation_type="swiglu", attention_norm_config=norm,
        ffn_norm_config=norm, lm_head_norm_config=norm, use_weight_tying=False, some_path=Path("/tmp/x"),
    )}}  # fmt: skip
    config["model"]["config"].pop("some_path")
    config["aux_path"] = Path("/tmp/not_json_serialisable")
    hf_config = HFModelAdapterConfig(config=config)
    assert hf_config.config["aux_path"] == "/tmp/not_json_serialisable"
    adapter = HFModelAdapter(hf_config, prediction_key="logits").eval()
    ids = torch.randint(0, 128, (1, 16))
    with torch.no_grad():
        a = adapter(input_ids=ids)
        assert adapter(input_ids=ids, return_dict=True).logits.shape == (1, 16, 128)
    adapter.save_pretrained(tmp_path, safe_serialization=False)
    again = HFModelAdapter.from_pretrained(tmp_path, prediction_key="logits").eval()
    with torch.no_grad():
        assert torch.allclose(again(input_ids=ids), a, atol=1e-6)
