"""Checkpointing pieces on one CPU process (reference analogues: tests/checkpointing/pytorch/test_torch_checkpoint_loading.py,
test_checkpoint_execution_functions.py, test_fsdp2_dcp_checkpoint_loading_and_saving.py, test_fsdp1_to_disc_checkpointing.py)."""

import json
from unittest.mock import MagicMock

import pytest
import torch
import torch.nn as nn

from modalities_b200.checkpointing.checkpoint_saving import CheckpointSaving
from modalities_b200.checkpointing.checkpoint_saving_execution import CheckpointSavingExecutionABC
from modalities_b200.checkpointing.checkpoint_saving_instruction import CheckpointingInstruction
from modalities_b200.checkpointing.checkpoint_saving_strategies import SaveKMostRecentCheckpointsStrategy
from modalities_b200.checkpointing.fsdp.fsdp_checkpoint_saving import DCPCheckpointSaving, FSDP1CheckpointSaving
from modalities_b200.checkpointing.stateful.app_state import AppState
from modalities_b200.checkpointing.stateful.app_state_factory import AppStateFactory
from modalities_b200.checkpointing.torch.torch_checkpoint_loading import TorchCheckpointLoading
from modalities_b200.training.training_progress import TrainingProgress


def _tp(step: int) -> TrainingProgress:
    return TrainingProgress(num_seen_steps_current_run=step, num_seen_tokens_current_run=step * 10, num_target_steps=20, num_target_tokens=200)


class _Net(nn.Module):
    def __init__(self):
        super().__init__()
        self.a = nn.Linear(4, 8)
        self.b = nn.Linear(8, 2, bias=False)

    def forward(self, x):
        return self.b(torch.relu(self.a(x)))


def _trained_state(seed: int = 0):
    torch.manual_seed(seed)
    model = _Net()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-2)
    sched = torch.optim.lr_scheduler.StepLR(opt, step_size=2, gamma=0.5)
    for _ in range(3):
        model(torch.randn(5, 4)).square().mean().backward()
        opt.step()
        sched.step()
        opt.zero_grad()
    return AppState(model, opt, sched)


def test_torch_checkpoint_loading_meta_model_compile_prefix_and_precision(tmp_path):
    src = _Net()
    # a checkpoint written from a torch.compile'd model carries `_orig_mod.` in its keys
    torch.save({k.replace("a.", "_orig_mod.a.") if k.startswith("a.") else k: v for k, v in src.state_dict().items()}, tmp_path / "m.bin")
    with torch.device("meta"):
        dst = _Net()
    loaded = TorchCheckpointLoading(device=torch.device("cpu"), precision=torch.bfloat16).load_model_checkpoint(dst, tmp_path / "m.bin")
    assert all(p.device.type == "cpu" and p.dtype == torch.bfloat16 for p in loaded.parameters())
    assert torch.allclose(loaded.a.weight.float(), src.a.weight, atol=1e-2)
    with pytest.raises(NotImplementedError):
        TorchCheckpointLoading(device=torch.device("cpu")).load_optimizer_checkpoint_(None, loaded, tmp_path / "m.bin")
    # the layout `torch.distributed.checkpoint.format_utils dcp_to_torch` gives a sharded checkpoint (app/{model,optimizer,...})
    torch.save({"app": {"model": src.state_dict(), "optimizer": {}, "lr_scheduler": {}}}, tmp_path / "converted.pth")
    again = TorchCheckpointLoading(device=torch.device("cpu")).load_model_checkpoint(_Net(), tmp_path / "converted.pth")
    assert torch.equal(again.a.weight, src.a.weight)


def test_strategy_times_execution_orchestration():
    """CheckpointSaving asks the strategy WHAT to do and hands the instruction to the execution (HOW)."""
    execution = MagicMock(spec=CheckpointSavingExecutionABC)
    saving = CheckpointSaving(SaveKMostRecentCheckpointsStrategy(k=1), execution)
    app_state = object()
    for step in (1, 2):
        saving.save_checkpoint(training_progress=_tp(step), evaluation_result=None, app_state=app_state)
    first, second = (c.kwargs["checkpointing_instruction"] for c in execution.run_checkpoint_instruction.call_args_list)
    assert isinstance(first, CheckpointingInstruction) and first.save_current and first.checkpoints_to_delete == []
    assert second.save_current and [t.num_seen_steps_total for t in second.checkpoints_to_delete] == [1]
    assert all(c.kwargs["app_state"] is app_state for c in execution.run_checkpoint_instruction.call_args_list)


def test_execution_runs_delete_then_save(tmp_path):
    calls = []

    class Exec(CheckpointSavingExecutionABC):
        def _save_checkpoint(self, app_state, training_progress):
            calls.append(("save", training_progress.num_seen_steps_total))

        def _delete_checkpoint(self, training_progress):
            calls.append(("delete", training_progress.num_seen_steps_total))

    Exec().run_checkpoint_instruction(CheckpointingInstruction(save_current=True, checkpoints_to_delete=[_tp(1), _tp(2)]), _tp(3), app_state=None)
    assert calls == [("save", 3), ("delete", 1), ("delete", 2)] or calls == [("delete", 1), ("delete", 2), ("save", 3)]
    calls.clear()
    Exec().run_checkpoint_instruction(CheckpointingInstruction(save_current=False, checkpoints_to_delete=[]), _tp(3), app_state=None)
    assert calls == []


def test_dcp_roundtrip_restores_model_optimizer_scheduler_and_is_single_use(tmp_path, dist_env_single):
    state = _trained_state(seed=0)
    saver = DCPCheckpointSaving(checkpoint_path=tmp_path, experiment_id="exp", global_rank=0)
    saver._save_checkpoint(state, _tp(3))
    folder = tmp_path / "eid_exp-seen_steps_3-seen_tokens_30-target_steps_20-target_tokens_200"  # directly below checkpoint_path
    assert {p.name for p in folder.iterdir()} == {".metadata", "__0_0.distcp"}
    info = json.loads((tmp_path / "last_checkpoint_info.json").read_text())
    assert info == {"checkpoint_folder_path": str(folder.absolute())}

    fresh = _trained_state(seed=1)  # different weights / moments / schedule position
    assert not torch.equal(fresh.model_parts[0].a.weight, state.model_parts[0].a.weight)
    fresh = AppState(fresh.model_parts[0], fresh.optimizer, torch.optim.lr_scheduler.StepLR(fresh.optimizer, step_size=2, gamma=0.5))
    loaded = AppStateFactory.get_dcp_checkpointed_app_state_(fresh, folder)
    assert loaded is fresh and loaded.is_loaded
    for (k, a), (_, b) in zip(state.model_parts[0].state_dict().items(), loaded.model_parts[0].state_dict().items()):
        assert torch.equal(a, b), k
    sa, sb = state.optimizer.state_dict(), loaded.optimizer.state_dict()
    for idx in sa["state"]:
        assert torch.equal(sa["state"][idx]["exp_avg"], sb["state"][idx]["exp_avg"])
        assert torch.equal(sa["state"][idx]["exp_avg_sq"], sb["state"][idx]["exp_avg_sq"])
    assert sb["param_groups"][0]["lr"] == pytest.approx(sa["param_groups"][0]["lr"])
    assert loaded.lr_scheduler.last_epoch == state.lr_scheduler.last_epoch == 3
    with pytest.raises(RuntimeError):  # an AppState may be loaded once
        AppStateFactory.get_dcp_checkpointed_app_state_(loaded, folder)


@pytest.mark.parametrize("optimizer_kind", ["torch_adamw", "fused_adamw"])
def test_dcp_warmstart_into_untrained_optimizer_restores_moments_and_step(tmp_path, dist_env_single, optimizer_kind):
    """A fresh optimizer has no state: the warm start must still restore exp_avg / exp_avg_sq / step (ADVICE r1)."""
    from modalities_b200.optim.fused_adam import FusedAdamW

    def make(train: bool):
        torch.manual_seed(0 if train else 1)
        model = _Net()
        opt = (torch.optim.AdamW if optimizer_kind == "torch_adamw" else FusedAdamW)(model.parameters(), lr=1e-2)
        sched = torch.optim.lr_scheduler.StepLR(opt, step_size=2, gamma=0.5)
        if train:
            for _ in range(3):
                model(torch.randn(5, 4)).square().mean().backward()
                opt.step()
                sched.step()
                opt.zero_grad()
        return AppState(model, opt, sched)

    state = make(train=True)
    DCPCheckpointSaving(checkpoint_path=tmp_path, experiment_id="exp", global_rank=0)._save_checkpoint(state, _tp(3))
    folder = tmp_path / "eid_exp-seen_steps_3-seen_tokens_30-target_steps_20-target_tokens_200"
    fresh = make(train=False)
    assert len(fresh.optimizer.state) == 0
    loaded = AppStateFactory.get_dcp_checkpointed_app_state_(fresh, folder)
    sa, sb = state.optimizer.state_dict(), loaded.optimizer.state_dict()
    assert len(sb["state"]) == len(sa["state"]) == 3
    for idx in sa["state"]:
        for key in ("exp_avg", "exp_avg_sq"):
            assert torch.equal(sa["state"][idx][key], sb["state"][idx][key]), (idx, key)
        assert float(sb["state"][idx]["step"]) == float(sa["state"][idx]["step"]) == 3.0
    # and the next update is identical to continuing the original run
    x = torch.randn(5, 4)
    for st in (state, loaded):
        st.model_parts[0](x).square().mean().backward()
        st.optimizer.step()
    for a, b in zip(state.model_parts[0].parameters(), loaded.model_parts[0].parameters()):
        assert torch.allclose(a, b, atol=1e-7)


def test_fsdp1_full_state_files_and_deletion(tmp_path, dist_env_single):
    state = _trained_state()
    saver = FSDP1CheckpointSaving(checkpoint_path=tmp_path, experiment_id="exp", global_rank=0)
    saver._save_checkpoint(state, _tp(4))
    names = sorted(p.name for p in tmp_path.glob("*.bin"))
    assert names == ["eid_exp-model-seen_steps_4-seen_tokens_40-target_steps_20-target_tokens_200.bin",
                     "eid_exp-optimizer-seen_steps_4-seen_tokens_40-target_steps_20-target_tokens_200.bin"]  # fmt: skip
    model_sd = torch.load(tmp_path / names[0], weights_only=True)
    assert set(model_sd) == set(state.model_parts[0].state_dict()) and torch.equal(model_sd["a.weight"], state.model_parts[0].a.weight)
    info = json.loads((tmp_path / "last_checkpoint_info.json").read_text())
    assert set(info) == {"model_checkpoint_path", "optimizer_checkpoint_path"}
    assert len(saver._get_paths_to_delete(_tp(4))) == 2  # files sit directly in checkpoint_path, like the reference
    saver._delete_checkpoint(_tp(4))
    assert not list(tmp_path.glob("*.bin"))


def test_checkpoint_written_through_the_reference_classes_loads_here(tmp_path):
    """The opposite direction of the cross-load in test_engine.py: the REFERENCE's AppState + torch AdamW + OneCycleLR
    trained a tiny GPT2LLM three steps and wrote a checkpoint with ``dcp.save`` (tests/golden/reference/tiny_checkpoint.*);
    this framework's AppState restores it — into plain torch objects and into the sharded runtime + FusedAdamW — with the
    same weights, Adam moments and step, learning rate and scheduler position the reference reports."""
    import json
    import subprocess
    import sys
    import tarfile
    from pathlib import Path

    from conftest import REFERENCE_GOLDEN, reference_golden

    repo = Path(__file__).resolve().parents[1]
    with tarfile.open(REFERENCE_GOLDEN / "tiny_checkpoint.tar.gz") as tar:
        tar.extractall(tmp_path, filter="data")
    ckpt = tmp_path / "tiny_checkpoint"

    def run(*args):
        r = subprocess.run([sys.executable, "tests/workers/reference_checkpoint_load.py", *args], cwd=repo, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        return json.loads(r.stdout.strip().splitlines()[-1])

    written = reference_golden("tiny_checkpoint")
    assert written["adam_steps"] == [3.0] and written["n_state"] == 19
    assert run("ours", str(ckpt), "tiny") == written
    assert run("ours_sharded", str(ckpt), "tiny") == written
