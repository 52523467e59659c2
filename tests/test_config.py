"""Config loading / interpolation / registry / component factory semantics (reference tier A: tests/config/*)."""
import os
from pathlib import Path

import pytest
from pydantic import BaseModel

from modalities_b200.config.factory import ComponentFactory
from modalities_b200.config.interpolation import InterpolationError, resolve_config
from modalities_b200.config.loader import load_app_config_dict
from modalities_b200.config.registry import Registry


def test_interpolation_types_and_strings():
    cfg = {"a": {"b": 3, "c": "${a.b}", "s": "x_${a.b}_y", "lst": [1, "${..b}"]}, "f": 1e-5, "p": "${a.lst.1}", "q": "${a.lst[0]}"}
    out = resolve_config(cfg)
    assert out["a"]["c"] == 3 and isinstance(out["a"]["c"], int)
    assert out["a"]["s"] == "x_3_y"
    assert out["a"]["lst"] == [1, 3]
    assert out["p"] == 3 and out["q"] == 1


def test_interpolation_resolvers_nested_and_container_results():
    cfg = {"n": 2, "r": "${mul:${n},3}", "w": "${ws:x}", "deep": "${w.k.1}", "esc": "\\${keep}"}
    out = resolve_config(cfg, {"mul": lambda a, b: int(a) * int(b), "ws": lambda _: {"k": [7, 8]}})
    assert out["r"] == 6 and out["w"] == {"k": [7, 8]} and out["deep"] == 8 and out["esc"] == "${keep}"


def test_interpolation_errors():
    with pytest.raises(InterpolationError, match="circular"):
        resolve_config({"a": "${b}", "b": "${a}"})
    with pytest.raises(InterpolationError, match="not found"):
        resolve_config({"a": "${missing.key}"})
    with pytest.raises(InterpolationError, match="unknown resolver"):
        resolve_config({"a": "${nope:1}"})


def test_loader_resolvers(tmp_path, monkeypatch):
    monkeypatch.setenv("RANK", "3")
    monkeypatch.setenv("SOME_VAR", "hello")
    p = tmp_path / "c.yaml"
    p.write_text("r: ${cuda_env:RANK}\nv: ${cuda_env:SOME_VAR}\ne: ${modalities_env:experiment_id}\n"
                 "f: ${modalities_env:config_folder_path}\nlr: 3e-4\nroot: ${modalities_env:experiments_root_path}/x\nn: ${node_env:num_cpus}\n")
    d = load_app_config_dict(p, experiments_root_path=Path("/exp"), experiment_id="eid")
    assert d["r"] == 3 and d["v"] == "hello" and d["e"] == "eid" and d["f"] == tmp_path
    assert d["lr"] == pytest.approx(3e-4) and d["root"] == "/exp/x" and d["n"] == os.cpu_count()


class _ACfg(BaseModel):
    val: int


class _A:
    def __init__(self, val):
        self.val = val


class _BCfg(BaseModel):
    model_config = {"arbitrary_types_allowed": True}
    a: _A
    items: list = []


class _B:
    def __init__(self, a, items):
        self.a, self.items = a, items


def _factory():
    reg = Registry()
    reg.add_entity("comp_a", "default", _A, _ACfg)
    reg.add_entity("comp_b", "default", _B, _BCfg)
    return ComponentFactory(reg, verbose=False)


class _Top(BaseModel):
    model_config = {"arbitrary_types_allowed": True}
    b1: _B
    b2: _B
    shared: _A
    opt: _A | None = None


def test_by_reference_identity_forward_and_backward_references():
    cfg = {
        "b1": {"component_key": "comp_b", "variant_key": "default", "config": {"a": {"instance_key": "shared", "pass_type": "BY_REFERENCE"}}},
        "shared": {"component_key": "comp_a", "variant_key": "default", "config": {"val": 5}},
        "b2": {"component_key": "comp_b", "variant_key": "default",
               "config": {"a": {"instance_key": "shared", "pass_type": "BY_REFERENCE"},
                          "items": [{"component_key": "comp_a", "variant_key": "default", "config": {"val": 1}}, 7]}},
    }
    out = _factory().build_components(cfg, _Top)
    assert out.b1.a is out.shared and out.b2.a is out.shared and out.opt is None
    assert isinstance(out.b2.items[0], _A) and out.b2.items[0].val == 1 and out.b2.items[1] == 7


def test_unknown_keys_missing_components_and_cycles():
    f = _factory()
    with pytest.raises(ValueError, match="Invalid keys"):
        f.instantiate("comp_a", "default", {"val": 1, "bogus": 2})
    with pytest.raises(ValueError, match="unknown variant_key"):
        f.instantiate("comp_a", "nope", {"val": 1})
    with pytest.raises(KeyError):
        f.build_components({"b1": {}}, _Top)

    class Cyc(BaseModel):
        model_config = {"arbitrary_types_allowed": True}
        x: _B

    cyc = {"x": {"component_key": "comp_b", "variant_key": "default", "config": {"a": {"instance_key": "x", "pass_type": "BY_REFERENCE"}}}}
    with pytest.raises(ValueError, match="cyclic"):
        f.build_components(cyc, Cyc)


def test_registry_matches_reference_catalogue():
    from modalities_b200.registry.components import COMPONENTS

    from conftest import reference_golden

    mine = {(e.component_key, e.variant_key) for e in COMPONENTS}
    ref = {tuple(e) for e in reference_golden("components")}  # the ComponentEntity entries of the reference's registry
    assert len(ref) >= 90 and ref <= mine, sorted(ref - mine)
    assert len(mine) >= 94


def test_custom_component_registration_through_main(tmp_path):
    """``Main.add_custom_component`` (library usage): a user-defined collator is built from YAML like a stock one."""
    import importlib.util
    from pathlib import Path

    import torch

    example = Path(__file__).resolve().parents[1] / "examples" / "library_usage"
    spec = importlib.util.spec_from_file_location("library_usage_example", example / "main.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    components = mod.build(example / "custom_collator.yaml", tmp_path)
    batch = components.collate_fn([{"input_ids": torch.arange(10)}, {"input_ids": torch.arange(10, 20)}])
    assert batch.samples["input_ids"].tolist() == [[0, 2, 4, 6], [10, 12, 14, 16]]
    assert batch.targets["target_ids"].tolist() == [[2, 4, 6, 8], [12, 14, 16, 18]]


@pytest.mark.timeout(600)
def test_custom_model_example_trains_through_main(tmp_path):
    """examples/custom_model: a user-defined model registered with ``Main.add_custom_component`` trains on 2 gloo ranks
    with the stock stack (sharded DP over its own block type, fused AdamW, checkpoints, evaluation).
    Reference: tutorials/einsum_transformer."""
    import json
    import os
    import subprocess
    import sys
    from pathlib import Path

    repo = Path(__file__).resolve().parents[1]
    env = dict(os.environ, MB200_DEVICE_TYPE="cpu", MB200_PARAM_DTYPE="FP_32", CUDA_VISIBLE_DEVICES="", MB200_BACKEND="gloo",
               MB200_DATA_PATH=str(repo / "data" / "lorem_ipsum_long.pbin"))  # fmt: skip
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29741", "examples/custom_model/train.py", str(tmp_path)]  # fmt: skip
    r = subprocess.run(cmd, cwd=repo, env=env, capture_output=True, text=True, timeout=550)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    (results,) = list(tmp_path.glob("*/evaluation_results.jsonl"))
    train = [json.loads(line) for line in results.read_text().splitlines()]
    losses = [rec["losses"]["train loss last"] for rec in train if rec["dataloader_tag"] == "train"]
    assert len(losses) == 6 and losses[-1] < losses[0]
    assert len(list(results.parent.glob("checkpoints/*/*.distcp"))) >= 2


def test_component_nodes_of_the_reference_yaml_files_fit_our_schemas():
    """Schema parity, checked mechanically: every ``{component_key, variant_key, config}`` node in the reference's shipped
    training / data-preparation / tutorial / test YAML files must name a registered component and use only config keys that
    our pydantic schema of that component knows (deprecated aliases included). The nodes are those recorded from the
    reference's files in tests/golden/reference/yaml_nodes.json.gz; its unit-test fixtures with made-up components (COMP_X …,
    dataset/test) are not real configs."""
    from conftest import reference_golden

    from modalities_b200.registry.components import COMPONENTS

    golden = reference_golden("yaml_nodes")
    entities = {(c.component_key, c.variant_key): c for c in COMPONENTS}
    assert golden["n_files"] > 50
    fixture_components = {"COMP_V", "COMP_W", "COMP_X", "COMP_Y", "COMP_Z"}
    # registered at run time by the reference's own tutorials / tests (add_custom_component) or by its inference entry point
    custom_or_runtime = {("inference_component", "text"), ("model", "einsum_transformer"), ("collate_fn", "custom_gpt_2_llm_collator"),
                         ("steppable_component", "steppable_norm"), ("results_subscriber", "save_all"), ("dataset", "test")}  # fmt: skip
    # variants that the reference's current registry does not know either (files left behind by renames)
    stale_variants = {("model", "fsdp_wrapped"), ("gradient_clipper", "fsdp"), ("model", "selective_activation_checkpointed")}
    # keys that the reference's own schemas reject as well (stale files in its repository)
    known_stale = {
        ("tokenizer", "pretrained_sp_tokenizer"): {"padding", "truncation"},
        ("number_conversion", "num_steps_from_num_samples"): {"dp_degree"},
        ("number_conversion", "num_steps_from_raw_dataset_index"): {"dp_degree"},
        ("model", "gpt2"): {"attention_norm", "ffn_norm", "lm_head_norm"},  # pre-``*_norm_config`` spelling in one tutorial file
    }
    problems, nodes = [], 0
    for component, variant, config_keys, count, where in golden["nodes"]:
        key = (component, variant)
        if key[0] not in fixture_components and key not in custom_or_runtime and key not in stale_variants:
            nodes += count
            entity = entities.get(key)
            if entity is None:
                problems.append((where, "unknown component", key))
            elif config_keys is not None:
                schema = entity.component_config_type
                allowed = set(schema.model_fields) | set(getattr(schema, "__deprecated_aliases__", {}))
                extra = set(config_keys) - allowed - known_stale.get(key, set())
                if extra:
                    problems.append((where, key, sorted(extra)))
    assert nodes > 900
    assert not problems, problems[:20]
