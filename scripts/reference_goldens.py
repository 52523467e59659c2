"""Writes tests/golden/reference/: what the reference implementation (Modalities) computes or ships for the differential
tests, so that the suite compares this framework with it without the reference at hand. Needs a checkout of the
reference and its package installed under baseline/_ref (see baseline/shims/README.md); rerun it when the reference
version this framework follows changes.

    python scripts/reference_goldens.py <reference checkout>
"""

import gzip
import json
import os
import re
import shutil
import subprocess
import sys
import tarfile
import tempfile
from pathlib import Path

import yaml

REPO = Path(__file__).resolve().parents[1]
OUT = REPO / "tests" / "golden" / "reference"
TRAINING_CONFIGS = ["config_lorem_ipsum_long_fsdp2.yaml", "config_lorem_ipsum_long_fsdp2_pp_tp.yaml"]
MODEL_VARIANTS = ["swiglu_gqa_rope_layernorm", "gelu_mha_abs_rmsnorm_bias_tied", "coca", "vit"]


def worker(*args) -> dict:
    env = dict(os.environ, PYTHONPATH=str(REPO))  # (the reference's third-party shims import this package's helpers)
    r = subprocess.run([sys.executable, *map(str, args)], cwd=REPO, env=env, capture_output=True, text=True, check=False)
    if r.returncode != 0:
        raise RuntimeError(f"{args}: {r.stderr[-3000:]}")
    return json.loads(r.stdout.strip().splitlines()[-1])


def write(name: str, obj) -> None:
    (OUT / f"{name}.json.gz").write_bytes(gzip.compress(json.dumps(obj, sort_keys=True).encode(), mtime=0))


def yaml_nodes(ref: Path) -> dict:
    """The {component_key, variant_key} nodes of the reference's YAML files, one entry per distinct
    [component, variant, config keys (null: no config mapping)] with its number of nodes and the first file that has it."""
    files = sorted(f for pattern in ("config_files/**/*.yaml", "tutorials/**/*.yaml", "tests/**/*.yaml") for f in ref.glob(pattern))
    nodes = {}

    def walk(node, where):
        if isinstance(node, dict):
            if "component_key" in node and "variant_key" in node:
                config = node.get("config")
                key = json.dumps([node["component_key"], node["variant_key"], sorted(config) if isinstance(config, dict) else None])
                nodes.setdefault(key, [0, where])[0] += 1
            for v in node.values():
                walk(v, where)
        elif isinstance(node, list):
            for v in node:
                walk(v, where)

    for f in files:
        try:
            content = yaml.safe_load(f.read_text())
        except yaml.YAMLError:
            continue
        walk(content, f.relative_to(ref).as_posix())
    return {"n_files": len(files), "nodes": sorted([*json.loads(k), *v] for k, v in nodes.items())}


def main(ref: Path) -> None:
    OUT.mkdir(parents=True, exist_ok=True)
    src = ref / "src" / "modalities"
    write("surface", worker("tests/workers/reference_surface_probe.py", "extract", src))
    components = re.findall(r'ComponentEntity\(\s*"([a-z_0-9]+)",\s*"([a-z_0-9]+)"', (src / "registry" / "components.py").read_text())
    write("components", sorted(map(list, set(components))))
    write("yaml_nodes", yaml_nodes(ref))
    for name in TRAINING_CONFIGS:
        shutil.copyfile(ref / "config_files" / "training" / name, OUT / name)

    write("cli_api", worker("tests/workers/cli_tree_dump.py", "ref"))
    write("pydantic_schemas", worker("tests/workers/pydantic_schema_dump.py", "ref"))
    write("differential", worker("tests/workers/reference_differential.py", "ref"))
    with tempfile.TemporaryDirectory() as tmp:
        tmp = Path(tmp)
        write("data_pipeline", worker("tests/workers/reference_data_pipeline.py", "ref", tmp / "data"))
        for v in MODEL_VARIANTS:
            worker("tests/workers/reference_model_forward.py", "ref", OUT / f"model_{v}.json.gz", v)
        # a checkpoint written through the reference's classes (tiny model), and what the reference reports after loading it
        write("tiny_checkpoint", worker("tests/workers/reference_checkpoint_load.py", "ref", tmp / "tiny", "save", "tiny"))
        with tarfile.open(OUT / "tiny_checkpoint.tar.gz", "w:gz") as tar:
            tar.add(tmp / "tiny", arcname="tiny_checkpoint")
        # the entries the reference's AppState writes — and requests on load — for the model of configs/config_lorem_ipsum_fsdp2.yaml
        worker("tests/workers/reference_checkpoint_load.py", "ref", tmp / "full", "save")
        write("checkpoint_layout", worker("tests/workers/reference_checkpoint_load.py", "layout", tmp / "full"))


if __name__ == "__main__":
    main(Path(sys.argv[1]).resolve())
