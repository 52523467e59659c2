"""Utilities and CPU data tools that had no direct coverage (reference analogues: tests/test_util.py, utils/test_*.py,
dataloader/test_dummy_dataset.py, test_filter_packed_data.py, end2end_tests/test_shuffle_*.py,
test_create_shuffled_*_chunk.py, test_tokenization.py, utils/test_communication_test.py)."""

import json
import pickle
import time
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.nn as nn

from modalities_b200.api import (
    FileExistencePolicy,
    create_filtered_tokenized_dataset,
    create_shuffled_dataset_chunk,
    create_shuffled_jsonl_dataset_chunk,
    enforce_file_existence_policy,
    merge_packed_data_files,
    shuffle_jsonl_data,
    shuffle_tokenized_data,
)
from modalities_b200.data.dataset import DummyDataset, DummySampleConfig, PackedMemMapDatasetBase
from modalities_b200.data.packed_format import update_data_length_in_pre_allocated_header, write_pbin
from modalities_b200.exceptions import TimeRecorderStateError
from modalities_b200.util import (
    TimeRecorder,
    format_metrics_to_gb,
    get_experiment_id_from_config,
    get_module_class_from_name,
    get_synced_experiment_id_of_run,
    get_total_number_of_trainable_parameters,
)
from modalities_b200.utils.file_ops import get_file_md5sum
from modalities_b200.utils.maybe_list_parameter import maybe_list_parameter
from modalities_b200.utils.seeding import calculate_hashed_seed

REPO = Path(__file__).resolve().parents[1]


def _pbin(path: Path, docs: list[list[int]], width: int = 2) -> Path:
    dtype = {1: "<u1", 2: "<u2", 4: "<u4"}[width]
    write_pbin(path, (np.asarray(d).astype(dtype).tobytes() for d in docs), width)
    return path


def _docs(path: Path) -> list[list[int]]:
    ds = PackedMemMapDatasetBase(raw_data_path=path, sample_key="t", load_index=True)
    return [ds[i]["t"].tolist() for i in range(len(ds))]


# ------------------------------------------------------------------------------------------------------------ util.py
def test_time_recorder_state_machine():
    t = TimeRecorder()
    with pytest.raises(TimeRecorderStateError):
        t.stop()
    with t:
        time.sleep(0.01)
        with pytest.raises(TimeRecorderStateError):
            t.start()
        with pytest.raises(TimeRecorderStateError):
            t.reset()
    first = t.delta_t
    assert first >= 0.01
    with t:
        time.sleep(0.01)
    assert t.delta_t > first  # accumulates
    t.reset()
    assert t.delta_t == 0.0


def test_experiment_id_is_timestamp_plus_config_hash(tmp_path, dist_env_single):
    cfg = tmp_path / "a.yaml"
    cfg.write_text("x: 1\n")
    eid = get_experiment_id_from_config(cfg, hash_length=8)
    date, digest = eid.rsplit("_", 1)
    assert len(digest) == 8 and date.count("-") == 4 and "__" in date
    other = tmp_path / "b.yaml"
    other.write_text("x: 2\n")
    assert get_experiment_id_from_config(other, hash_length=8).rsplit("_", 1)[1] != digest
    assert get_experiment_id_from_config(cfg, hash_length=None).rsplit("_", 1)[1].startswith(digest)
    synced = get_synced_experiment_id_of_run(cfg, hash_length=8)
    assert synced.rsplit("_", 1)[1] == digest


def test_parameter_counting_and_class_lookup():
    model = nn.Sequential(nn.Linear(4, 8), nn.ReLU(), nn.Linear(8, 2, bias=False))
    model[0].bias.requires_grad_(False)
    assert get_total_number_of_trainable_parameters(model) == 4 * 8 + 8 * 2
    assert get_total_number_of_trainable_parameters([model, nn.Linear(2, 2)]) == 4 * 8 + 8 * 2 + 6
    assert get_module_class_from_name(model, "ReLU") is nn.ReLU and get_module_class_from_name(model, "GELU") is None
    assert format_metrics_to_gb(3 * 1024**3) == pytest.approx(3.0)


def test_maybe_list_parameter_maps_over_model_parts():
    @maybe_list_parameter("model")
    def wrap(model, tag="x"):
        return f"{tag}:{model}"

    assert wrap("a") == "x:a" and wrap(["a", "b"], tag="y") == ["y:a", "y:b"] and wrap(model=["c"]) == ["x:c"]

    @maybe_list_parameter("model", apply_to_list_result=tuple)
    def ident(model):
        return model

    assert ident([1, 2]) == (1, 2)
    with pytest.raises(ValueError):
        maybe_list_parameter("nope")(lambda model: model)


def test_hashed_seed_and_md5(tmp_path):
    a = calculate_hashed_seed(["42", "3", "7"])
    # sum of the sha256 digests: deterministic, order independent (like the reference), sensitive to every input
    assert a == calculate_hashed_seed(["42", "7", "3"]) and a != calculate_hashed_seed(["42", "3", "8"]) and 0 <= a < 2**32
    assert calculate_hashed_seed(["1"], max_seed=10) < 10
    f = tmp_path / "f.bin"
    f.write_bytes(b"abc" * 1000)
    import hashlib

    assert get_file_md5sum(f, chunk_size=7) == hashlib.md5(b"abc" * 1000).hexdigest()


def test_file_existence_policy(tmp_path):
    f = tmp_path / "x"
    f.write_text("1")
    with pytest.raises(ValueError):
        enforce_file_existence_policy(f, FileExistencePolicy.ERROR)
    assert enforce_file_existence_policy(f, FileExistencePolicy.SKIP) is True and f.exists()
    assert enforce_file_existence_policy(f, FileExistencePolicy.OVERRIDE) is False and not f.exists()


def test_communication_test_on_a_single_gloo_rank(dist_env_single):
    from modalities_b200.utils.communication_test import run_communication_test

    run_communication_test()


# ------------------------------------------------------------------------------------------------------------ datasets
def test_dummy_dataset_shapes_and_types():
    ds = DummyDataset(num_samples=5, sample_definition=[DummySampleConfig(sample_key="img", sample_shape=(3, 4, 4), sample_type="float"),
                                                        DummySampleConfig(sample_key="ids", sample_shape=(7,), sample_type="int")])  # fmt: skip
    assert len(ds) == 5
    s = ds[3]
    assert s["img"].shape == (3, 4, 4) and np.issubdtype(s["img"].dtype, np.floating)
    assert s["ids"].shape == (7,) and np.issubdtype(s["ids"].dtype, np.integer)


def test_pbin_header_patch_and_empty_file(tmp_path):
    p = _pbin(tmp_path / "a.pbin", [[1, 2, 3], [4, 5]])
    raw = p.read_bytes()
    assert int.from_bytes(raw[:8], "little") == 10 and int.from_bytes(raw[8:12], "little") == 2
    with p.open("rb+") as f:  # corrupt the length field, then repair it from the index
        f.write((0).to_bytes(8, "little"))
    update_data_length_in_pre_allocated_header(p, [(0, 6), (6, 4)])
    assert _docs(p) == [[1, 2, 3], [4, 5]]
    empty = _pbin(tmp_path / "e.pbin", [])
    with pytest.warns(UserWarning):
        update_data_length_in_pre_allocated_header(empty, [])
    assert int.from_bytes(empty.read_bytes()[:8], "little") == 0


def test_filter_shuffle_merge_tools(tmp_path):
    docs = [[i] * (i % 4 + 1) for i in range(40)]
    src = _pbin(tmp_path / "src.pbin", docs)
    # filter: keep even document indices
    create_filtered_tokenized_dataset(src, lambda idx: idx % 2 == 0, tmp_path / "even.pbin", FileExistencePolicy.ERROR)
    assert _docs(tmp_path / "even.pbin") == docs[::2]
    # seeded document shuffle: a permutation, deterministic per seed, different across seeds
    shuffle_tokenized_data(src, tmp_path / "s1.pbin", batch_size=8, file_existence_policy=FileExistencePolicy.ERROR, seed=1)
    shuffle_tokenized_data(src, tmp_path / "s1b.pbin", batch_size=3, file_existence_policy=FileExistencePolicy.ERROR, seed=1)
    shuffle_tokenized_data(src, tmp_path / "s2.pbin", batch_size=8, file_existence_policy=FileExistencePolicy.ERROR, seed=2)
    s1, s1b, s2 = _docs(tmp_path / "s1.pbin"), _docs(tmp_path / "s1b.pbin"), _docs(tmp_path / "s2.pbin")
    assert sorted(s1) == sorted(docs) and s1 != docs and s1 == s1b and s1 != s2
    # chunks: every document of every input file lands in exactly one of the num_chunks outputs
    other = _pbin(tmp_path / "other.pbin", [[100 + i] for i in range(10)])
    chunks = []
    for cid in range(3):
        out = tmp_path / f"chunk{cid}.pbin"
        create_shuffled_dataset_chunk([src, other], out, chunk_id=cid, num_chunks=3, file_existence_policy=FileExistencePolicy.ERROR, global_seed=7)
        chunks.append(_docs(out))
    assert sorted(d for c in chunks for d in c) == sorted(docs + [[100 + i] for i in range(10)])
    assert all(len(c) > 0 for c in chunks)
    merge_packed_data_files([tmp_path / f"chunk{c}.pbin" for c in range(3)], tmp_path / "merged.pbin")
    assert _docs(tmp_path / "merged.pbin") == [d for c in chunks for d in c]
    with pytest.raises(ValueError):
        create_shuffled_dataset_chunk([src], tmp_path / "bad.pbin", chunk_id=3, num_chunks=3, file_existence_policy=FileExistencePolicy.ERROR)


def test_jsonl_shuffle_and_chunks(tmp_path):
    lines = [json.dumps({"id": i, "text": f"düsseldorf {i}"}, ensure_ascii=False) for i in range(30)]
    src = tmp_path / "a.jsonl"
    src.write_text("\n".join(lines) + "\n", encoding="utf-8")
    shuffle_jsonl_data(src, tmp_path / "shuf.jsonl", FileExistencePolicy.ERROR, seed=3)
    out = (tmp_path / "shuf.jsonl").read_text(encoding="utf-8").splitlines()
    assert sorted(out) == sorted(lines) and out != lines
    shuffle_jsonl_data(src, tmp_path / "shuf2.jsonl", FileExistencePolicy.ERROR, seed=3)
    assert (tmp_path / "shuf2.jsonl").read_text(encoding="utf-8").splitlines() == out
    got = []
    for cid in range(2):
        create_shuffled_jsonl_dataset_chunk([src], tmp_path / f"c{cid}.jsonl", chunk_id=cid, num_chunks=2,
                                            file_existence_policy=FileExistencePolicy.ERROR, global_seed=5)  # fmt: skip
        got += (tmp_path / f"c{cid}.jsonl").read_text(encoding="utf-8").splitlines()
    assert sorted(got) == sorted(lines)


# ------------------------------------------------------------------------------------------------------------ tokenizers
def test_hf_tokenizer_wrapper_padding_truncation_and_special_tokens():
    from modalities_b200.tokenization.tokenizer_wrapper import PreTrainedHFTokenizer

    tok = PreTrainedHFTokenizer(pretrained_model_name_or_path=str(REPO / "data" / "tokenizer" / "hf_gpt2"), truncation=False, padding=False)
    ids = tok.tokenize("Hello world, hello B200!")
    assert tok.decode(ids) == "Hello world, hello B200!" and tok.vocab_size >= 50257
    assert tok.get_token_id("<|endoftext|>") == 50256 and tok.is_special_token_id(50256)
    with pytest.warns(UserWarning):  # not in the vocabulary: mapped to the unk id with a warning (reference behaviour)
        assert tok.get_token_id("two tokens") == tok.tokenizer.unk_token_id
    padded = PreTrainedHFTokenizer(pretrained_model_name_or_path=str(REPO / "data" / "tokenizer" / "hf_gpt2"), truncation=True,
                                   padding="max_length", max_length=12, special_tokens={"pad_token": "<|endoftext|>"})  # fmt: skip
    short, long = padded.tokenize("Hi"), padded.tokenize("word " * 40)
    assert len(short) == 12 and short[-1] == 50256 and len(long) == 12
    with pytest.raises(NotImplementedError):  # growing the vocabulary is forbidden (the embedding matrix would not match)
        PreTrainedHFTokenizer(pretrained_model_name_or_path=str(REPO / "data" / "tokenizer" / "hf_gpt2"),
                              special_tokens={"pad_token": "<a brand new pad token>"})  # fmt: skip


def test_sentencepiece_tokenizer_wrapper():
    from modalities_b200.tokenization.tokenizer_wrapper import PreTrainedSPTokenizer

    model = next((REPO / "data" / "tokenizer" / "sentencepiece_dclm").glob("*.model"))
    tok = PreTrainedSPTokenizer(tokenizer_model_file=str(model))
    ids = tok.tokenize("Tensor memory holds the accumulators.")
    assert len(ids) > 3 and tok.decode(ids) == "Tensor memory holds the accumulators." and tok.vocab_size > 1000


# ------------------------------------------------------------------------------------------------------------ device mesh
class _MockSubMesh:
    def __init__(self, coord: int, size: int):
        self._coord, self._size = coord, size

    def get_coordinate(self):
        return [self._coord]

    def size(self) -> int:
        return self._size


class _MockMesh:
    """Stand-in for a DeviceMesh seen from ONE rank (reference analogue: MockDeviceMesh in
    tests/dataloader/samplers/test_resumable_distributed_multi_dim_sampler.py)."""

    def __init__(self, sizes: dict[str, int], coords: dict[str, int]):
        self.mesh_dim_names = tuple(sizes)
        self._sizes, self._coords = sizes, coords

    def size(self, dim: int) -> int:
        return self._sizes[self.mesh_dim_names[dim]]

    def __getitem__(self, name: str):
        return _MockSubMesh(self._coords[name], self._sizes[name])


def test_multi_dim_sampler_partitions_by_data_parallel_coordinate_only():
    from modalities_b200.data.sampler_factory import SamplerFactory
    from modalities_b200.parallel.device_mesh import ParallelismDegrees, get_parallel_degree, get_parallel_rank

    sizes = {"pp": 2, "dp_shard": 3, "tp": 2}
    dataset = list(range(31))
    per_rank = {}
    for pp in range(2):
        for dp in range(3):
            for tp in range(2):
                mesh = _MockMesh(sizes, {"pp": pp, "dp_shard": dp, "tp": tp})
                assert get_parallel_rank(mesh, ParallelismDegrees.DP_SHARD) == dp
                assert get_parallel_degree(mesh, [ParallelismDegrees.DP_SHARD, ParallelismDegrees.DP_REPLICATE]) == 3
                sampler = SamplerFactory.create_resumable_distributed_multi_dim_sampler(
                    dataset=dataset, device_mesh=mesh, data_parallel_key=ParallelismDegrees.DP_SHARD, shuffle=True, seed=4,
                    drop_last=True, skip_num_global_samples=6)  # fmt: skip
                per_rank[(pp, dp, tp)] = list(sampler)
    # ranks that differ only in their pp / tp coordinate read the SAME samples ...
    for dp in range(3):
        ref = per_rank[(0, dp, 0)]
        assert all(per_rank[(pp, dp, tp)] == ref for pp in range(2) for tp in range(2))
    # ... different dp coordinates read disjoint ones; together: the shuffled dataset minus the skipped global samples
    parts = [per_rank[(0, dp, 0)] for dp in range(3)]
    assert len({len(p) for p in parts}) == 1 and len(parts[0]) == (31 - 6) // 3
    flat = [i for p in parts for i in p]
    assert len(set(flat)) == len(flat) and set(flat) <= set(dataset)


def test_device_mesh_config_infers_and_validates_degrees():
    from modalities_b200.exceptions import ConfigError
    from modalities_b200.parallel.device_mesh import DeviceMeshConfig

    cfg = DeviceMeshConfig(device_type="cpu", data_parallel_replicate_degree=2, data_parallel_shard_degree=-1, tensor_parallel_degree=2,
                           pipeline_parallel_degree=2, world_size=32)  # fmt: skip
    assert cfg.data_parallel_shard_degree == 4
    cfg = DeviceMeshConfig(device_type="cpu", data_parallel_replicate_degree=-1, data_parallel_shard_degree=8, world_size=32)
    assert cfg.data_parallel_replicate_degree == 4
    with pytest.raises((ConfigError, ValueError)):
        DeviceMeshConfig(device_type="cpu", data_parallel_replicate_degree=-1, data_parallel_shard_degree=-1, world_size=8)
    with pytest.raises((ConfigError, ValueError)):
        DeviceMeshConfig(device_type="cpu", data_parallel_shard_degree=3, world_size=8)
    with pytest.raises((ConfigError, ValueError)):
        DeviceMeshConfig(device_type="cpu", data_parallel_shard_degree=8, enable_loss_parallel=True, world_size=8)


# ------------------------------------------------------------------------------------------------------------ data CLI
def test_data_cli_verbs_in_process(tmp_path):
    """`data` sub-commands through click (in process): shuffle_tokenized_data, shuffle_jsonl_data,
    create_shuffled_dataset_chunk, create_shuffled_jsonl_chunk, merge_packed_data, create_raw_index — same options as
    the reference CLI (src/modalities/__main__.py:230-588)."""
    from click.testing import CliRunner

    from modalities_b200.__main__ import main

    run = CliRunner().invoke
    docs = [[i, i + 1] for i in range(0, 40, 2)]
    a = _pbin(tmp_path / "a.pbin", docs[:10])
    b = _pbin(tmp_path / "b.pbin", docs[10:])
    r = run(main, ["data", "shuffle_tokenized_data", "--input_data_path", str(a), "--output_data_path", str(tmp_path / "a_shuf.pbin"),
                   "--batch_size", "4", "--seed", "3"])  # fmt: skip
    assert r.exit_code == 0, r.output
    assert sorted(_docs(tmp_path / "a_shuf.pbin")) == sorted(docs[:10])
    (tmp_path / "list.txt").write_text("a.pbin\nb.pbin\n")
    for cid in range(2):
        r = run(main, ["data", "create_shuffled_dataset_chunk", "--input_file_list_path", str(tmp_path / "list.txt"),
                       "--input_data_root_path", str(tmp_path), "--output_chunk_file_path", str(tmp_path / f"chunk{cid}.pbin"),
                       "--chunk_id", str(cid), "--num_chunks", "2", "--global_seed", "1"])  # fmt: skip
        assert r.exit_code == 0, r.output
    r = run(main, ["data", "merge_packed_data", str(tmp_path / "chunk0.pbin"), str(tmp_path / "chunk1.pbin"), str(tmp_path / "merged.pbin")])
    assert r.exit_code == 0, r.output
    assert sorted(_docs(tmp_path / "merged.pbin")) == sorted(docs)

    lines = [json.dumps({"text": f"line {i}"}) for i in range(12)]
    (tmp_path / "x.jsonl").write_text("\n".join(lines) + "\n")
    r = run(main, ["data", "shuffle_jsonl_data", "--input_data_path", str(tmp_path / "x.jsonl"), "--output_data_path",
                   str(tmp_path / "x_shuf.jsonl"), "--seed", "5"])  # fmt: skip
    assert r.exit_code == 0, r.output
    assert sorted((tmp_path / "x_shuf.jsonl").read_text().splitlines()) == sorted(lines)
    (tmp_path / "jl.txt").write_text("x.jsonl\n")
    r = run(main, ["data", "create_shuffled_jsonl_chunk", "--input_file_list_path", str(tmp_path / "jl.txt"), "--input_data_root_path",
                   str(tmp_path), "--output_chunk_file_path", str(tmp_path / "jc0.jsonl"), "--chunk_id", "0", "--num_chunks", "1",
                   "--global_seed", "2"])  # fmt: skip
    assert r.exit_code == 0, r.output
    assert sorted((tmp_path / "jc0.jsonl").read_text().splitlines()) == sorted(lines)
    r = run(main, ["data", "create_raw_index", str(tmp_path / "x.jsonl"), "--index_path", str(tmp_path / "x.idx")])
    assert r.exit_code == 0, r.output
    index = pickle.loads((tmp_path / "x.idx").read_bytes())
    raw = (tmp_path / "x.jsonl").read_bytes()
    assert len(index) == 12 and all(json.loads(raw[o : o + n]) == json.loads(lines[i]) for i, (o, n) in enumerate(index))
    # file existence policy: the default refuses to overwrite
    r = run(main, ["data", "shuffle_jsonl_data", "--input_data_path", str(tmp_path / "x.jsonl"), "--output_data_path",
                   str(tmp_path / "x_shuf.jsonl")])  # fmt: skip
    assert r.exit_code != 0


# ------------------------------------------------------------------------------------------------------------ running env
def test_cuda_env_owns_the_process_group_life_cycle(free_port, monkeypatch, caplog):
    """``CudaEnv`` (gloo here): initialises the group from torchrun's env variables, logs exceptions with the rank and the
    traceback, always destroys the group it created — and leaves a group it did not create alone."""
    import torch.distributed as dist

    from modalities_b200.running_env.cuda_env import CudaEnv

    for k, v in {"RANK": "0", "LOCAL_RANK": "0", "WORLD_SIZE": "1", "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": str(free_port)}.items():
        monkeypatch.setenv(k, v)
    assert not dist.is_initialized()
    with CudaEnv(process_group_backend="gloo"):
        assert dist.is_initialized() and dist.get_backend() == "gloo" and dist.get_world_size() == 1
    assert not dist.is_initialized()
    with pytest.raises(ZeroDivisionError):
        with CudaEnv(process_group_backend="gloo"):
            1 / 0
    assert not dist.is_initialized()  # cleaned up although the body raised
    # nested use: the inner context must not tear down the outer group
    with CudaEnv(process_group_backend="gloo"):
        with CudaEnv(process_group_backend="gloo"):
            pass
        assert dist.is_initialized()
    assert not dist.is_initialized()
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):
            with CudaEnv(process_group_backend="nccl"):
                pass


@pytest.mark.parametrize("config", ["gpt2_2p7b", "llama3_8b_tp2", "llama3_8b_instruct_ac"])
def test_bench_configs_resolve_to_the_named_model_graphs(config, tmp_path, monkeypatch):
    """bench.py --config: the generated YAML of every BASELINE configuration loads through the config loader (all
    interpolations resolve) and wires model_raw -> [gpt2_tp] -> [activation_checkpointed] -> fsdp2_wrapped."""
    import sys

    sys.path.insert(0, str(REPO))
    import bench
    from modalities_b200.config.loader import load_app_config_dict

    for k, v in {"RANK": "0", "LOCAL_RANK": "0", "WORLD_SIZE": "8"}.items():
        monkeypatch.setenv(k, v)
    bench.MODEL.clear()
    bench.MODEL.update(bench.CONFIGS[config], name=config)
    path = bench.write_config("b200", bench.CONFIGS[config]["mbs"], 8, 10, tmp_path)
    cfg = load_app_config_dict(path)
    spec = bench.CONFIGS[config]
    assert cfg["model_raw"]["config"]["n_embd"] == spec["n_embd"] and cfg["model_raw"]["config"]["vocab_size"] == spec["vocab_size"]
    assert cfg["device_mesh"]["config"]["tensor_parallel_degree"] == spec["tp"]
    chain = cfg["fsdp_model"]["config"]["model"]["instance_key"]
    assert chain == ("ac_model" if spec["ac"] else "tp_model" if spec["tp"] > 1 else "model_raw")
    if spec["ac"]:
        assert cfg["ac_model"]["config"]["ac_variant"] == "full_activation_checkpointing"
    if spec["tp"] > 1:
        assert cfg["tp_model"]["variant_key"] == "gpt2_tp"
    # both arms get byte-identical graphs (the reference arm reads the same template)
    assert path.read_text() == bench.write_config("reference", spec["mbs"], 8, 10, tmp_path).read_text()


def test_reference_module_paths_resolve_through_the_alias_finder():
    """Every module path of the reference imports below ``modalities_b200.`` and — after the opt-in alias — below
    ``modalities.`` (custom components written against the reference keep their imports), and every public top-level name
    of every reference module (430+ classes / functions / constants) exists on the module the path resolves to."""
    import subprocess
    import sys
    import textwrap
    from pathlib import Path

    from conftest import reference_golden

    surface = reference_golden("surface")  # the reference's modules (tests/workers/reference_surface_probe.py extract)
    names = sorted(surface)
    # ... and every PUBLIC top-level name (classes, functions, upper-case constants) each of those modules defines
    # (modeling_gpt2: the exported HF model code; here an independent implementation with own helpers)
    public = {mod: s["defs"] for mod, s in surface.items() if mod != "conversion.gpt2.modeling_gpt2"}
    assert len(names) > 100 and sum(map(len, public.values())) > 400
    code = textwrap.dedent(
        f"""
        import importlib, sys
        import modalities_b200
        from modalities_b200.compat import install_modalities_alias
        install_modalities_alias()
        bad = []
        for n in {names!r}:
            for prefix in ("modalities_b200", "modalities"):
                try:
                    importlib.import_module(prefix + "." + n)
                except Exception as e:  # noqa: BLE001
                    bad.append((prefix + "." + n, repr(e)[:100]))
        from modalities.dataloader.dataset import PackedMemMapDatasetContinuous as A
        from modalities_b200.data.dataset import PackedMemMapDatasetContinuous as B
        from modalities.optimizers.optimizer_factory import OptimizerFactory
        from modalities.config.component_factory import ComponentFactory
        from modalities.models.coca.text_decoder import TextDecoder
        from modalities.dataloader.collate_fns.collator_fn_wrapper_for_loss_masking import LossMaskingCollateFnWrapper
        from modalities.utils.profilers.steppable_components_if import SteppableComponentIF
        from modalities.config.config import TokenizerTypes
        assert A is B
        import modalities
        assert modalities is modalities_b200
        for mod, defs in {public!r}.items():
            m = importlib.import_module("modalities." + mod)
            bad += [(mod, d) for d in defs if not hasattr(m, d)]
        print("BAD", bad)
        """
    )
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=str(Path(__file__).resolve().parents[1]))
    assert out.returncode == 0, out.stderr[-2000:]
    assert "BAD []" in out.stdout, out.stdout[-2000:]


# ------------------------------------------------------------------ behaviours pinned by the reference's own test-suite
# (found by running it against this package, scripts/conformance/run_reference_tests.sh)
def test_lines_reader_without_index_lengths_keeps_the_line_terminator(tmp_path):
    from modalities_b200.api import create_raw_data_index
    from modalities_b200.data.large_file_lines_reader import LargeFileLinesReader

    src = tmp_path / "d.jsonl"
    src.write_text('{"text": "a"}\n{"text": "bb"}\n{"text": "ccc"}\n')
    create_raw_data_index(src, tmp_path / "d.idx")
    exact = LargeFileLinesReader(src, index_path=tmp_path / "d.idx", use_sample_length_from_index=True)
    verbatim = LargeFileLinesReader(src, index_path=tmp_path / "d.idx", use_sample_length_from_index=False)
    assert [x for x in exact] == ['{"text": "a"}', '{"text": "bb"}', '{"text": "ccc"}']
    assert [x for x in verbatim] == [x + "\n" for x in exact] and verbatim[-1] == '{"text": "ccc"}\n'
    assert "".join(verbatim) == src.read_text()  # writing the items back reproduces the file


def test_token_width_is_derived_from_the_vocabulary_size_and_empty_output_is_refused(tmp_path):
    from modalities_b200.data.filter_packed_data import filter_dataset
    from modalities_b200.preprocessing.tokenization.tokenized_file_writer import TokenizedFileWriter as W

    assert [W.get_required_num_of_bytes_to_repr(n) for n in (10, 256, 257, 50257, 65536, 65537, 2**32)] == [1, 1, 2, 2, 2, 4, 4]
    with pytest.raises(ValueError):
        W.get_required_num_of_bytes_to_repr(2**32 + 1)
    docs = [np.array([1, 2, 3]), np.array([7, 8, 65536])]
    with pytest.raises(ValueError):  # 65536 does not fit the two bytes of a 65536-entry vocabulary
        W.write_tokenized_dataset(docs, tmp_path / "x.pbin", token_size_in_bytes=W.get_required_num_of_bytes_to_repr(65536))
    with pytest.raises(ValueError, match="did not create any data"):
        W.write_tokenized_dataset([], tmp_path / "empty.pbin", token_size_in_bytes=2)
    src = _pbin(tmp_path / "src.pbin", [[1, 2], [3]])
    with pytest.warns(UserWarning):  # the filter tool, in contrast, writes a valid empty file
        filter_dataset(src, tmp_path / "none.pbin", lambda item: False, sample_key="t")
    assert _docs(tmp_path / "none.pbin") == []


def test_reference_names_for_user_code():
    from unittest.mock import MagicMock

    from torch.distributed.algorithms._checkpoint.checkpoint_wrapper import CheckpointWrapper

    import modalities_b200.__main__ as entry
    from modalities_b200.exceptions import ModelStateError
    from modalities_b200.main import Main
    from modalities_b200.models.model_factory import ModelFactory
    from modalities_b200.training.activation_checkpointing.activation_checkpointing import ActivationCheckpointing
    from modalities_b200.training.gradient_clipping.fsdp_gradient_clipper import FSDP1LoggingOnlyGradientClipper, GradientClippingMode
    from modalities_b200.utils.typing_utils import FSDP2, FSDPX

    assert entry.Main is Main and callable(entry.load_app_config_dict)
    assert not isinstance(nn.Linear(2, 2), FSDP2) and FSDPX is not None
    # half-materialised plain module
    mixed = nn.Sequential(nn.Linear(2, 2), nn.Linear(2, 2, device="meta"))
    with pytest.raises(ModelStateError):
        ModelFactory._is_model_on_meta_device(mixed)
    assert ModelFactory._is_model_on_meta_device(nn.Linear(2, 2, device="meta")) and not ModelFactory._is_model_on_meta_device(nn.Linear(2, 2))
    # a foreign FSDP1 object is clipped through its own API
    foreign = MagicMock()
    FSDP1LoggingOnlyGradientClipper(wrapped_model=foreign, norm_type=GradientClippingMode.P2_NORM).clip_gradients()
    foreign.clip_grad_norm_.assert_called_once_with(max_norm=torch.inf, norm_type=2)
    # checkpointed blocks are recognisable, keep their class name (block_names matching) and their attribute protocol
    block = nn.Sequential(nn.Linear(2, 2))
    ActivationCheckpointing._apply_full_ac(block)
    assert isinstance(block, CheckpointWrapper) and type(block).__name__ == "Sequential" and not hasattr(block, "nope")
    assert [n for n, _ in block.named_parameters()] == ["0.weight", "0.bias"]
    x = torch.randn(3, 2, requires_grad=True)
    block(x).sum().backward()
    assert x.grad is not None


def test_cli_command_tree_and_library_api_match_the_reference():
    """Every command of the reference's ``modalities`` CLI exists here with the same options (names, required, flags); the
    only additions are ``--backend`` on the distributed verbs. ``api.py``: same public functions / enums, same parameter
    names and required-ness. Introspected from this package and compared with the reference's introspection
    (tests/golden/reference/cli_api.json.gz)."""
    import json
    import os
    import subprocess
    import sys
    from pathlib import Path

    repo = Path(__file__).resolve().parents[1]
    from conftest import reference_golden, run_arms

    env = dict(os.environ, PYTHONPATH=str(repo))
    dumps = run_arms(lambda which: [sys.executable, str(repo / "tests" / "workers" / "cli_tree_dump.py"), which], arms=("ours",), cwd=repo, env=env)
    dumps["ref"] = reference_golden("cli_api")
    assert dumps["ours"]["api"] == dumps["ref"]["api"] and len(dumps["ref"]["api"]) >= 12, (dumps["ours"]["api"], dumps["ref"]["api"])
    ours, ref = dumps["ours"]["cli"], dumps["ref"]["cli"]
    assert set(ours) == set(ref) and len(ref) >= 15, (sorted(set(ref) - set(ours)), sorted(set(ours) - set(ref)))
    for cmd in ref:
        mine = {tuple(p[1]): p[2:] for p in ours[cmd]}
        theirs = {tuple(p[1]): p[2:] for p in ref[cmd]}
        assert all(k in mine and mine[k] == v for k, v in theirs.items()), (cmd, sorted(set(theirs) - set(mine)))
        assert set(mine) - set(theirs) <= {("--backend",)}, (cmd, sorted(set(mine) - set(theirs)))


def test_public_classes_methods_and_parameter_names_match_the_reference():
    """tests/workers/reference_surface_probe.py: for every module of the reference — every public method and annotated field
    of its 320+ public classes exists on the class its import path resolves to here, and every public function / method /
    constructor (400+) accepts the reference's parameter names (user code calls them by keyword)."""
    import json
    import subprocess
    import sys
    from pathlib import Path

    repo = Path(__file__).resolve().parents[1]
    r = subprocess.run([sys.executable, str(repo / "tests" / "workers" / "reference_surface_probe.py")], capture_output=True, text=True, cwd=repo)
    assert r.returncode == 0, r.stderr[-3000:]
    rep = json.loads(r.stdout.strip().splitlines()[-1])
    assert rep["classes"] > 300 and rep["methods"] > 250 and rep["callables"] > 380, rep
    assert rep["missing_members"] == {} and rep["missing_parameters"] == {}, rep


def test_every_pydantic_schema_and_enum_of_the_reference_has_the_same_fields_here():
    """All 120+ pydantic models of the reference (component configs, instantiation models, settings): every field exists on
    the model its import path resolves to here with the same required-ness, alias and (for literal defaults) default
    value; this framework only ADDS optional fields (e.g. ``low_memory``)."""
    import json
    import subprocess
    import sys
    from pathlib import Path

    repo = Path(__file__).resolve().parents[1]
    from conftest import reference_golden, run_arms

    dumps = run_arms(lambda which: [sys.executable, str(repo / "tests" / "workers" / "pydantic_schema_dump.py"), which], arms=("ours",), cwd=repo)
    dumps["ref"] = reference_golden("pydantic_schemas")
    # enums (37): same members, same values where the value is a literal (MixedPrecisionSettings maps onto other policy objects)
    for name, members in dumps["ref"]["enums"].items():
        mine = dumps["ours"]["enums"].get(name)
        assert mine is not None and set(members) <= set(mine), (name, members, mine)
        for k, v in members.items():
            assert mine[k] == v or "(" in v or "<" in v, (name, k, mine[k], v)
    assert len(dumps["ref"]["enums"]) > 30
    ours, ref = dumps["ours"]["models"], dumps["ref"]["models"]
    assert len(ref) > 110 and set(ref) <= set(ours), sorted(set(ref) - set(ours))
    problems = []
    for model, fields in ref.items():
        for fname, (required, default, alias) in fields.items():
            mine = ours[model].get(fname)
            if mine is None or mine[0] != required or mine[2] != alias:
                problems.append((model, fname, mine, (required, default, alias)))
            elif not default.startswith("<") and "object at" not in default and mine[1] != default and not mine[1].startswith("<"):
                problems.append((model, fname, mine, (required, default, alias)))
        extra_required = [f for f, v in ours[model].items() if f not in fields and v[0]]
        if extra_required:
            problems.append((model, "extra required fields", extra_required))
    assert not problems, problems[:10]
