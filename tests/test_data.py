"""Data layer: index / pbin formats, datasets, samplers, collators, dataloader fast path, data tools."""
from pathlib import Path
import json
import pickle

import numpy as np
import pytest
import torch
from torch.utils.data import BatchSampler

from modalities_b200.api import FileExistencePolicy, create_raw_data_index, create_shuffled_dataset_chunk, merge_packed_data_files
from modalities_b200.batch import DatasetBatch
from modalities_b200.data import jq
from modalities_b200.data.collators import GPT2LLMCollateFn, LossMaskingCollateFnWrapper, LossMaskingTokenConfig
from modalities_b200.data.create_index import IndexGenerator
from modalities_b200.data.create_packed_data import PackedDataGenerator
from modalities_b200.data.dataloader_factory import DataloaderFactory
from modalities_b200.data.dataset import PackedMemMapDatasetBase, PackedMemMapDatasetContinuous
from modalities_b200.data.dataset_factory import DatasetFactory
from modalities_b200.data.large_file_lines_reader import LargeFileLinesReader
from modalities_b200.data.packed_format import EmbeddedStreamData, token_size_for_vocab
from modalities_b200.data.samplers import ResumableDistributedSampler
from modalities_b200.preprocessing.create_chunks import Chunking
from modalities_b200.preprocessing.shuffle_data import DataShuffler
from modalities_b200.tokenization.tokenizer_wrapper import TokenizerWrapper


class CharTokenizer(TokenizerWrapper):
    """byte-level toy tokenizer, id 255 = <eod>"""

    def tokenize(self, text):
        return list(text.encode("utf-8")[:200])

    def decode(self, ids):
        return bytes(i for i in ids if i < 255).decode("utf-8", errors="ignore")

    @property
    def vocab_size(self):
        return 256

    def get_token_id(self, token):
        if token == "<eod>":
            return 255
        raise ValueError(token)

    def is_special_token_id(self, token_id):
        return token_id == 255


def test_jq_subset():
    assert jq.compile(".text").input_text('{"text": "hi"}').first() == "hi"
    assert jq.compile(".a.b[1].c").input_text('{"a": {"b": [1, {"c": 5}]}}').first() == 5
    assert jq.compile('.["k y"]').input_text('{"k y": 2}').first() == 2
    assert jq.compile(".missing").input_text("{}").first() is None
    with pytest.raises(ValueError):
        jq.compile(".a | length")


def test_index_native_equals_python_and_shipped_index(lorem_jsonl, tmp_path):
    gen = IndexGenerator(lorem_jsonl)
    assert gen._scan() == gen._scan_python()
    idx_path = tmp_path / "x.idx"
    create_raw_data_index(lorem_jsonl, idx_path, FileExistencePolicy.ERROR)
    index = pickle.loads(idx_path.read_bytes())
    assert len(index) == 12
    reader = LargeFileLinesReader(lorem_jsonl, idx_path)
    assert all("text" in json.loads(reader[i]) for i in range(len(reader)))
    with pytest.raises(ValueError):
        create_raw_data_index(lorem_jsonl, idx_path, FileExistencePolicy.ERROR)


def test_index_faulty_lines_and_missing_trailing_newline(tmp_path):
    p = tmp_path / "d.jsonl"
    p.write_bytes('{"text": "æøå"}\n\n{"broken": \n{"text": "last"}'.encode("utf-8"))
    with pytest.raises(ValueError):
        IndexGenerator(p).create_index(tmp_path / "a.idx")
    IndexGenerator(p, drop_faulty_entries=True).create_index(tmp_path / "b.idx")
    idx = pickle.loads((tmp_path / "b.idx").read_bytes())
    raw = p.read_bytes()
    assert [json.loads(raw[o : o + n])["text"] for o, n in idx] == ["æøå", "last"]


def test_pack_roundtrip_and_shipped_pbin(tmp_path, lorem_pbin):
    src = tmp_path / "d.jsonl"
    docs = ["hello world", "second doc", "x"]
    src.write_text("".join(json.dumps({"text": t}) + "\n" for t in docs))
    create_raw_data_index(src, None)
    for procs in (1, 2):
        dst = tmp_path / f"out{procs}.pbin"
        PackedDataGenerator(src, CharTokenizer(), "<eod>", procs, ".text", 2, 4, 4).run(dst)
        data = EmbeddedStreamData(dst)
        assert data.token_size_in_bytes == 1 and len(data.index_base) == 3
        ds = PackedMemMapDatasetBase(dst, "input_ids")
        assert [bytes(ds[i]["input_ids"][:-1]).decode() for i in range(3)] == docs
        assert all(ds[i]["input_ids"][-1] == 255 for i in range(3))
    assert (tmp_path / "out1.pbin").read_bytes() == (tmp_path / "out2.pbin").read_bytes()
    shipped = EmbeddedStreamData(lorem_pbin)
    assert shipped.num_tokens == 332875 and len(shipped.index_base) == 500 and shipped.token_size_in_bytes == 2
    assert token_size_for_vocab(50257) == 2 and token_size_for_vocab(256) == 1 and token_size_for_vocab(70000) == 4


@pytest.mark.parametrize("reuse", [True, False])
def test_continuous_packing_index(lorem_pbin, reuse):
    ds = PackedMemMapDatasetContinuous(lorem_pbin, "input_ids", block_size=129 if reuse else 128, reuse_last_target=reuse)
    total = 332875
    assert len(ds) == ((total - 129) // 128 + 1 if reuse else total // 128)
    a, b = ds[0]["input_ids"], ds[1]["input_ids"]
    assert (b[0] == a[-1]) == reuse and len(a) == (129 if reuse else 128)
    with pytest.raises(ValueError):
        PackedMemMapDatasetContinuous(lorem_pbin, "input_ids", block_size=10**7, reuse_last_target=True)


def test_combined_and_megatron(lorem_pbin):
    ds = DatasetFactory.get_packed_mem_map_dataset_continuous(lorem_pbin, 256, "input_ids")
    comb = DatasetFactory.get_combined_dataset([ds, ds])
    assert len(comb) == 2 * len(ds) and (comb[len(ds) + 3]["input_ids"] == ds[3]["input_ids"]).all()
    mega = DatasetFactory.get_packed_mem_map_dataset_megatron(lorem_pbin, 256, "input_ids")
    assert len(mega) > 0 and all(len(mega[i]["input_ids"]) == 257 for i in (0, len(mega) - 1))


@pytest.mark.parametrize("n,replicas,skip,shuffle", [(100, 4, 0, False), (103, 4, 10, True), (17, 3, 5, True)])
def test_resumable_sampler(n, replicas, skip, shuffle):
    data = list(range(n))
    per_rank = [list(ResumableDistributedSampler(data, r, replicas, epoch=1, shuffle=shuffle, seed=7, drop_last=True,
                                                 skip_num_global_samples=skip)) for r in range(replicas)]  # fmt: skip
    lengths = {len(x) for x in per_rank}
    assert len(lengths) == 1
    flat = [i for x in per_rank for i in x]
    assert len(set(flat)) == len(flat)
    if shuffle:
        g = torch.Generator()
        g.manual_seed(7 + 1)
        order = torch.randperm(n, generator=g).tolist()
    else:
        order = data
    expected = order[skip:][: len(flat)]
    assert sorted(flat) == sorted(expected)
    assert per_rank[1][:2] == expected[1 : 1 + 2 * replicas : replicas]
    # resuming: skipping k more samples continues the same global order
    resumed = list(ResumableDistributedSampler(data, 0, replicas, epoch=1, shuffle=shuffle, seed=7, drop_last=True,
                                               skip_num_global_samples=skip + replicas))  # fmt: skip
    assert resumed[: len(per_rank[0]) - 2] == per_rank[0][1:][: len(per_rank[0]) - 2]


def test_gpt2_collator_and_loss_masking_truth_table():
    coll = GPT2LLMCollateFn("input_ids", "target_ids")
    batch = coll([{"input_ids": np.arange(6)}, {"input_ids": np.arange(6) + 10}])
    assert batch.samples["input_ids"].tolist() == [[0, 1, 2, 3, 4], [10, 11, 12, 13, 14]]
    assert batch.targets["target_ids"].tolist() == [[1, 2, 3, 4, 5], [11, 12, 13, 14, 15]]

    class Tok(CharTokenizer):
        def get_token_id(self, token):
            return {"<b>": 3, "<e>": 4}[token]

    wrapper = LossMaskingCollateFnWrapper(coll, ["target_ids"], -100, LossMaskingTokenConfig(b_include_to_loss_token="<b>", e_include_to_loss_token="<e>"), Tok())
    out = wrapper([{"input_ids": np.array([2, 2, 3, 2, 2, 4, 2, 2, 2])}])
    assert out.targets["target_ids"].tolist() == [[-100, -100, 2, 2, -100, -100, -100, -100]]
    # end marker before begin marker -> error; no markers -> everything ignored
    with pytest.raises(ValueError):
        wrapper([{"input_ids": np.array([2, 4, 2, 3, 2, 2])}])
    assert set(wrapper([{"input_ids": np.array([2, 2, 2, 2])}]).targets["target_ids"].flatten().tolist()) == {-100}
    with pytest.raises(ValueError):
        class Same(CharTokenizer):
            def get_token_id(self, token):
                return 3
        LossMaskingCollateFnWrapper(coll, ["target_ids"], -100, LossMaskingTokenConfig(b_include_to_loss_token="<b>", e_include_to_loss_token="<e>"), Same())


def test_dataloader_fast_path_is_bit_identical(lorem_pbin):
    ds = DatasetFactory.get_packed_mem_map_dataset_continuous(lorem_pbin, 64, "input_ids")
    for dataset in (ds, DatasetFactory.get_combined_dataset([ds, ds])):
        batches = []
        for fast in (True, False):
            sampler = ResumableDistributedSampler(dataset, rank=1, num_replicas=2, shuffle=True, seed=3, drop_last=True, skip_num_global_samples=8)
            dl = DataloaderFactory.get_dataloader("train", dataset, BatchSampler(sampler, 4, True), GPT2LLMCollateFn("input_ids", "target_ids"), 0, False)
            dl._fast_path_enabled = fast
            batches.append([b for _, b in zip(range(6), dl)])
            assert dl.dataloader_tag == "train" and dl.batch_size == 4 and isinstance(batches[-1][0], DatasetBatch)
        for a, b in zip(*batches):
            assert torch.equal(a.samples["input_ids"].long(), b.samples["input_ids"].long())
            assert torch.equal(a.targets["target_ids"].long(), b.targets["target_ids"].long())


def test_chunks_shuffle_merge(tmp_path, lorem_pbin):
    assert [Chunking._get_chunk_range(3, 10, i) for i in range(3)] == [[0, 4], [4, 7], [7, 10]]
    assert [Chunking._get_chunk_range(2, 10, i) for i in range(2)] == [[0, 5], [5, 10]]
    out = tmp_path / "shuf.pbin"
    DataShuffler.shuffle_tokenized_data(lorem_pbin, out, batch_size=64, seed=1)
    a, b = PackedMemMapDatasetBase(lorem_pbin, "t"), PackedMemMapDatasetBase(out, "t")
    assert len(a) == len(b) and sorted(len(a[i]["t"]) for i in range(len(a))) == sorted(len(b[i]["t"]) for i in range(len(b)))
    assert any((len(a[i]["t"]) != len(b[i]["t"])) for i in range(20))
    chunk = tmp_path / "chunk.pbin"
    create_shuffled_dataset_chunk([lorem_pbin, out], chunk, chunk_id=1, num_chunks=4, file_existence_policy=FileExistencePolicy.ERROR, global_seed=5)
    assert len(PackedMemMapDatasetBase(chunk, "t")) == 250
    merged = tmp_path / "merged.pbin"
    merge_packed_data_files([lorem_pbin, out], merged)
    m = EmbeddedStreamData(merged)
    assert m.num_tokens == 2 * 332875 and len(m.index_base) == 1000


@pytest.mark.parametrize("kind", ["hugging_face", "sentence_piece"])
def test_end_to_end_indexation_and_tokenization_consistency(kind, tmp_path, monkeypatch):
    """index → tokenize+pack → verify against a fresh tokenization (reference analogue:
    /root/reference/tests/end2end_tests/test_tokenization_consistency.py... verify_tokenization_consistency)."""
    import json

    from modalities_b200.utils.verify_tokenization_consistency import (
        build_hf_tokenization_components,
        build_sp_tokenization_components,
        verify_tokenization_consistency,
    )

    tok_root = Path(__file__).resolve().parents[1] / "data" / "tokenizer"
    src = tmp_path / "docs.jsonl"
    texts = ["Hello world, this is a test.", "Zweiter Text mit Umlauten: äöü ß.", "x", "Final document\twith a tab and 数字 123."]
    src.write_text("".join(json.dumps({"text": t, "id": i}, ensure_ascii=False) + "\n" for i, t in enumerate(texts)), encoding="utf-8")
    for k, v in {"RANK": "0", "LOCAL_RANK": "0", "WORLD_SIZE": "1"}.items():
        monkeypatch.setenv(k, v)
    if kind == "hugging_face":
        eod = "<|endoftext|>"
        fn, cfg, eod_id = build_hf_tokenization_components(str(tok_root / "hf_gpt2"), eod)
    else:
        eod = "</s>"
        fn, cfg, eod_id = build_sp_tokenization_components(tok_root / "sentencepiece_dclm" / "en_32k_tokenizer.model", eod)
    verify_tokenization_consistency(src_path=src, eod_token=eod, eod_token_id=eod_id, tokenizer=fn, tokenizer_config=cfg, jsonl_text_key="text")


def test_sentencepiece_tokenizer_conversion_to_hf(tmp_path):
    """Reference analogue: /root/reference/tests/conversion/gpt2/test_conversion_tokenizer.py."""
    from transformers import AutoTokenizer

    from modalities_b200.conversion.gpt2.conversion_tokenizer import convert_tokenizer
    from modalities_b200.tokenization.tokenizer_wrapper import PreTrainedSPTokenizer

    model_file = Path(__file__).resolve().parents[1] / "data" / "tokenizer" / "sentencepiece_dclm" / "en_32k_tokenizer.model"
    bos, eos, pad, unk = convert_tokenizer(str(model_file), str(tmp_path))
    sp = PreTrainedSPTokenizer(str(model_file))
    assert (bos, eos, pad, unk) == (sp.tokenizer.bos_id(), sp.tokenizer.eos_id(), sp.tokenizer.pad_id(), sp.tokenizer.unk_id())
    hf = AutoTokenizer.from_pretrained(tmp_path)
    # (runs of leading spaces are normalised differently by the tokenizers-backed LlamaTokenizer of transformers >= 5)
    for text in ["Hello world!", "A longer sentence, with punctuation; and numbers 12345.", "Two\nlines and a tab\t."]:
        assert hf(text, add_special_tokens=False)["input_ids"] == sp.tokenize(text)


def test_chat_template_application_and_split(tmp_path):
    """Instruction-tuning preparation step 1 (reference analogue: tests/instruction_tuning/test_e2e_instruction_tuning.py):
    role mapping, sandboxed jinja2 rendering into ``chat``, hash-suffixed outputs, weighted train/val/test split."""
    import yaml

    from modalities_b200.data.apply_chat_template import split_and_apply_chat_template

    src = tmp_path / "conversations.jsonl"
    rows = [{"id": i, "conversations": [{"from": "human", "value": f"question {i}"}, {"from": "gpt", "value": f"answer {i}"}]} for i in range(40)]
    src.write_text("".join(json.dumps(r) + "\n" for r in rows))
    template = (
        "{{ chat_template_data.system_instruction + '\\n' }}"
        "{% for turn in messages %}{{ turn.role + ': ' + turn.content + '\\n' }}"
        "{% if turn.role == chat_template_data.assistant_role %}{{ chat_template_data.special_tokens.e_include_to_loss_token }}{% endif %}"
        "{% endfor %}"
    )
    config = {
        "settings": {"src_path": str(src), "dst_path": str(tmp_path / "out" / "chat.jsonl"), "messages_key": "conversations",
                     "split_config": {"splitting": {"train": 70, "val": 20, "test": 10}, "seed": 1234}},
        "instruction_data_transformation": {"role_mapping": {"human": "User", "gpt": "Assistant"}},
        "jinja2_chat_template": template,
        "chat_template_data": {"assistant_role": "Assistant", "system_instruction": "Be nice.",
                               "special_tokens": {"b_include_to_loss_token": "^", "e_include_to_loss_token": "$"}},
    }  # fmt: skip
    # the conversation turns use from/value: map them to role/content before the template sees them
    for r in rows:
        for t in r["conversations"]:
            t["role"], t["content"] = t.pop("from"), t.pop("value")
    src.write_text("".join(json.dumps(r) + "\n" for r in rows))
    cfg_file = tmp_path / "apply_chat_template.yaml"
    cfg_file.write_text(yaml.safe_dump(config))
    paths = split_and_apply_chat_template(cfg_file, config)
    assert set(paths) <= {"train", "val", "test"} and "train" in paths
    total = 0
    for part, path in paths.items():
        assert path.parent.name.startswith("conversations_") and path.exists()
        lines = path.read_text().splitlines()
        total += len(lines)
        rec = json.loads(lines[0])
        assert rec["chat"].startswith("Be nice.\n") and "User: question" in rec["chat"] and rec["chat"].rstrip().endswith("$")
    assert total == 40
    # same seed -> same split
    again = split_and_apply_chat_template(cfg_file, config)
    assert {p: len(path.read_text().splitlines()) for p, path in again.items()} == {p: len(path.read_text().splitlines()) for p, path in paths.items()}


def test_cli_index_and_pack_with_shipped_config(tmp_path):
    """`data create_raw_index` + `data pack_encoded_data` through the CLI with configs/data_preparation (GPT-2 tokenizer)."""
    import os
    import subprocess
    import sys

    repo = Path(__file__).resolve().parents[1]
    src = tmp_path / "docs.jsonl"
    src.write_text("".join(json.dumps({"text": f"document number {i} says hello to the world"}) + "\n" for i in range(12)))
    env = dict(os.environ, MB200_SRC_JSONL=str(src), MB200_SRC_IDX=str(tmp_path / "docs.idx"), MB200_DST_PBIN=str(tmp_path / "docs.pbin"),
               RANK="0", LOCAL_RANK="0", WORLD_SIZE="1", CUDA_VISIBLE_DEVICES="")  # fmt: skip
    r = subprocess.run([sys.executable, "-m", "modalities_b200", "data", "create_raw_index", str(src), "--index_path", str(tmp_path / "docs.idx")],
                       cwd=repo, env=env, capture_output=True, text=True, timeout=300)  # fmt: skip
    assert r.returncode == 0, r.stderr[-2000:]
    r = subprocess.run([sys.executable, "-m", "modalities_b200", "data", "pack_encoded_data", "configs/data_preparation/packed_dataset_config.yaml"],
                       cwd=repo, env=env, capture_output=True, text=True, timeout=600)  # fmt: skip
    assert r.returncode == 0, r.stderr[-2000:]
    ds = PackedMemMapDatasetBase(raw_data_path=tmp_path / "docs.pbin", sample_key="text", load_index=True)
    assert len(ds) == 12
    assert ds[0]["text"][-1] == 50256  # <|endoftext|>


def test_index_and_packed_file_are_byte_identical_to_the_reference_pipeline(tmp_path):
    """The reference's own indexer + multi-process tokeniser / packer (the md5 of its files:
    tests/golden/reference/data_pipeline.json.gz) and this framework's, driven through the same library calls on the shipped
    corpus with the local GPT-2 tokenizer, write byte-identical ``.idx`` and ``.pbin`` files (md5)."""
    import sys
    from pathlib import Path

    repo = Path(__file__).resolve().parents[1]
    from conftest import reference_golden, run_arms

    res = run_arms(lambda which: [sys.executable, "tests/workers/reference_data_pipeline.py", which, str(tmp_path / which)], arms=("ours",), cwd=repo)
    res["ref"] = reference_golden("data_pipeline")
    assert res["ours"] == res["ref"] and res["ref"]["pbin_bytes"] > 10_000, res
