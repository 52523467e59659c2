import os
import sys
import tempfile
from pathlib import Path

import pytest

REPO = Path(__file__).resolve().parents[1]
if str(REPO) not in sys.path:
    sys.path.insert(0, str(REPO))

# transformers copies the code of a trust_remote_code model into HF_MODULES_CACHE (by default under HF_HOME, which need not
# be writable by the user running the tests); the tests export and reload such models, so the copies go to a temporary
# directory of the session — set before anything imports transformers, and inherited by the tests' subprocesses
_HF_MODULES = tempfile.TemporaryDirectory(prefix="mb200_hf_modules_")
os.environ["HF_MODULES_CACHE"] = _HF_MODULES.name

DATA = REPO / "data"
# what the reference implementation computes for the differential tests (scripts/reference_goldens.py writes it)
REFERENCE_GOLDEN = REPO / "tests" / "golden" / "reference"


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: test needs a CUDA device (run on the B200 box: pytest -m gpu)")


def pytest_unconfigure(config):
    _HF_MODULES.cleanup()


def pytest_collection_modifyitems(config, items):
    import torch

    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="needs a GPU")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture
def lorem_pbin() -> Path:
    return DATA / "lorem_ipsum_long.pbin"


@pytest.fixture
def lorem_jsonl() -> Path:
    return DATA / "lorem_ipsum.jsonl"


@pytest.fixture
def free_port() -> int:
    import socket

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.fixture
def dist_env_single(free_port, monkeypatch):
    """gloo process group of size 1 in this process (reference analogue: tests/conftest.py:231-262)."""
    import torch.distributed as dist

    for k, v in {"RANK": "0", "LOCAL_RANK": "0", "WORLD_SIZE": "1", "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": str(free_port)}.items():
        monkeypatch.setenv(k, v)
    dist.init_process_group("gloo")
    yield
    dist.destroy_process_group()


def reference_golden(name: str):
    import gzip
    import json

    return json.loads(gzip.decompress((REFERENCE_GOLDEN / f"{name}.json.gz").read_bytes()))


def run_arms(make_cmd, arms=("ref", "ours"), cwd=None, env=None, timeout=600):
    """Start one worker process per arm (the reference through baseline/_ref, this framework) concurrently and return
    ``{arm: last stdout line parsed as JSON}``; asserts on the exit codes."""
    import json
    import subprocess

    procs = {a: subprocess.Popen(make_cmd(a), cwd=cwd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for a in arms}
    out = {}
    for a, p in procs.items():
        so, se = p.communicate(timeout=timeout)
        assert p.returncode == 0, (a, se[-3000:])
        out[a] = json.loads(so.strip().splitlines()[-1])
    return out
