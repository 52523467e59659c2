"""Dumps every pydantic model of the reference's module tree — of the installed reference (``ref``, baseline/_ref) or of what
the same module paths resolve to here (``ours``; the class names are those of the reference's dump stored in
tests/golden/reference/pydantic_schemas.json.gz) — as JSON: {module.Class: {field: [required, default repr, alias]}}, plus every
Enum: {module.Class: {member: value repr}}."""

import enum
import gzip
import importlib
import json
import os
import sys
from pathlib import Path

REPO = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(REPO))
which = sys.argv[1]
if which == "ref":
    sys.path.insert(0, str(REPO / "baseline"))
    import ref_env

    ref_env.prepare()
else:
    import modalities_b200  # noqa: F401
    from modalities_b200 import compat

    compat.install_modalities_alias()
from pydantic import BaseModel  # noqa: E402


def reference_classes():
    """{module: [class names]} — the classes the REFERENCE's files define."""
    if which != "ref":
        golden = json.loads(gzip.decompress((REPO / "tests" / "golden" / "reference" / "pydantic_schemas.json.gz").read_bytes()))
        classes = {}
        for key in [*golden["models"], *golden["enums"]]:
            rel, name = key.rsplit(".", 1)
            classes.setdefault(rel, []).append(name)
        return classes
    import re

    root = REPO / "baseline" / "_ref" / "modalities"
    classes = {}
    for dp, _, fs in os.walk(root):
        for f in fs:
            rel = os.path.relpath(os.path.join(dp, f), root)[:-3].replace(os.sep, ".").removesuffix(".__init__").removesuffix("__init__")
            if f.endswith(".py") and rel and rel != "__main__":
                classes[rel] = re.findall(r"^class (\w+)\(", (Path(dp) / f).read_text(), flags=re.M)
    return classes


out, failed, enums = {}, [], {}
for rel, names in reference_classes().items():
    try:
        m = importlib.import_module("modalities." + rel)
    except Exception as e:  # noqa: BLE001
        failed.append((rel, type(e).__name__))
        continue
    for name in names:
        obj = getattr(m, name, None)  # (getattr: some schemas are resolved lazily here)
        if isinstance(obj, type) and issubclass(obj, enum.Enum):
            enums[f"{rel}.{name}"] = {k: repr(v.value)[:60] for k, v in obj.__members__.items()}
        if isinstance(obj, type) and issubclass(obj, BaseModel) and obj is not BaseModel:
            fields = {}
            for fname, fi in obj.model_fields.items():
                d = fi.default
                default = "<required>" if fi.is_required() else ("<factory>" if fi.default_factory is not None else repr(d))
                fields[fname] = [fi.is_required(), default, fi.alias]
            out[f"{rel}.{name}"] = fields
print(json.dumps({"models": out, "enums": enums, "import_failed": failed}))
