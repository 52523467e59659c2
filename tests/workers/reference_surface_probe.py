"""Compares the public surface of every reference module with what its import path resolves to here (through the alias
finder): public methods / annotated fields of every public class, and the parameter NAMES of every public function,
method and constructor. The reference's surface is read from tests/golden/reference/surface.json.gz (written by
``extract`` from a reference checkout, see scripts/reference_goldens.py). Prints a JSON report;
tests/test_utils_and_tools.py asserts that it is empty.

    python tests/workers/reference_surface_probe.py                          # check this package
    python tests/workers/reference_surface_probe.py extract <src/modalities>  # print the surface of a reference checkout
"""

import ast
import gzip
import importlib
import inspect
import json
import os
import sys
from pathlib import Path

REPO = Path(__file__).resolve().parents[2]
GOLDEN = REPO / "tests" / "golden" / "reference" / "surface.json.gz"
SKIP = {"__main__", "conversion.gpt2.modeling_gpt2"}  # (the exported HF model code is an independent implementation here)


def ref_params(fn):
    a = fn.args
    return [x.arg for x in a.posonlyargs + a.args + a.kwonlyargs if x.arg not in ("self", "cls")]


def extract(root: str) -> dict:
    """{module: {"defs": public top-level names, "functions": {name: params},
    "classes": {name: {"methods": [...], "fields": [...], "callables": {method: params}}}}} of every module under root."""
    surface = {}
    for dp, _, fs in os.walk(root):
        for f in sorted(fs):
            if not f.endswith(".py"):
                continue
            rel = os.path.relpath(os.path.join(dp, f), root)[:-3].replace(os.sep, ".")
            rel = rel.removesuffix(".__init__").removesuffix("__init__")
            if not rel or rel == "__main__":
                continue
            body = ast.parse(open(os.path.join(dp, f)).read()).body
            defs = [n.name for n in body if isinstance(n, (ast.ClassDef, ast.FunctionDef)) and not n.name.startswith("_")]
            defs += [t.id for n in body if isinstance(n, ast.Assign) for t in n.targets if isinstance(t, ast.Name) and t.id.isupper()]
            functions, classes = {}, {}
            for node in body:
                if isinstance(node, ast.FunctionDef) and not node.name.startswith("_"):
                    functions[node.name] = ref_params(node)
                if isinstance(node, ast.ClassDef) and not node.name.startswith("_"):
                    c = classes[node.name] = {"methods": [], "fields": [], "callables": {}}
                    for b in node.body:
                        if isinstance(b, (ast.FunctionDef, ast.AsyncFunctionDef)):
                            if not b.name.startswith("_"):
                                c["methods"].append(b.name)
                            if not b.name.startswith("_") or b.name == "__init__":
                                c["callables"][b.name] = ref_params(b)
                        elif isinstance(b, ast.AnnAssign) and isinstance(b.target, ast.Name) and not b.target.id.startswith("_"):
                            c["fields"].append(b.target.id)
            surface[rel] = {"defs": defs, "functions": functions, "classes": classes}
    return dict(sorted(surface.items()))


def our_params(obj):
    try:
        sig = inspect.signature(obj)
    except (TypeError, ValueError):
        return None
    names = [p.name for p in sig.parameters.values() if p.kind not in (p.VAR_POSITIONAL, p.VAR_KEYWORD)]
    return names, any(p.kind == p.VAR_KEYWORD for p in sig.parameters.values())


def check(surface: dict) -> dict:
    sys.path.insert(0, str(REPO))
    import modalities_b200  # noqa: F401
    from modalities_b200 import compat

    compat.install_modalities_alias()
    report = {"missing_members": {}, "missing_parameters": {}, "classes": 0, "methods": 0, "callables": 0}
    for rel, mod in surface.items():
        if rel in SKIP:
            continue
        m = importlib.import_module("modalities." + rel)
        callables = [(name, params, getattr(m, name)) for name, params in mod["functions"].items() if hasattr(m, name)]
        for cname, c in mod["classes"].items():
            if not hasattr(m, cname):
                continue
            cls = getattr(m, cname)
            report["classes"] += 1
            fields = set(getattr(cls, "model_fields", None) or {}) | set(getattr(cls, "__dataclass_fields__", None) or {})
            fields |= set(getattr(cls, "__annotations__", None) or {})
            report["methods"] += len(c["methods"])
            missing = [b for b in c["methods"] if not hasattr(cls, b)]
            missing += [b for b in c["fields"] if not hasattr(cls, b) and b not in fields]
            callables += [(f"{cname}.{b}", params, getattr(cls, b)) for b, params in c["callables"].items() if hasattr(cls, b)]
            if missing:
                report["missing_members"][f"{rel}.{cname}"] = missing
        for name, params, obj in callables:
            ours = our_params(obj)
            if ours is None:
                continue
            report["callables"] += 1
            names, has_kwargs = ours
            lacking = [p for p in params if p not in names]
            if lacking and not has_kwargs:
                report["missing_parameters"][f"{rel}.{name}"] = lacking
    return report


if __name__ == "__main__":
    if len(sys.argv) > 2 and sys.argv[1] == "extract":
        print(json.dumps(extract(sys.argv[2])))
    else:
        print(json.dumps(check(json.loads(gzip.decompress(GOLDEN.read_bytes())))))
