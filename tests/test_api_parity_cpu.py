"""Name-level parity with the reference's three public bindings (C++ classes / methods of include/mlsl.hpp, the C
functions of include/mlsl.h, the classes / methods of the Python binding) and its enum values.  The reference's names
are stored in tests/golden/reference_api.json; `python tests/test_api_parity_cpu.py <reference checkout>` regenerates
that file with the same extraction the tests apply to this repository's headers and binding."""
import ast
import json
import os
import re
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden", "reference_api.json")


def _golden():
    with open(GOLDEN) as f:
        return json.load(f)


def _cpp_methods(path):
    s = open(path, errors="ignore").read()
    s = re.sub(r"/\*.*?\*/", "", s, flags=re.S)
    s = re.sub(r"//[^\n]*", "", s)
    out = {}
    for m in re.finditer(r"class\s+(\w+)\s*(?::[^{]*)?\{(.*?)\n\s*\};", s, flags=re.S):
        out.setdefault(m.group(1), set()).update(re.findall(r"(\w+)\s*\([^;{]*\)\s*(?:const)?\s*;", m.group(2)))
    return out


def _c_functions(path):
    return set(re.findall(r"\b(mlsl_\w+)\s*\(", open(path, errors="ignore").read()))


def _py_classes(path):
    tree = ast.parse(open(path, errors="ignore").read())
    out = {}
    for node in tree.body:
        if isinstance(node, ast.ClassDef):
            names = {f.name for f in node.body if isinstance(f, ast.FunctionDef) and not f.name.startswith("_")}
            names |= {t.id for a in node.body if isinstance(a, ast.Assign) for t in a.targets
                      if isinstance(t, ast.Name) and not t.id.startswith("_")}
            out[node.name.lstrip("_")] = names
    return out


def _enums(path):
    s = open(path, errors="ignore").read()
    s = re.sub(r"/\*.*?\*/", "", s, flags=re.S)
    s = re.sub(r"//[^\n]*", "", s)
    out = {}
    for m in re.finditer(r"enum\s+(\w+)\s*\{(.*?)\}", s, flags=re.S):
        vals, nxt = {}, 0
        for item in (i.strip() for i in m.group(2).split(",")):
            if not item:
                continue
            if "=" in item:
                item, v = (x.strip() for x in item.split("="))
                nxt = int(v, 0)
            vals[item] = nxt
            nxt += 1
        out[m.group(1)] = vals
    return out


def test_cpp_classes_and_methods():
    ref, mine = _golden()["cpp_methods"], _cpp_methods(os.path.join(ROOT, "include", "mlsl.hpp"))
    assert len(ref) >= 9
    for cls, methods in ref.items():
        assert cls in mine, cls
        missing = sorted(m for m in methods if m not in mine[cls] and m != cls and m != "NO_EXPLICIT_CREATION")
        assert not missing, (cls, missing)


def test_c_functions():
    ref, mine = set(_golden()["c_functions"]), _c_functions(os.path.join(ROOT, "include", "mlsl.h"))
    assert len(ref) >= 100 and not (ref - mine), sorted(ref - mine)


def test_python_classes_and_methods():
    ref = _golden()["python_classes"]
    src = open(os.path.join(ROOT, "mlsl_b200", "api.py")).read()
    mine = _py_classes(os.path.join(ROOT, "mlsl_b200", "api.py"))
    generated = set(re.findall(r'"(\w+)"', src))      # getters generated from name tables (_getters)
    assert len(ref) >= 14
    for cls, methods in ref.items():
        methods = {m for m in methods if m.islower() or "_" in m}
        if not methods:
            continue
        assert cls in mine, cls
        missing = sorted(m for m in methods if m not in mine[cls] and not (m.startswith("get_") and m[4:] in generated)
                         and not (m.startswith("is_") and m[3:] in generated))
        assert not missing, (cls, missing)


def test_enum_values():
    ref, mine = _golden()["enums"], _enums(os.path.join(ROOT, "include", "mlsl.hpp"))
    assert len(ref) >= 6
    for name, vals in ref.items():
        for k, v in vals.items():
            assert mine.get(name, {}).get(k) == v, (name, k, v, mine.get(name, {}).get(k))


if __name__ == "__main__":
    ref = sys.argv[1]
    table = {
        "cpp_methods": {c: sorted(m) for c, m in _cpp_methods(os.path.join(ref, "include", "mlsl.hpp")).items()},
        "c_functions": sorted(_c_functions(os.path.join(ref, "include", "mlsl.h"))),
        "python_classes": {c: sorted(m) for c, m in _py_classes(os.path.join(ref, "include", "mlsl", "mlsl.py")).items()},
        "enums": _enums(os.path.join(ref, "include", "mlsl.hpp")),
    }
    os.makedirs(os.path.dirname(GOLDEN), exist_ok=True)
    with open(GOLDEN, "w") as f:
        json.dump(table, f, indent=1, sort_keys=True)
        f.write("\n")
