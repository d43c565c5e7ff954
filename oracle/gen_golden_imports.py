"""Golden for tests/test_overlay_reference_tree.py: the module structure of the reference files that swap() imports and
that hairfastgan_b200.install() redirects -> tests/golden/reference_imports.json.

    python oracle/gen_golden_imports.py REFERENCE_CHECKOUT

Per file it records names only, read with `ast` (no code is executed or copied): the module-level
`from X import a, b` statements, whether the file puts its own directory on sys.path (FeatureStyleEncoder), the
top-level classes with their method names, and the top-level functions.  The test rebuilds a stand-in tree with
exactly these names and checks that under install() they resolve to this package."""
from __future__ import annotations

import ast
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(os.path.dirname(HERE), "tests", "golden", "reference_imports.json")
FILES = ["models/Net.py", "models/Encoders.py", "models/Embedding.py", "models/Blending.py",
         "models/encoder4editing/models/psp.py", "models/FeatureStyleEncoder/FSencoder.py",
         "models/FeatureStyleEncoder/trainer.py", "models/CtrlHair/external_code/face_parsing/my_parsing_util.py",
         "utils/image_utils.py"]


def _inserts_own_dir(tree) -> bool:
    for node in tree.body:
        if isinstance(node, ast.Expr) and isinstance(node.value, ast.Call):
            f = node.value.func
            if isinstance(f, ast.Attribute) and f.attr == "insert" and ast.unparse(f.value) == "sys.path":
                return True
    return False


def describe(path: str) -> dict:
    tree = ast.parse(open(path).read())
    imports, classes, functions = [], {}, []
    for node in tree.body:
        if isinstance(node, ast.ImportFrom) and node.level == 0:
            imports.append([node.module, [a.name for a in node.names]])
        elif isinstance(node, ast.ClassDef):
            classes[node.name] = [n.name for n in node.body if isinstance(n, (ast.FunctionDef, ast.AsyncFunctionDef))]
        elif isinstance(node, (ast.FunctionDef, ast.AsyncFunctionDef)):
            functions.append(node.name)
    return {"sys_path_insert_own_dir": _inserts_own_dir(tree), "imports": imports, "classes": classes,
            "functions": functions}


def main(ref: str) -> None:
    out = {rel: describe(os.path.join(ref, rel)) for rel in FILES}
    os.makedirs(os.path.dirname(GOLD), exist_ok=True)
    with open(GOLD, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", GOLD, sum(len(d["imports"]) for d in out.values()), "import statements")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
