"""Records what tests/test_dropin.py::test_real_reference_tree_imports checks the launcher against, from a checkout of
the original FGT project:

* the module-level import statements of tool/video_inpainting.py that load modules of the project's own tree
  (RAFT, utils.*, get_flowNN_gradient), normalised by ast.unparse;
* the relative path of every .py file of the tree (the package layout that decides how those imports resolve).

No source text beyond those import statements is stored.

    python tests/golden/make_dropin_golden.py /path/to/original/FGT   -> tests/golden/reference_driver_imports.json
"""
import ast
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DRIVER = "tool/video_inpainting.py"


def main(ref):
    modules = sorted(os.path.relpath(os.path.join(d, f), ref).replace(os.sep, "/")
                     for d, _, files in os.walk(ref) for f in files if f.endswith(".py"))
    # where the driver's imports are searched in its own tree: its directory, then the roots it appends (:4-6)
    roots = [os.path.join(ref, "tool"), ref, os.path.join(ref, "FGT"), os.path.join(ref, "LAFC")]
    local = {n[:-3] if n.endswith(".py") else n for r in roots for n in os.listdir(r)
             if n.endswith(".py") or os.path.isdir(os.path.join(r, n))}
    with open(os.path.join(ref, DRIVER)) as fh:
        tree = ast.parse(fh.read())
    imports = []
    for node in tree.body:
        if isinstance(node, ast.Import):
            tops = [a.name.split(".")[0] for a in node.names]
        elif isinstance(node, ast.ImportFrom) and node.level == 0:
            tops = [node.module.split(".")[0]]
        else:
            continue
        if any(t in local for t in tops):
            imports.append(ast.unparse(node))
    out = os.path.join(HERE, "reference_driver_imports.json")
    with open(out, "w") as fh:
        json.dump({"driver": DRIVER, "imports": imports, "modules": modules}, fh, indent=1)
        fh.write("\n")
    print(out, len(imports), "imports,", len(modules), "modules")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: python tests/golden/make_dropin_golden.py /path/to/original/FGT")
    main(os.path.abspath(sys.argv[1]))
