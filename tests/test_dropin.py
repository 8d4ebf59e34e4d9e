"""The drop-in boundary under the reference driver's own import block (VERDICT r1 item 6).

`python tool/video_inpainting.py` resolves `utils.region_fill`, `utils.Poisson_blend_img` and `get_flowNN_gradient`
from the script's directory before PYTHONPATH; dropin/run_driver.py reorders the path. The test builds a miniature
reference tree (same package layout and the same import statements as tool/video_inpainting.py:1-33, marker modules
instead of the real code), runs its driver through the launcher in a fresh interpreter and checks that every one
of the six hot-path symbols comes from fgt_b200 while the modules the shims do not replace (RAFT.utils, other
utils.*) still come from the reference tree. The same check also runs against the real driver's import statements
and the real tree's module layout, both recorded from the original project in tests/golden/reference_driver_imports.json
(the driver itself needs cvbase / imageio / skimage, so its imports are replayed rather than executed).
"""
import json
import os
import subprocess
import sys
import textwrap

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LAUNCHER = os.path.join(ROOT, "dropin", "run_driver.py")

# the driver's import block (tool/video_inpainting.py:4-6 path appends, :25-33 imports, :200-230 importlib loads)
DRIVER = textwrap.dedent('''
    import os, sys, json
    sys.path.append(os.path.abspath(os.path.join(__file__, "..", "..")))
    sys.path.append(os.path.abspath(os.path.join(__file__, "..", "..", "FGT")))
    sys.path.append(os.path.abspath(os.path.join(__file__, "..", "..", "LAFC")))
    from RAFT import utils
    from RAFT import RAFT
    from importlib import import_module
    import utils.region_fill as rf
    from utils.Poisson_blend_img import Poisson_blend_img
    from get_flowNN_gradient import get_flowNN_gradient
    fgt = import_module("FGT.models.model")
    lafc = import_module("LAFC.models.lafc")
    import utils.other_helper as oh
    out = {
        "RAFT": RAFT.__module__, "regionfill": rf.regionfill.__module__, "Poisson_blend_img": Poisson_blend_img.__module__,
        "get_flowNN_gradient": get_flowNN_gradient.__module__, "FGT.Model": fgt.Model.__module__,
        "LAFC.Model": lafc.Model.__module__, "RAFT.utils": utils.__file__, "utils.other_helper": oh.__file__,
        "argv": sys.argv[1:],
    }
    print("RESULT " + json.dumps(out))
''')


def _mini_reference(tmp):
    def w(rel, text=""):
        p = os.path.join(tmp, rel)
        os.makedirs(os.path.dirname(p), exist_ok=True)
        with open(p, "w") as fh:
            fh.write(text)

    w("tool/video_inpainting.py", DRIVER)
    w("tool/get_flowNN_gradient.py", "def get_flowNN_gradient(*a):\n    raise RuntimeError('reference')\n")
    w("tool/utils/__init__.py")
    w("tool/utils/region_fill.py", "def regionfill(*a):\n    raise RuntimeError('reference')\n")
    w("tool/utils/Poisson_blend_img.py", "def Poisson_blend_img(*a):\n    raise RuntimeError('reference')\n")
    w("tool/utils/other_helper.py", "X = 1\n")
    w("RAFT/__init__.py", "class RAFT:\n    pass\n")
    w("RAFT/utils/__init__.py")
    w("FGT/__init__.py")
    w("FGT/models/__init__.py")
    w("FGT/models/model.py", "class Model:\n    pass\n")
    w("LAFC/__init__.py")
    w("LAFC/models/__init__.py")
    w("LAFC/models/lafc.py", "class Model:\n    pass\n")
    return os.path.join(tmp, "tool", "video_inpainting.py")


def _run(cmd, cwd):
    env = {k: v for k, v in os.environ.items() if k != "PYTHONPATH"}
    r = subprocess.run(cmd, cwd=cwd, env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")][-1]
    return json.loads(line[len("RESULT "):])


def test_launcher_resolves_all_six_symbols_to_fgt_b200(tmp_path):
    driver = _mini_reference(str(tmp_path))
    got = _run([sys.executable, LAUNCHER, driver, "--opt", "x.yaml"], str(tmp_path))
    for key in ("RAFT", "regionfill", "Poisson_blend_img", "get_flowNN_gradient", "FGT.Model", "LAFC.Model"):
        assert got[key].startswith("fgt_b200."), (key, got[key])
    # modules the shims do not replace still come from the reference tree
    assert got["RAFT.utils"].startswith(str(tmp_path)) and got["utils.other_helper"].startswith(str(tmp_path))
    assert got["argv"] == ["--opt", "x.yaml"]


def test_plain_invocation_is_why_the_launcher_exists(tmp_path):
    """Without the launcher (python tool/video_inpainting.py with PYTHONPATH=dropin:repo) the three tool/ modules
    shadow the shims — the behaviour VERDICT r1 reproduced; kept as a regression check of the premise."""
    driver = _mini_reference(str(tmp_path))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "dropin"), ROOT]))
    r = subprocess.run([sys.executable, driver], cwd=str(tmp_path), env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    got = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")][-1][len("RESULT "):])
    assert got["FGT.Model"].startswith("fgt_b200.") and got["RAFT"].startswith("fgt_b200.")
    assert not got["regionfill"].startswith("fgt_b200.")


def test_real_reference_tree_imports(tmp_path):
    """Replays the real driver's import statements for the modules of its own tree (as recorded from its source)
    under the launcher's path order, in a tree with the real tree's package layout (empty modules)."""
    with open(os.path.join(ROOT, "tests", "golden", "reference_driver_imports.json")) as fh:
        rec = json.load(fh)
    for stmt in ("from RAFT import utils", "from RAFT import RAFT", "import utils.region_fill as rf",
                 "from utils.Poisson_blend_img import Poisson_blend_img",
                 "from get_flowNN_gradient import get_flowNN_gradient"):
        assert stmt in rec["imports"], stmt
    ref = str(tmp_path / "reference")
    for rel in rec["modules"]:
        p = os.path.join(ref, rel)
        os.makedirs(os.path.dirname(p), exist_ok=True)
        open(p, "w").close()
    imports = "\n".join(rec["imports"])
    prog = textwrap.dedent(f'''
        import sys, json
        sys.path.insert(0, {os.path.join(ROOT, "dropin")!r})
        import run_driver
        run_driver.setup_path({os.path.join(ref, rec["driver"])!r})
        sys.path += [{ref!r}, {os.path.join(ref, "FGT")!r}, {os.path.join(ref, "LAFC")!r}]
        exec({imports!r})
        from importlib import import_module
        fgt = import_module("FGT.models.model"); lafc = import_module("LAFC.models.lafc")
        print("RESULT " + json.dumps({{"RAFT": RAFT.__module__, "regionfill": rf.regionfill.__module__,
              "Poisson_blend_img": Poisson_blend_img.__module__, "get_flowNN_gradient": get_flowNN_gradient.__module__,
              "FGT.Model": fgt.Model.__module__, "LAFC.Model": lafc.Model.__module__, "RAFT.utils": utils.__file__}}))
    ''')
    got = _run([sys.executable, "-c", prog], str(tmp_path))
    for key in ("RAFT", "regionfill", "Poisson_blend_img", "get_flowNN_gradient", "FGT.Model", "LAFC.Model"):
        assert got[key].startswith("fgt_b200."), (key, got[key])
    assert got["RAFT.utils"].startswith(os.path.join(ref, "RAFT", "utils"))
