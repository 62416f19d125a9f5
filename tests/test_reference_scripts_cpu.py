"""The reference's own demo/ and samples/ scripts must import unchanged on top of the drop-in packages (SURVEY.md
section 8(b)): `PYTHONPATH=<repo>/face-diffusion-model_b200`, cwd = the reference checkout. The hot-path names must
resolve to this repository's classes, everything else of the reference's packages (utiles.flame_utils,
models.lib.base_models, ...) to the reference's own files. The checkout is tests/golden/reference_checkout, laid out like
the reference's: its scripts hold the import blocks of the reference's scripts as recorded in INTEGRATION.md section 1 and
SURVEY.md section 8(b), its utiles/flame_utils.py and models/lib/base_models.py stand in for the reference-only modules.
FDM_B200_REFERENCE_DIR=<reference checkout> runs the same checks on the reference's own scripts."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "face-diffusion-model_b200")
REF = os.environ.get("FDM_B200_REFERENCE_DIR") or os.path.join(ROOT, "tests", "golden", "reference_checkout")

SCRIPTS = ["samples/sample_diffusion_vocaset.py", "samples/sample_diffusion_biwi.py", "samples/sample_diffusion_mead.py",
           "demo/demo_3d_mead.py", "demo/demo_vocaset.py", "demo/demo_biwi.py", "samples/sample_mead_vqvae.py"]

RUNNER = r'''
import importlib.machinery, sys, types
import os
scripts = sys.argv[1:]
sys.argv = [scripts[0]]
sys.path[0] = os.path.dirname(os.path.abspath(scripts[0]))  # what `python samples/x.py` puts first (not the cwd); PYTHONPATH follows
def stub(name, **attrs):
    m = types.ModuleType(name)
    m.__spec__ = importlib.machinery.ModuleSpec(name, None)
    m.__path__ = []
    m.__dict__.update(attrs)
    sys.modules[name] = m
# third-party / licensed pieces that are not installed here and are not on the hot path (transformers is imported first:
# it probes for librosa at import time and must see "not installed", not the stub)
import transformers
from transformers import HubertModel as _h, Wav2Vec2Model as _w, Wav2Vec2Processor as _p
stub("librosa")
stub("datasets")
for n in ("data_loader_mead", "data_loader_vocaset", "data_loader_biwi", "data_loader", "data_loader_mead_vqvae"):
    stub("datasets." + n, get_dataloaders=None)
stub("FLAME_PyTorch")
stub("FLAME_PyTorch.FLAME", FLAME=object)
stub("FLAME_PyTorch.config", get_config=None)
import fdm_b200.modules as M
REF = os.path.join(os.getcwd(), "")  # the reference checkout (the test runs this with cwd = the checkout)
for script in scripts:
    sys.path[0] = os.path.dirname(os.path.abspath(script))
    src = open(script).read()
    head = src.split("\ndef ", 1)[0]          # the import block: everything before the first function
    ns = {"__name__": "ref_script", "__file__": script}
    exec(compile(head, script, "exec"), ns)
    checked = []
    for name, base in (("FDM", M.FDMBase), ("GaussianDiffusion", M.GaussianDiffusionBase), ("VQAutoEncoder", M.VQAutoEncoderBase)):
        if name in ns:
            assert issubclass(ns[name], base), (script, name, ns[name].__module__)
            checked.append(name)
    for name in ("HubertModel", "Wav2Vec2Model"):
        if name in ns:
            assert hasattr(ns[name], "_engine"), (script, name)   # the CUDA-engine wrapper, not the plain HF class
            checked.append(name)
    for name in ("torch2mesh", "get_mesh"):
        if name in ns:
            assert REF in ns[name].__code__.co_filename, ns[name].__code__.co_filename
            checked.append(name)
    print("OK", script, ",".join(checked))
import models.lib.base_models as bm      # reference-only module of a package this repo also provides
assert bm.__file__.startswith(REF), bm.__file__
print("DONE")
'''


def test_reference_scripts_import_on_the_drop_in():
    scripts = [p for p in SCRIPTS if os.path.exists(os.path.join(REF, p))]
    assert len(scripts) >= 4
    env = {**os.environ, "PYTHONPATH": PKG, "PYTHONDONTWRITEBYTECODE": "1"}
    r = subprocess.run([sys.executable, "-c", RUNNER] + scripts, cwd=REF, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = r.stdout.strip().splitlines()
    assert lines[-1] == "DONE"
    ok = {l.split()[1]: l.split()[2] if len(l.split()) > 2 else "" for l in lines if l.startswith("OK ")}
    assert set(ok) == set(scripts)
    for p in ("samples/sample_diffusion_vocaset.py", "samples/sample_diffusion_biwi.py"):
        assert {"FDM", "GaussianDiffusion", "VQAutoEncoder"} <= set(ok[p].split(",")), ok[p]
    for p in ("samples/sample_diffusion_mead.py", "demo/demo_3d_mead.py"):  # the two that need utiles.flame_utils
        assert {"FDM", "GaussianDiffusion", "VQAutoEncoder", "torch2mesh"} <= set(ok[p].split(",")), ok[p]
