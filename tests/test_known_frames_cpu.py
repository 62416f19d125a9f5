"""CPU: the known-frames boundary - fdm_known_args mirror, refusal of a library without the entry point, and the argument
checks of the sampling calls (they run before anything touches a device)."""
import os
import re
import subprocess
import tempfile

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HDR = os.path.join(ROOT, "include", "fdm_b200.h")


def test_known_args_mirror_the_header():
    import ctypes as C
    from fdm_b200 import lib
    hdr = re.sub(r"/\*.*?\*/", "", open(HDR).read(), flags=re.S)
    body = re.search(r"typedef struct fdm_known_args \{(.*?)\} fdm_known_args;", hdr, flags=re.S).group(1)
    width = {"int64_t": 8, "uint64_t": 8, "int32_t": 4, "float": 4}
    fields = []
    for decl in filter(None, (x.strip() for x in body.split(";"))):
        m = re.match(r"(const\s+)?(\w+)\s*(\*?)\s*(.*)", decl)
        for nm in m.group(4).split(","):
            nm = nm.strip()
            fields.append((nm.lstrip("* "), 8 if (m.group(3) or nm.startswith("*")) else width[m.group(2)]))
    assert [(n, C.sizeof(t)) for n, t in lib.KnownArgs._fields_] == fields
    with tempfile.TemporaryDirectory() as td:
        src, exe = os.path.join(td, "s.c"), os.path.join(td, "s")
        with open(src, "w") as f:
            f.write('#include <stdio.h>\n#include "%s"\nint main(void){printf("%%zu\\n", sizeof(fdm_known_args));return 0;}\n' % HDR)
        subprocess.check_call(["gcc", "-o", exe, src])
        assert int(subprocess.check_output([exe])) == C.sizeof(lib.KnownArgs)


def test_load_refuses_a_library_without_a_bound_symbol(monkeypatch):
    """A library built before an entry point existed must fail with a rebuild hint, not an AttributeError."""
    import ctypes as C
    from fdm_b200 import lib
    monkeypatch.setattr(lib, "_lib", None)
    monkeypatch.setitem(lib.EXPORTS, "fdm_not_in_this_library", (C.c_int, []))
    with pytest.raises(lib.FdmError, match="does not export fdm_not_in_this_library: rebuild"):
        lib.load()
    monkeypatch.delitem(lib.EXPORTS, "fdm_not_in_this_library")
    assert lib.load().fdm_known_frames is not None


@pytest.fixture(scope="module")
def meta_vocaset():
    import warnings
    warnings.simplefilter("ignore")
    os.environ["FDM_B200_RANDOM_AUDIO_ENCODER"] = "1"
    with torch.device("meta"):
        from models.fdm_vocaset import FDM
        from video_diffusion_pytorch.diffusion_BIWI_encoder_decoder import GaussianDiffusion
        return GaussianDiffusion(FDM(feature_dim=1024), timesteps=1000, loss_type="l2")


@pytest.mark.parametrize("case, match", [
    ("known_only", "give both or neither"),
    ("mask_only", "give both or neither"),
    ("known_dtype", "float32"),
    ("known_rows", r"shape \(2, 64, 64\).*\(3 or 1, 64, 64\)"),
    ("known_length", "shape"),
    ("mask_dtype", "bool"),
    ("mask_shape", r"3 sequences of 4 frames"),
    ("mask_rows", r"3 sequences of 4 frames"),
])
def test_known_arguments_are_checked(meta_vocaset, case, match):
    """VOCASET: fq = 16, zdim = 64; a call of 3 sequences x 4 frames."""
    diff = meta_vocaset
    shape = (3, 64, 64)
    known, mask = torch.zeros(shape), torch.zeros(3, 4, dtype=torch.bool)
    kw = {"known_only": dict(known=known), "mask_only": dict(known_mask=mask),
          "known_dtype": dict(known=known.double(), known_mask=mask),
          "known_rows": dict(known=known[:2], known_mask=mask),
          "known_length": dict(known=known[:, :48], known_mask=mask),
          "mask_dtype": dict(known=known, known_mask=mask.to(torch.uint8)),
          "mask_shape": dict(known=known, known_mask=mask[:, :3]),
          "mask_rows": dict(known=known, known_mask=mask[:2])}[case]
    audio, idh = torch.zeros(3, 16000), torch.eye(8)[:3]
    with pytest.raises(ValueError, match=match):
        diff.p_sample_loop(shape, audio, idh, steps=[1, 0], **kw)
    with pytest.raises(ValueError, match=match):
        diff.sample(audio, shape, idh, steps=[1, 0], **kw)
    with pytest.raises(ValueError, match=match):
        diff.ddim_sample(audio, shape, idh, 2, **kw)
