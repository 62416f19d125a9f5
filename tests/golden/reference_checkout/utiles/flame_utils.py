"""Stand-in for utiles/flame_utils.py of the original project: a module of the `utiles` package that this repository
does not provide (FLAME mesh helpers, off the sampling path). The scripts must find it in their own checkout."""
from FLAME_PyTorch.FLAME import FLAME  # noqa: F401
from FLAME_PyTorch.config import get_config  # noqa: F401


def torch2mesh(*args, **kwargs):
    raise NotImplementedError("stand-in")
