"""Import shim for running the UNMODIFIED reference (the copy build() staged under oracle/_ref, else the checkout)
(TEST INFRASTRUCTURE — see oracle/__init__.py).  Optional third-party packages the reference
imports at module level but never touches on the palette / unet_mha / resnet / NLayerD arithmetic
path are replaced by MagicMock modules (SURVEY.md top table).  Used by the golden generators and by the tests
that drive the reference's own training code.
"""
import importlib.abc
import importlib.machinery
import os
import sys
from unittest import mock

_STAGED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")
REFERENCE_ROOT = _STAGED if os.path.isdir(_STAGED) else os.environ.get("JG_REFERENCE_ROOT", "")


def available():
    """True where the reference's own code can run: the copy build() staged under oracle/_ref, or the checkout."""
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "models", "base_model.py"))


MISSING = [
    "thop", "torchviz", "piq", "lpips", "positional_encodings", "clip", "timm", "bitsandbytes", "imgaug",
    "dominate", "visdom", "aim", "diffusers", "peft", "segment_anything", "mobile_sam", "torchinfo", "addict",
    "onnx", "DISTS_pytorch", "vision_aided_loss", "ouisdom", "tifffile", "wget", "xformers", "ftfy", "iopath",
    "pytorchvideo", "open_clip", "kornia", "onnxruntime", "cv2", "torchvision",
]


class _MockLoader(importlib.abc.Loader):
    def create_module(self, spec):
        m = mock.MagicMock(name=spec.name)
        m.__name__ = spec.name
        m.__path__ = []
        m.__spec__ = spec
        m.__loader__ = self
        return m

    def exec_module(self, module):
        pass


class _StubFinder(importlib.abc.MetaPathFinder):
    def __init__(self, names):
        self.names = set(names)

    def find_spec(self, fullname, path, target=None):
        root = fullname.split(".")[0]
        if root in self.names:
            return importlib.machinery.ModuleSpec(fullname, _MockLoader(), is_package=True)
        return None


def _importable(name):
    try:
        __import__(name)
        return True
    except Exception:
        return False


def install():
    """Make `import models.modules...` resolve to the reference, stubbing what is not installed."""
    sys.dont_write_bytecode = True
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    missing = [m for m in MISSING if not _importable(m)]
    sys.meta_path.insert(0, _StubFinder(missing))
    return missing
