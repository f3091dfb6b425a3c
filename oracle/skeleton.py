"""Module trees of the UNMODIFIED reference as test data (TEST INFRASTRUCTURE — see oracle/__init__.py).

accelerate() takes a module the reference built and reads only its structure: class names (and the class names of their
bases), constructor attributes, child modules, parameters and buffers.  `save` pickles such a tree with every class and
function defined by the reference replaced by a named stand-in, so `load` rebuilds it — same names, attributes,
parameters and buffers — without any reference source.  A stand-in has no arithmetic: the golden next to it stores what
the reference module computed (oracle/gen_golden_accelerate.py).

Parameters are stored by shape only (they are loaded zero-filled): the golden's module was given seeded weights
(`seed_`, or an oracle's seeded state_dict) before it computed, and the test seeds the loaded tree the same way.
"""
import copy
import pickle
import types

import torch

REFERENCE_PACKAGES = ("models", "options", "util", "data", "train")
_classes = {}


def _from_reference(obj):
    return (getattr(obj, "__module__", None) or "").split(".")[0] in REFERENCE_PACKAGES


def _refuse(what):
    def call(*args, **kwargs):
        raise RuntimeError("%s is a stand-in for a reference object: the golden holds what it computed" % what)
    return call


def standin_class(module, qualname, bases):
    key = (module, qualname)
    if key not in _classes:
        name = "%s.%s" % (module, qualname)
        _classes[key] = type(qualname.rsplit(".", 1)[-1], tuple(bases),
                             {"__module__": module, "__qualname__": qualname, "forward": _refuse(name)})
    return _classes[key]


def standin_function(module, qualname):
    f = _refuse("%s.%s" % (module, qualname))
    f.__name__ = f.__qualname__ = qualname.rsplit(".", 1)[-1]
    return f


class _Pickler(pickle.Pickler):
    def reducer_override(self, obj):
        if isinstance(obj, type) and _from_reference(obj):
            return standin_class, (obj.__module__, obj.__qualname__, obj.__bases__)
        if isinstance(obj, types.FunctionType) and _from_reference(obj):
            return standin_function, (obj.__module__, obj.__qualname__)
        return NotImplemented


_PICKLE = types.SimpleNamespace(Pickler=_Pickler, Unpickler=pickle.Unpickler, load=pickle.load, __name__="pickle")


def _modules_of(obj):
    if isinstance(obj, torch.nn.Module):
        yield from obj.modules()
    elif isinstance(obj, dict):
        for v in obj.values():
            yield from _modules_of(v)
    elif isinstance(obj, (list, tuple)):
        for v in obj:
            yield from _modules_of(v)


def save(obj, path):
    """torch.save of `obj` (any structure of tensors and modules) with the reference's classes as stand-ins and the
    modules' parameters (and tensors cached from them, such as a spectral-norm `weight`) reduced to their shapes."""
    obj = copy.deepcopy(obj)
    for m in _modules_of(obj):
        for k, v in list(vars(m).items()):
            if isinstance(v, torch.Tensor) and not isinstance(v, torch.nn.Parameter):
                setattr(m, k, v.detach().to("meta"))
        for k, p in m._parameters.items():
            if p is not None:
                m._parameters[k] = torch.nn.Parameter(p.detach().to("meta"), requires_grad=p.requires_grad)
    torch.save(obj, path, pickle_module=_PICKLE)


def load(path):
    obj = torch.load(path, weights_only=False)
    for m in _modules_of(obj):
        for k, v in list(vars(m).items()):
            if isinstance(v, torch.Tensor) and v.is_meta:
                setattr(m, k, torch.zeros(v.shape, dtype=v.dtype))
        for k, p in m._parameters.items():
            if p is not None and p.is_meta:
                m._parameters[k] = torch.nn.Parameter(torch.zeros(p.shape, dtype=p.dtype), requires_grad=p.requires_grad)
    return obj


@torch.no_grad()
def seed_(module, seed):
    """Seeded weights for every parameter, from its name and shape alone: N(0, 1/fan_in) for matrices and kernels,
    1 + N(0, 0.1^2) for normalisation gains, N(0, 0.1^2) for biases."""
    g = torch.Generator().manual_seed(seed)
    for name, p in module.named_parameters():
        v = torch.randn(p.shape, generator=g, dtype=torch.float64)
        if p.dim() > 1:
            v = v / (p[0].numel() ** 0.5)
        else:
            v = 0.1 * v + (1.0 if name.endswith("weight") else 0.0)
        p.copy_(v)
    return module
