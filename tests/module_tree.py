"""Module trees as data: ``record`` stores ``nn.Module`` trees built by another package (class names,
instance attributes, evaluated properties, parameters and buffers) as one ``.npz`` payload, and
``rebuild`` turns it back into modules without importing that package.

Classes outside torch come back as stand-ins with the recorded class name and ``__module__``, derived
from the nearest torch class of the original (``nn.Sequential``, ``nn.Linear``, ``nn.Module`` ...), so
that iteration, indexing, ``state_dict`` and ``_apply`` behave as on the original.  torch's own
classes come back as themselves.  A recorded property returns its value as recorded, with the module's
own parameters and buffers looked up at access time (so ``_apply`` / ``load_state_dict`` are seen).
Callables outside torch (constructors passed as arguments) come back as empty classes of the same
name; ``functools.partial`` keeps its arguments.

Integer and boolean tensors (masks, orders, permutations) and small floating-point ones are stored
exactly.  Floating-point tensors of more than ``EXACT_FLOATS`` elements (initial weights) are stored
by shape and dtype and come back filled from a fixed seed: what they are made of is the module's
structure, not its values, and random weights would make the payload large.
"""

from __future__ import annotations

import functools
import importlib
import json

import numpy as np
import torch
import torch.nn as nn

_MODULE_INTERNALS = frozenset(vars(nn.Module()))
EXACT_FLOATS = 64


def _is_torch(module_name: str) -> bool:
    return module_name.split(".")[0] == "torch"


def _torch_base(cls: type) -> type:
    return next(c for c in cls.__mro__ if _is_torch(c.__module__))


def _path(obj) -> dict:  # noqa: ANN001
    return {"module": obj.__module__, "name": obj.__qualname__}


def _own_name(m: nn.Module, t: torch.Tensor) -> str | None:
    for name, v in [*m._parameters.items(), *m._buffers.items()]:
        if v is t:
            return name
    return None


class _Recorder:
    def __init__(self) -> None:
        self.tensors: dict[str, np.ndarray] = {}
        self.seeded: dict[str, dict] = {}
        self.keys: dict[int, str] = {}

    def tensor(self, t: torch.Tensor) -> str:
        if id(t) not in self.keys:
            key = f"t{len(self.keys)}"
            self.keys[id(t)] = key
            if t.is_floating_point() and t.numel() > EXACT_FLOATS:
                self.seeded[key] = {"shape": list(t.shape), "dtype": str(t.dtype).removeprefix("torch.")}
            else:
                self.tensors[key] = t.detach().cpu().numpy()
        return self.keys[id(t)]

    def value(self, v, owner: nn.Module):  # noqa: ANN001, ANN201
        if v is None or isinstance(v, (bool, int, float, str)):
            return v
        if isinstance(v, torch.Tensor):
            name = _own_name(owner, v)
            return {"own": name} if name is not None else {"tensor": self.tensor(v)}
        if isinstance(v, (list, tuple)):
            return {"list" if isinstance(v, list) else "tuple": [self.value(x, owner) for x in v]}
        if isinstance(v, dict):
            return {"dict": {str(k): self.value(x, owner) for k, x in v.items()}}
        if isinstance(v, functools.partial):
            return {"partial": self.value(v.func, owner), "args": self.value(v.args, owner),
                    "keywords": self.value(v.keywords, owner)}  # fmt: skip
        if isinstance(v, type) or callable(v) and hasattr(v, "__qualname__"):
            return {"callable": _path(v)}
        raise TypeError(f"cannot record a value of type {type(v).__name__}")

    def module(self, m: nn.Module) -> dict:
        cls = type(m)
        props = {}
        for c in reversed(cls.__mro__):
            if _is_torch(c.__module__):
                continue
            for k, p in vars(c).items():
                if isinstance(p, property):
                    v = getattr(m, k)
                    if not isinstance(v, nn.Module):  # e.g. a lazy `.inv`: rebuilt by whoever needs it
                        props[k] = self.value(v, m)
        return {
            "class": _path(cls),
            "base": _path(_torch_base(cls)),
            "training": m.training,
            "attrs": {k: self.value(v, m) for k, v in vars(m).items() if k not in _MODULE_INTERNALS},
            "props": props,
            "params": [[k, None if p is None else self.tensor(p), None if p is None else p.requires_grad]
                       for k, p in m._parameters.items()],
            "buffers": [[k, None if b is None else self.tensor(b), k not in m._non_persistent_buffers_set]
                        for k, b in m._buffers.items()],
            "children": [[k, None if c is None else self.module(c)] for k, c in m._modules.items()],
        }  # fmt: skip


def record(modules: dict[str, nn.Module]) -> dict[str, np.ndarray]:
    """The ``np.savez`` payload of ``modules`` (name -> root module).  Tensors shared between modules
    are stored once and come back shared."""
    r = _Recorder()
    trees = {name: r.module(m) for name, m in modules.items()}
    return {"trees": np.array(json.dumps(trees)), "seeded": np.array(json.dumps(r.seeded)), **r.tensors}


def _import(path: dict):  # noqa: ANN202
    obj = importlib.import_module(path["module"])
    for part in path["name"].split("."):
        obj = getattr(obj, part)
    return obj


class _Rebuilder:
    def __init__(self, payload) -> None:  # noqa: ANN001
        self.payload = payload
        self.seeded = json.loads(str(payload["seeded"]))
        self.tensors: dict[str, torch.Tensor] = {}
        self.params: dict[str, nn.Parameter] = {}
        self.classes: dict[tuple, type] = {}

    def tensor(self, key: str) -> torch.Tensor:
        if key not in self.tensors:
            if key in self.seeded:
                spec, g = self.seeded[key], torch.Generator().manual_seed(int(key[1:]))
                t = torch.empty(spec["shape"], dtype=getattr(torch, spec["dtype"])).uniform_(-0.1, 0.1, generator=g)
            else:
                t = torch.from_numpy(np.array(self.payload[key]))
            self.tensors[key] = t
        return self.tensors[key]

    def param(self, key: str, requires_grad: bool) -> nn.Parameter:
        if key not in self.params:
            self.params[key] = nn.Parameter(self.tensor(key), requires_grad=requires_grad)
        return self.params[key]

    def stand_in(self, path: dict, bases: tuple, props: tuple = ()) -> type:
        key = (path["module"], path["name"], bases, props)
        if key not in self.classes:
            ns = {"__module__": path["module"], "__qualname__": path["name"]}
            for k in props:
                ns[k] = property(lambda self, k=k: _decode(self._recorded_props[k], self, self._rebuilder))
            self.classes[key] = type(path["name"].rsplit(".", 1)[-1], bases, ns)
        return self.classes[key]

    def callable(self, path: dict):  # noqa: ANN201
        return _import(path) if _is_torch(path["module"]) else self.stand_in(path, ())

    def module(self, node: dict) -> nn.Module:
        if _is_torch(node["class"]["module"]):
            cls = _import(node["class"])
        else:
            cls = self.stand_in(node["class"], (_import(node["base"]),), tuple(sorted(node["props"])))
        m = cls.__new__(cls)
        nn.Module.__init__(m)
        m.training = node["training"]
        for k, key, requires_grad in node["params"]:
            m._parameters[k] = None if key is None else self.param(key, requires_grad)
        for k, key, persistent in node["buffers"]:
            m._buffers[k] = None if key is None else self.tensor(key)
            if not persistent:
                m._non_persistent_buffers_set.add(k)
        for k, child in node["children"]:
            m._modules[k] = None if child is None else self.module(child)
        for k, v in node["attrs"].items():
            m.__dict__[k] = _decode(v, m, self)
        if node["props"]:
            m.__dict__["_recorded_props"], m.__dict__["_rebuilder"] = node["props"], self
        return m


def _decode(v, owner: nn.Module, rb: _Rebuilder):  # noqa: ANN001, ANN202
    if not isinstance(v, dict):
        return v
    (kind, x), *_ = v.items()
    if kind == "own":
        return owner._parameters[x] if x in owner._parameters else owner._buffers[x]
    if kind == "tensor":
        return rb.tensor(x)
    if kind in ("list", "tuple"):
        out = [_decode(y, owner, rb) for y in x]
        return out if kind == "list" else tuple(out)
    if kind == "dict":
        return {k: _decode(y, owner, rb) for k, y in x.items()}
    if kind == "partial":
        return functools.partial(_decode(x, owner, rb), *_decode(v["args"], owner, rb), **_decode(v["keywords"], owner, rb))
    if kind == "callable":
        return rb.callable(x)
    raise ValueError(f"unknown recorded value {kind!r}")


def rebuild(payload) -> dict[str, nn.Module]:  # noqa: ANN001
    """Fresh modules (fresh tensors) from a ``record`` payload (e.g. an opened ``.npz``)."""
    rb = _Rebuilder(payload)
    return {name: rb.module(node) for name, node in json.loads(str(payload["trees"])).items()}
