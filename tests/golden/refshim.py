"""Make the UNMODIFIED reference importable in the build container.

Used only by ``tests/golden/make_golden.py`` (golden-vector generation; runs in
a machine where FOD_REFERENCE_DIR points at a checkout of the reference project).

The reference (fewx/ + CenterNet2/ + the vendored detectron2 inside
detectron2.7z) needs third-party packages that are not installed here
(fvcore, iopath, yacs, termcolor, pycocotools, omegaconf, matplotlib, black,
nis, a non-shipped ``Visualizer`` package, and the prebuilt ``detectron2._C``).
None of them does arithmetic on the hot path, so they are replaced by
stand-ins:

  * a meta-path finder that fabricates empty "anything goes" modules for the
    missing top-level packages (attributes resolve to inert dummy callables);
  * real, minimal implementations of the three fvcore pieces the model code
    actually executes: ``Registry``, ``CfgNode`` and ``weight_init``.

The reference sources themselves are imported from where they lie
(FOD_REFERENCE_DIR, and the archive unpacked to a temp dir); nothing is copied
into the repository.
"""
from __future__ import annotations

import copy
import importlib.abc
import importlib.machinery
import io
import lzma
import os
import struct
import sys
import types

REFERENCE = os.environ.get("FOD_REFERENCE_DIR", "")     # checkout of the reference project (fewx/, configs/, detectron2.7z)

MISSING = {
    "fvcore", "iopath", "yacs", "termcolor", "pycocotools", "omegaconf", "matplotlib", "black", "nis",
    "demo_visualizer", "Visualizer", "lvis", "cityscapesscripts", "panopticapi", "shapely", "pydot",
    "mmcv", "mmdet", "caffe2", "onnx", "tensorboard", "fairscale", "timm", "skimage", "seaborn",
}
# present in the stdlib but unusable here (turtle needs tkinter): force a stand-in
FORCED = ("turtle",)


# --------------------------------------------------------------------------- #
# 7z unpacking (stdlib only).  The archive is one solid LZMA2 folder.
# --------------------------------------------------------------------------- #
def _u64(f):
    b = f.read(1)[0]
    mask, v = 0x80, 0
    for i in range(8):
        if not b & mask:
            return v | ((b & (mask - 1)) << (8 * i))
        v |= f.read(1)[0] << (8 * i)
        mask >>= 1
    return v


def _bits(f, n):
    out, b, m = [], 0, 0
    for _ in range(n):
        if not m:
            b, m = f.read(1)[0], 0x80
        out.append(bool(b & m))
        m >>= 1
    return out


def _defined(f, n):
    return [True] * n if f.read(1)[0] else _bits(f, n)


def _streams(f):
    s = {}
    while True:
        t = f.read(1)[0]
        if t == 0:
            return s
        if t == 6:
            s["pos"] = _u64(f)
            n = _u64(f)
            while True:
                t = f.read(1)[0]
                if t == 0:
                    break
                if t == 9:
                    s["psz"] = [_u64(f) for _ in range(n)]
                if t == 10:
                    [f.read(4) for d in _defined(f, n) if d]
        elif t == 7:
            assert f.read(1)[0] == 11 and _u64(f) == 1 and f.read(1)[0] == 0 and _u64(f) == 1
            fl = f.read(1)[0]
            s["cid"] = f.read(fl & 15)
            s["props"] = f.read(_u64(f)) if fl & 0x20 else b""
            assert f.read(1)[0] == 12
            s["usz"] = _u64(f)
            s["sub"] = [s["usz"]]
            t = f.read(1)[0]
            if t == 10:
                [f.read(4) for d in _defined(f, 1) if d]
                t = f.read(1)[0]
            assert t == 0
        elif t == 8:
            t = f.read(1)[0]
            n = 1
            if t == 13:
                n = _u64(f)
                t = f.read(1)[0]
            if t == 9:
                sz = [_u64(f) for _ in range(n - 1)]
                s["sub"] = sz + [s["usz"] - sum(sz)]
                t = f.read(1)[0]
            if t == 10:
                [f.read(4) for d in _defined(f, n) if d]
                t = f.read(1)[0]
            assert t == 0


def _unpack(raw, s):
    data = raw[32 + s["pos"]: 32 + s["pos"] + s["psz"][0]]
    if s["cid"] == b"\x21":
        p = s["props"][0]
        flt = {"id": lzma.FILTER_LZMA2, "dict_size": (2 | (p & 1)) << (p // 2 + 11)}
    else:
        flt = lzma._decode_filter_properties(lzma.FILTER_LZMA1, s["props"])
    return lzma.LZMADecompressor(lzma.FORMAT_RAW, filters=[flt]).decompress(data, s["usz"])


def unpack_7z(path: str, out: str) -> None:
    raw = open(path, "rb").read()
    assert raw[:6] == b"7z\xbc\xaf'\x1c"
    off, size = struct.unpack("<QQ", raw[12:28])
    f = io.BytesIO(raw[32 + off: 32 + off + size])
    if f.read(1)[0] == 0x17:
        f = io.BytesIO(_unpack(raw, _streams(f)))
        assert f.read(1)[0] == 1
    names, empty, s = [], None, None
    while True:
        t = f.read(1)[0]
        if t == 0:
            break
        if t == 4:
            s = _streams(f)
        if t == 5:
            n = _u64(f)
            while True:
                p = f.read(1)[0]
                if p == 0:
                    break
                blob = f.read(_u64(f))
                if p == 14:
                    empty = _bits(io.BytesIO(blob), n)
                if p == 17:
                    names = blob[1:].decode("utf-16-le").split("\0")[:-1]
    data, pos, sizes = _unpack(raw, s), 0, iter(s["sub"])
    empty = empty or [False] * len(names)
    for name, e in zip(names, empty):
        p = os.path.join(out, name)
        if e:
            if "." not in os.path.basename(p):
                os.makedirs(p, exist_ok=True)
            continue
        os.makedirs(os.path.dirname(p) or ".", exist_ok=True)
        n = next(sizes)
        with open(p, "wb") as fh:
            fh.write(data[pos:pos + n])
        pos += n


# --------------------------------------------------------------------------- #
# stand-ins
# --------------------------------------------------------------------------- #
class _DummyMeta(type):
    def __getattr__(cls, name):
        if name.startswith("__") and name.endswith("__"):
            raise AttributeError(name)
        return _Dummy()


class _DummyBase(metaclass=_DummyMeta):
    def __init__(self, *a, **k):
        pass


class _Dummy:
    """Inert object: callable, subscriptable, attribute-chainable, usable as a
    decorator and as a base class."""

    def __init__(self, *a, **k):
        pass

    def __call__(self, *a, **k):
        if len(a) == 1 and not k and (isinstance(a[0], type) or callable(a[0])):
            return a[0]          # decorator use
        return _Dummy()

    def __getattr__(self, name):
        if name.startswith("__") and name.endswith("__"):
            raise AttributeError(name)
        return _Dummy()

    def __getitem__(self, k):
        return _Dummy()

    def __iter__(self):
        return iter(())

    def __mro_entries__(self, bases):
        return (_DummyBase,)


class _AutoModule(types.ModuleType):
    def __getattr__(self, name):
        if name.startswith("__") and name.endswith("__"):
            raise AttributeError(name)
        return _Dummy()


class _Finder(importlib.abc.MetaPathFinder, importlib.abc.Loader):
    def find_spec(self, fullname, path, target=None):
        if fullname.split(".")[0] in MISSING or fullname == "detectron2._C":
            return importlib.machinery.ModuleSpec(fullname, self, is_package=True)
        return None

    def create_module(self, spec):
        m = _AutoModule(spec.name)
        m.__path__ = []
        m.__version__ = "99.0.0"
        return m

    def exec_module(self, module):
        pass


class Registry:
    """fvcore.common.registry.Registry semantics used by the reference."""

    def __init__(self, name):
        self._name, self._obj_map = name, {}

    def register(self, obj=None):
        if obj is None:
            def deco(o):
                self._obj_map[o.__name__] = o
                return o
            return deco
        self._obj_map[obj.__name__] = obj

    def get(self, name):
        return self._obj_map[name]

    def __contains__(self, name):
        return name in self._obj_map


class CfgNode(dict):
    """Minimal yacs/fvcore CfgNode: attribute access, yaml + _BASE_, merge_from_list."""

    def __init__(self, init=None, key_list=None, new_allowed=False):
        super().__init__()
        for k, v in (init or {}).items():
            self[k] = CfgNode(v) if isinstance(v, dict) and not isinstance(v, CfgNode) else v
        self.__dict__["_frozen"] = False

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError:
            raise AttributeError(k)

    def __setattr__(self, k, v):
        self[k] = v

    def clone(self):
        return copy.deepcopy(self)

    def freeze(self):
        pass

    def defrost(self):
        pass

    def is_frozen(self):
        return False

    def merge_from_other_cfg(self, other):
        for k, v in other.items():
            if isinstance(v, dict) and isinstance(self.get(k), dict):
                self[k].merge_from_other_cfg(v)
            else:
                self[k] = CfgNode(v) if isinstance(v, dict) and not isinstance(v, CfgNode) else v

    @classmethod
    def load_yaml_with_base(cls, filename, allow_unsafe=False):
        import yaml
        with open(filename) as f:
            cfg = yaml.safe_load(f)
        if "_BASE_" in cfg:
            base = cfg.pop("_BASE_")
            if not os.path.isabs(base):
                base = os.path.join(os.path.dirname(filename), base)
            b = cls.load_yaml_with_base(base)

            def merge(a, bb):
                for k, v in a.items():
                    if isinstance(v, dict) and isinstance(bb.get(k), dict):
                        merge(v, bb[k])
                    else:
                        bb[k] = v
            merge(cfg, b)
            return b
        return cfg

    def merge_from_file(self, filename, allow_unsafe=True):
        self.merge_from_other_cfg(CfgNode(self.load_yaml_with_base(filename)))

    def merge_from_list(self, lst):
        import ast
        for k, v in zip(lst[0::2], lst[1::2]):
            node = self
            parts = k.split(".")
            for p in parts[:-1]:
                node = node[p]
            if isinstance(v, str):
                try:
                    v = ast.literal_eval(v)
                except Exception:
                    pass
            node[parts[-1]] = v

    def dump(self, **kw):
        return repr(self)


def _weight_init_module():
    import torch.nn as nn
    m = types.ModuleType("fvcore.nn.weight_init")

    def c2_xavier_fill(module):
        nn.init.kaiming_uniform_(module.weight, a=1)
        if module.bias is not None:
            nn.init.constant_(module.bias, 0)

    def c2_msra_fill(module):
        nn.init.kaiming_normal_(module.weight, mode="fan_out", nonlinearity="relu")
        if module.bias is not None:
            nn.init.constant_(module.bias, 0)

    m.c2_xavier_fill, m.c2_msra_fill = c2_xavier_fill, c2_msra_fill
    return m


_INSTALLED = {}


def install(workdir: str = "/tmp/fod_refshim") -> str:
    """Unpack the vendored detectron2, install the stand-ins, extend sys.path.
    Returns the directory holding the unpacked ``detectron2`` package."""
    if "dir" in _INSTALLED:
        return _INSTALLED["dir"]
    d2dir = os.path.join(workdir, "detectron2")
    if not os.path.exists(os.path.join(d2dir, "modeling", "poolers.py")):
        unpack_7z(os.path.join(REFERENCE, "detectron2.7z"), d2dir)
    sys.meta_path.append(_Finder())
    for name in FORCED:
        sys.modules[name] = _AutoModule(name)
    # isinstance() targets must be real types
    om = _AutoModule("omegaconf")
    om.__path__ = []
    om.__version__ = "99.0.0"
    for cname in ("DictConfig", "ListConfig", "OmegaConf", "SCMode"):
        setattr(om, cname, type(cname, (), {}))
    sys.modules["omegaconf"] = om
    # local-file PathManager (iopath): the prototype-cache branch reads images through it
    fio = _AutoModule("iopath.common.file_io")
    fio.__path__ = []

    class PathHandler:
        pass

    class PathManager:
        def register_handler(self, *a, **k):
            pass

        def open(self, path, mode="r", **k):
            return open(path, mode)

        def isfile(self, path):
            return os.path.isfile(path)

        def exists(self, path):
            return os.path.exists(path)

        def get_local_path(self, path, **k):
            return path

        def mkdirs(self, path):
            os.makedirs(path, exist_ok=True)

    fio.PathHandler, fio.PathManager = PathHandler, PathManager
    fio.HTTPURLHandler = fio.OneDrivePathHandler = type("Handler", (PathHandler,), {})
    sys.modules["iopath.common.file_io"] = fio
    # real pieces of fvcore
    reg = types.ModuleType("fvcore.common.registry")
    reg.Registry = Registry
    cfgm = types.ModuleType("fvcore.common.config")
    cfgm.CfgNode = CfgNode
    sys.modules["fvcore.common.registry"] = reg
    sys.modules["fvcore.common.config"] = cfgm
    sys.modules["fvcore.nn.weight_init"] = _weight_init_module()
    # library drift since the reference's pins (Pillow < 10, numpy < 1.24)
    import PIL.Image
    if not hasattr(PIL.Image, "LINEAR"):
        PIL.Image.LINEAR = PIL.Image.BILINEAR
    import numpy as np
    for name, typ in (("bool", bool), ("int", int), ("float", float), ("object", object)):
        if name not in np.__dict__:
            setattr(np, name, typ)
    sys.path.insert(0, workdir)
    sys.path.insert(0, REFERENCE)
    _INSTALLED["dir"] = workdir
    return workdir
