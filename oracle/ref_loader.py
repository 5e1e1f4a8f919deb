"""Execute the real reference sources (build container only).

TEST INFRASTRUCTURE -- see oracle/__init__.py.  Only ``oracle/gen_golden.py`` calls it: the tests compare
against what it recorded under ``tests/golden/``.  Where the reference tree (``CUNET_REFERENCE_ROOT``) is absent,
everything here raises ``ReferenceUnavailable``.

Recipe (SURVEY.md Appendix C): ``models/cu_net.py`` is python-2 source; two tokens stop it
from running under python 3:
  * ``models/cu_net.py:286``  ``print '...'`` statement  -> function-call form
  * ``models/cu_net.py:94``   ``adapter_out_num / 2``    -> floor division
Both are substituted in memory; nothing is copied into this repository.

``pylib/HumanAug.py``, ``pylib/Evaluation.py`` and ``pylib/HumanPts.py`` (validation path and target heat maps) are
python-2 sources as well: one ``print '...'`` statement each in a ``__main__`` block (HumanAug.py:277,
HumanPts.py:336), tab/space mixed indentation in HumanPts.py:43-44 (python 2 counts a tab as eight columns) and the
implicit relative ``import HumanAug`` of Evaluation.py:4.  ``load_reference_pylib`` executes them with those three
things patched in memory.  None of the executed functions relies on python-2 integer division.
"""
import re
import contextlib
import io
import os
import sys
import types

REF_ROOT = os.environ.get("CUNET_REFERENCE_ROOT", "/root/reference")


class ReferenceUnavailable(RuntimeError):
    pass


def available():
    return os.path.isfile(os.path.join(REF_ROOT, "models", "cu_net.py"))


def load_reference_cu_net():
    """Return a module object holding the reference's models/cu_net.py namespace."""
    if not available():
        raise ReferenceUnavailable("reference tree not present at %s" % REF_ROOT)
    path = os.path.join(REF_ROOT, "models", "cu_net.py")
    with open(path, "r") as f:
        src = f.read()
    a = "print 'order is larger than the layer number.'"
    b = "adapter_out_num = adapter_out_num / 2"
    assert a in src and b in src, "reference source changed; update the substitutions"
    src = src.replace(a, "print('order is larger than the layer number.')")
    src = src.replace(b, "adapter_out_num = adapter_out_num // 2")
    mod = types.ModuleType("reference_cu_net")
    mod.__file__ = path
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        exec(compile(src, path, "exec"), mod.__dict__)
    return mod


def create_reference_net(class_num, layer_num, order, loss_num,
                         neck_size=4, growth_rate=32, init_chan_num=128):
    """create_cu_net of the reference (models/cu_net.py:362-368), stdout suppressed."""
    mod = load_reference_cu_net()
    with contextlib.redirect_stdout(io.StringIO()):
        net = mod.create_cu_net(neck_size=neck_size, growth_rate=growth_rate,
                                init_chan_num=init_chan_num, class_num=class_num,
                                layer_num=layer_num, order=order, loss_num=loss_num)
    return net


def load_reference_util():
    """The REAL ``TrainHistory`` class (utils/util.py:8-46) and ``adjust_lr`` function (utils/util.py:106-119) in one
    namespace: only their text is executed (the module imports PIL / visdom-era helpers that are irrelevant here)."""
    if not available():
        raise ReferenceUnavailable("reference tree not present at %s" % REF_ROOT)
    from collections import OrderedDict
    with open(os.path.join(REF_ROOT, "utils", "util.py"), "r") as f:
        src = f.read()
    ns = {"OrderedDict": OrderedDict}
    exec(src[src.index("class TrainHistory():"):src.index("class TrainHistoryFace():")], ns)
    exec(src[src.index("def adjust_lr(opt, optimizer, epoch):"):src.index("def AdjustLR")], ns)
    return ns


def load_reference_quantize(bits_w, bits_i=8, bits_g=8, exp_dir="/tmp/cunet_ref_exp"):
    """Import the reference's utils/quantize.py (parses argv at import, quantize.py:8-11)."""
    if not available():
        raise ReferenceUnavailable("reference tree not present at %s" % REF_ROOT)
    os.makedirs(exp_dir, exist_ok=True)
    saved_argv = list(sys.argv)
    saved_path = list(sys.path)
    saved_mods = {k: sys.modules.get(k) for k in list(sys.modules)
                  if k == "utils" or k.startswith("utils.") or k == "options"
                  or k.startswith("options.")}
    for k in saved_mods:
        sys.modules.pop(k, None)
    try:
        sys.argv = ["x", "--exp_id", "q", "--exp_dir", exp_dir, "--bits_w", str(bits_w),
                    "--bits_i", str(bits_i), "--bits_g", str(bits_g)]
        sys.path.insert(0, REF_ROOT)
        import importlib
        with contextlib.redirect_stdout(io.StringIO()):
            q = importlib.import_module("utils.quantize")
        return q
    finally:
        sys.argv = saved_argv
        sys.path[:] = saved_path
        for k in list(sys.modules):
            if k == "utils" or k.startswith("utils.") or k == "options" or k.startswith("options."):
                sys.modules.pop(k, None)
        for k, v in saved_mods.items():
            if v is not None:
                sys.modules[k] = v


def load_reference_binop():
    """The reference's ``BinOp`` class (models/cu_net_prev_version.py:17-92) as an executable class object.

    The module itself cannot be imported (``torch._thnn`` / ``type2backend`` at :8 are gone), and the class body
    relies on torch-0.1.12 semantics in two ways.  Both are patched IN MEMORY on the text of lines 17-92 only, with
    exactly the substitutions the reference's own authors made when they ported the sibling class QuanOp from
    utils/quantize_prev_version.py (0.1.12) to utils/quantize.py (0.4) -- `diff` of those two files:
      * reductions kept their dimension: ``.mean(1)`` -> ``.mean(1, True)``, ``.norm(1, 3)`` -> ``.norm(1, 3, True)``,
        ``.sum(k)`` -> ``.sum(k, True)``                                   (quantize.py:113,130-131,162-163,169-170)
      * method calls with ``out=``: ``x.clamp(a, b, out=x)`` / ``x.sign().mul(m, out=x)`` -> assignment of the result
                                                                            (quantize.py:133-134)
    Nothing is copied into this repository."""
    if not available():
        raise ReferenceUnavailable("reference tree not present at %s" % REF_ROOT)
    path = os.path.join(REF_ROOT, "models", "cu_net_prev_version.py")
    with open(path, "r") as f:
        lines = f.read().split("\n")
    assert lines[16].startswith("class BinOp") and lines[93].startswith("class _SharedAllocation"), \
        "reference source changed; update the line range"
    src = "\n".join(lines[16:92])
    subs = [
        (".data.mean(1).", ".data.mean(1, True)."),
        (".norm(1, 3)", ".norm(1, 3, True)"),
        (".sum(2).sum(1).div(n)", ".sum(2, True).sum(1, True).div(n)"),
        ("m_add.sum(3)", "m_add.sum(3, True)"),
        ("self.target_modules[index].data.clamp(-1.0, 1.0,\n                    out = self.target_modules[index].data)",
         "self.target_modules[index].data = self.target_modules[index].data.clamp(-1.0, 1.0)"),
        ("self.target_modules[index].data.sign()\\\n                    .mul(m.expand(s), out=self.target_modules[index].data)",
         "self.target_modules[index].data = self.target_modules[index].data.sign().mul(m.expand(s))"),
    ]
    for a, b in subs:
        assert a in src, "reference BinOp source changed; update the substitution %r" % a
        src = src.replace(a, b)
    import numpy
    import torch
    ns = {"torch": torch, "nn": torch.nn, "numpy": numpy}
    exec(compile(src, path + ":17-92", "exec"), ns)
    return ns["BinOp"]


def load_reference_pylib():
    """Namespaces of the reference's pylib/HumanAug.py, pylib/Evaluation.py, pylib/HumanPts.py as module objects."""
    if not available():
        raise ReferenceUnavailable("reference tree not present at %s" % REF_ROOT)
    import warnings
    mods = {}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for name in ("HumanAug", "Evaluation", "HumanPts"):
            path = os.path.join(REF_ROOT, "pylib", name + ".py")
            with open(path, "r") as f:
                src = f.read().expandtabs(8)
            src = re.sub(r"^(\s*)print\s+'([^']*)'\s*$", r"\1print('\2')", src, flags=re.M)
            mod = types.ModuleType("reference_pylib_" + name)
            mod.__file__ = path
            # stand-ins during the exec only: the implicit relative import of Evaluation.py:4, and matplotlib.path
            # (HumanPts.py:6, used by a polygon helper that is not on the path) which this image does not have
            stubs = {}
            if name == "Evaluation":
                stubs["HumanAug"] = mods["HumanAug"]
            if name == "HumanPts" and "matplotlib" not in sys.modules:
                mpl, mpath = types.ModuleType("matplotlib"), types.ModuleType("matplotlib.path")
                mpath.Path = object
                mpl.path = mpath
                stubs.update({"matplotlib": mpl, "matplotlib.path": mpath})
            saved = {k: sys.modules.get(k) for k in stubs}
            sys.modules.update(stubs)
            try:
                with contextlib.redirect_stdout(io.StringIO()):
                    exec(compile(src, path, "exec"), mod.__dict__)
            finally:
                for k, v in saved.items():
                    if v is None:
                        sys.modules.pop(k, None)
                    else:
                        sys.modules[k] = v
            mods[name] = mod
    return mods
