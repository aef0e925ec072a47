"""TEST INFRASTRUCTURE ONLY -- compatibility shim that lets the *unmodified* reference
(`campx/` of a checkout of the original CampX, torch==0.3.1 / numpy==1.15 era code) execute on a
torch 2.x / numpy 2.x interpreter.  The checkout is not part of this repository; the environment
variable CAMPX_REFERENCE_ROOT names it (a directory holding `campx/` and `examples/`).

Nothing in `campx_b200/` imports this module.  It is used only by
`oracle/gen_golden.py` (fixture generation, which needs the checkout) and by the `not gpu` tests
that cross-check `oracle/campx_oracle.py` against the real reference when the checkout is given.

What it does (zero edits to reference files; see SURVEY.md section 8(c) / Appendix B):

1. injects stub modules for the reference's unavailable imports
   - `syft` with `_PointerTensor`, `_SNNTensor`           (campx/engine.py:26, used only by send/share :68-112)
   - `syft.core.frameworks.torch.utils.is_tensor`         (campx/engine.py:27)
   - `pycolab.protocols.logging.log`                      (campx/plot.py:25, used only by Plot.log :213-230)
2. numpy-2 patches needed by `campx/ascii_art.py:48`
   - `np.vstack(<generator>)`  -> `np.vstack(list(...))`
   - `np.fromstring(str, uint8)` (binary mode, removed in numpy 2) -> `np.frombuffer(bytes).copy()`
3. `torch.Tensor.set_(src)` with a dtype mismatch (legal in torch 0.3.1 where comparisons returned
   ByteTensor; an error today, hit at campx/engine.py:397, campx/rendering.py:209 and in user drapes
   after `gate * b` promotes to int64) first casts `src` to `self.dtype`.  Same-dtype calls fall
   through to the real `set_`, which preserves the storage-aliasing quirk Q1
   (campx/rendering.py:128,150).
"""
import os
import sys
import types

import numpy as np
import torch

REFERENCE_ROOT = os.path.abspath(os.environ["CAMPX_REFERENCE_ROOT"]) if os.environ.get("CAMPX_REFERENCE_ROOT") else ""

_installed = False


def reference_available(sub="campx"):
    """True when CAMPX_REFERENCE_ROOT names a checkout that has `sub` (campx/ or examples/)."""
    return bool(REFERENCE_ROOT) and os.path.isdir(os.path.join(REFERENCE_ROOT, sub))


def install(reference_root=REFERENCE_ROOT):
    """Install the shim (idempotent) and put the reference on sys.path."""
    global _installed
    if _installed:
        return
    if not os.path.isdir(os.path.join(reference_root, "campx")):
        raise RuntimeError("oracle/shim.py: %r holds no campx/; set CAMPX_REFERENCE_ROOT to a checkout of the "
                           "original CampX" % reference_root)
    _installed = True

    # --- 1. stub modules -------------------------------------------------------------------
    syft = types.ModuleType("syft")

    class _PointerTensor(object):
        pass

    class _SNNTensor(object):
        pass

    syft._PointerTensor = _PointerTensor
    syft._SNNTensor = _SNNTensor
    core = types.ModuleType("syft.core")
    frameworks = types.ModuleType("syft.core.frameworks")
    sy_torch = types.ModuleType("syft.core.frameworks.torch")
    utils = types.ModuleType("syft.core.frameworks.torch.utils")
    utils.is_tensor = torch.is_tensor
    syft.core = core
    core.frameworks = frameworks
    frameworks.torch = sy_torch
    sy_torch.utils = utils
    for name, mod in [("syft", syft), ("syft.core", core), ("syft.core.frameworks", frameworks),
                      ("syft.core.frameworks.torch", sy_torch),
                      ("syft.core.frameworks.torch.utils", utils)]:
        sys.modules.setdefault(name, mod)

    pycolab = types.ModuleType("pycolab")
    protocols = types.ModuleType("pycolab.protocols")
    logging = types.ModuleType("pycolab.protocols.logging")

    def log(the_plot, message):
        the_plot.setdefault("log_messages", []).append(message)

    logging.log = log
    pycolab.protocols = protocols
    protocols.logging = logging
    for name, mod in [("pycolab", pycolab), ("pycolab.protocols", protocols),
                      ("pycolab.protocols.logging", logging)]:
        sys.modules.setdefault(name, mod)

    # curses is imported (and unused) by the example files; make sure it cannot fail
    try:
        import curses  # noqa: F401
    except Exception:  # pragma: no cover
        sys.modules["curses"] = types.ModuleType("curses")

    # --- 2. numpy 2 patches -------------------------------------------------------------------
    _vstack = np.vstack

    def vstack(tup, *a, **k):
        if not isinstance(tup, (list, tuple)):
            tup = list(tup)
        return _vstack(tup, *a, **k)

    np.vstack = vstack

    _fromstring = np.fromstring

    def fromstring(string, dtype=float, count=-1, sep="", **k):
        if sep == "" and isinstance(string, str):
            return np.frombuffer(string.encode("latin-1"), dtype=dtype, count=count).copy()
        return _fromstring(string, dtype=dtype, count=count, sep=sep, **k)

    np.fromstring = fromstring

    # --- 3. Tensor.set_ dtype cast ---------------------------------------------------------------
    _set = torch.Tensor.set_

    def set_(self, *args, **kwargs):
        if len(args) == 1 and not kwargs and isinstance(args[0], torch.Tensor) \
                and args[0].dtype != self.dtype:
            return _set(self, args[0].to(self.dtype))
        return _set(self, *args, **kwargs)

    torch.Tensor.set_ = set_

    # --- 4. reference on sys.path ------------------------------------------------------------------
    for p in (reference_root, os.path.join(reference_root, "examples")):
        if p not in sys.path:
            sys.path.insert(0, p)


def load_notebook_world(notebook_filename, reference_root=REFERENCE_ROOT):
    """exec the game-defining code cells of a reference notebook and return its namespace.

    Cells that import/hook PySyft (Demo 3 cell 1) are reduced to their plain imports; cells that
    already *play* the game are skipped, so the caller gets the classes, GAME_ART and make_game().
    """
    import json
    install(reference_root)
    with open(os.path.join(reference_root, "examples", notebook_filename)) as f:
        nb = json.load(f)
    ns = {"__name__": "reference_notebook"}
    for cell in nb["cells"]:
        if cell["cell_type"] != "code":
            continue
        src = "".join(cell["source"])
        if not src.strip():
            continue
        # keep only cells that DEFINE things (imports, art, classes, make_game); cells that play the
        # game or just display values are skipped
        if not any(tok in src for tok in ("class ", "def ", "import ", "_ART")):
            continue
        lines = []
        syft_cell = "import syft" in src           # Demo 3 cell 1: keep its plain imports only
        for line in src.split("\n"):
            s = line.strip()
            if s.startswith("import syft") or s.startswith("from syft"):
                continue
            if syft_cell and not (s.startswith("import ") or s.startswith("from ")):
                continue
            # module-level "game = make_game()" / "game, board, ... = make_game()" lines play the game
            if not line.startswith(" ") and "= make_game()" in s:
                continue
            lines.append(line)
        exec(compile("\n".join(lines), notebook_filename, "exec"), ns)
    return ns
