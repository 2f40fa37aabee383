"""Drop-in installation into an UNMODIFIED checkout of zjukg/SNAG (SNAG_MMEA).

    python -m snag_b200.patch [--eval-precision fp32] [--link-precision fp32] [--train-precision fp32]
                              /path/to/SNAG_MMEA [main.py flags ...]
                                                      # runs main.py with the hot path replaced
or, from Python:
    import snag_b200.patch as sp; sp.patch()         # after SNAG_MMEA is on sys.path, before Runner is built

--eval-precision fp32 (patch(eval_precision="fp32")): Runner._test ranks the unrounded fp32 embeddings, as the reference
does, instead of their bf16 rounding (snag_b200.evaluate.EVAL_PRECISION). It governs Runner._test only.
--link-precision fp32 (patch(link_precision="fp32")): the two searches that choose training links — the
iterative-learning mining of SNAG.Iter_new_links and the seed induction of visual_pivot_induction (--unsup) — run on
the unrounded fp32 rows instead of their bf16 rounding (snag_b200.mining.LINK_PRECISION), so that the links are the
reference's.
--train-precision fp32 (patch(train_precision="fp32")): the icl_loss calls of the training step contract a split of the
unrounded fp32 rows instead of their bf16 rounding (snag_b200.loss.TRAIN_PRECISION), as the reference's fp32 training
does. It governs icl_loss only: ial_loss stays bf16 (SNAG never calls it).
The options come before the reference directory, in any order, and are consumed before main.py parses its arguments.

patch() assigns attributes — main.py, model/*.py and src/*.py stay byte-identical:
    model.SNAG_loss.icl_loss / ial_loss / CustomMultiLossLayer            -> snag_b200.loss
    model.SNAG.icl_loss / ial_loss / CustomMultiLossLayer                 (names already bound by `from .SNAG_loss import`)
    src.utils.pairwise_distances / csls_sim, model.SNAG.pairwise_distances -> snag_b200.evaluate
    model.SNAG.SNAG.add_noise_to_embeddings / get_mean_std / update_noise  -> snag_b200.noise
    model.SNAG.SNAG.Iter_new_links                                         -> snag_b200.mining
    model.SNAG_tools.MultiModalEncoder.forward                             -> snag_b200.noise.encoder_forward
    main.pairwise_distances / csls_sim, main.Runner._test                  -> snag_b200.evaluate / snag_b200.runner
There is no fallback: on a machine without a B200 the patched functions raise.
"""
from __future__ import annotations

import ast
import importlib
import os
import sys
import types

from . import evaluate, fusion, loss, mining, noise, runner, seeds


_ABSENT = object()
_SAVED: list = []          # (object, attribute name, original value) of everything patch() has rebound, oldest first


def unpatch() -> int:
    """Put back every attribute patch() replaced (newest first); returns how many were restored. Lets one process run
    the reference both ways (tests/test_reference_e2e_gpu.py compares the patched with the unpatched model)."""
    n = len(_SAVED)
    while _SAVED:
        obj, name, value = _SAVED.pop()
        if value is _ABSENT:
            delattr(obj, name)
        else:
            setattr(obj, name, value)
    return n


def patch(main_module: types.ModuleType | None = None, eval_precision: str | None = None,
          link_precision: str | None = None, train_precision: str | None = None) -> list[str]:
    """Install the replacements into whichever reference modules are importable; returns what was patched.
    eval_precision ("bf16" or "fp32", None = leave as is): what Runner._test evaluates with.
    link_precision (likewise): what Iter_new_links and visual_pivot_induction search with.
    train_precision (likewise): what the icl_loss calls of the training step contract."""
    done = []
    for precision in (eval_precision, link_precision):
        if precision is not None:
            evaluate._check_precision(precision)
    if train_precision is not None:
        loss._check_precision(train_precision)
        loss.TRAIN_PRECISION = train_precision
    if eval_precision is not None:
        evaluate.EVAL_PRECISION = eval_precision
    if link_precision is not None:
        mining.LINK_PRECISION = link_precision

    def _set(mod, name, value, label=None):
        # obj.__dict__ rather than getattr: a function stored on a class must be put back as the plain function
        own = getattr(mod, "__dict__", {})
        _SAVED.append((mod, name, own[name] if name in own else getattr(mod, name, _ABSENT)))
        setattr(mod, name, value)
        done.append(label or f"{mod.__name__}.{name}")

    try:
        ref_loss = importlib.import_module("model.SNAG_loss")
        for nm in ("icl_loss", "ial_loss", "CustomMultiLossLayer"):
            _set(ref_loss, nm, getattr(loss, nm))
    except ImportError:
        pass
    try:
        ref_utils = importlib.import_module("src.utils")
        _set(ref_utils, "pairwise_distances", evaluate.pairwise_distances)
        _set(ref_utils, "csls_sim", evaluate.csls_sim)
    except ImportError:
        pass
    try:
        ref_snag = importlib.import_module("model.SNAG")          # the module, not the class model/__init__ re-exports
        for nm in ("icl_loss", "ial_loss", "CustomMultiLossLayer"):
            _set(ref_snag, nm, getattr(loss, nm))
        _set(ref_snag, "pairwise_distances", evaluate.pairwise_distances)
        cls = ref_snag.SNAG
        _set(cls, "add_noise_to_embeddings", noise.add_noise_to_embeddings, "model.SNAG.SNAG.add_noise_to_embeddings")
        _set(cls, "get_mean_std", noise.get_mean_std, "model.SNAG.SNAG.get_mean_std")
        _set(cls, "update_noise", noise.update_noise, "model.SNAG.SNAG.update_noise")
        _set(cls, "Iter_new_links", mining.Iter_new_links, "model.SNAG.SNAG.Iter_new_links")
    except ImportError:
        pass
    try:
        ref_tools = importlib.import_module("model.SNAG_tools")
        _set(ref_tools.MultiModalEncoder, "forward", noise.encoder_forward, "model.SNAG_tools.MultiModalEncoder.forward")
        _set(ref_tools.MformerFusion, "forward", fusion.MformerFusion_forward, "model.SNAG_tools.MformerFusion.forward")
    except ImportError:
        pass
    try:
        ref_data = importlib.import_module("src.data")
        _set(ref_data, "visual_pivot_induction", seeds.visual_pivot_induction)
    except ImportError:
        pass
    main_mod = main_module or sys.modules.get("main")
    if main_mod is not None and hasattr(main_mod, "Runner"):
        _set(main_mod, "pairwise_distances", evaluate.pairwise_distances)
        _set(main_mod, "csls_sim", evaluate.csls_sim)
        _set(main_mod.Runner, "_test", runner._test, f"{main_mod.__name__}.Runner._test")
    return done


class Options(tuple):
    """(eval_precision or None, reference directory, main.py's arguments), with the link and training precisions (or
    None) as the attributes link_precision and train_precision: a three-tuple, so that callers which unpack parse_args'
    result keep working."""

    def __new__(cls, eval_precision: str | None, reference_dir: str, argv: list[str], link_precision: str | None = None,
                train_precision: str | None = None):
        self = super().__new__(cls, (eval_precision, reference_dir, argv))
        self.link_precision = link_precision
        self.train_precision = train_precision
        return self


_OPTIONS = ("--eval-precision", "--link-precision", "--train-precision")


def parse_args(argv: list[str]) -> Options:
    """Options from this module's command line: the options of snag_b200.patch (--eval-precision, --link-precision,
    --train-precision, in any order) precede the reference directory; everything after it belongs to main.py."""
    values = dict.fromkeys(_OPTIONS)
    i = 0
    while i < len(argv) and argv[i].split("=", 1)[0] in _OPTIONS:
        name = argv[i].split("=", 1)[0]
        if argv[i] == name:
            if i + 1 >= len(argv):
                raise SystemExit(f"{name} needs a value (bf16 or fp32)")
            value, i = argv[i + 1], i + 2
        else:
            value, i = argv[i].split("=", 1)[1], i + 1
        if value not in evaluate.PRECISIONS:
            raise SystemExit(f"{name} {value}: expected one of {evaluate.PRECISIONS}")
        values[name] = value
    if i >= len(argv):
        raise SystemExit(__doc__)
    return Options(values["--eval-precision"], argv[i], list(argv[i + 1:]), values["--link-precision"],
                   values["--train-precision"])


def run_main(reference_dir: str, argv: list[str], eval_precision: str | None = None,
             link_precision: str | None = None, train_precision: str | None = None) -> None:
    """Execute the reference's main.py (unchanged on disk) with the hot path patched in: the module body is executed
    first, the patch is applied (Runner now exists), then the `if __name__ == "__main__":` block runs."""
    reference_dir = os.path.abspath(reference_dir)
    path = os.path.join(reference_dir, "main.py")
    sys.path.insert(0, reference_dir)
    os.chdir(reference_dir)
    sys.argv = [path] + list(argv)
    patch(eval_precision=eval_precision, link_precision=link_precision,     # model.*, src.* before main.py binds them
          train_precision=train_precision)
    tree = ast.parse(open(path).read(), filename=path)
    body, tail = [], []
    for node in tree.body:
        is_main = (isinstance(node, ast.If) and isinstance(node.test, ast.Compare) and
                   isinstance(node.test.left, ast.Name) and node.test.left.id == "__name__")
        (tail if is_main else body).append(node)
    mod = types.ModuleType("__main__")
    mod.__file__ = path
    sys.modules["main"] = mod
    exec(compile(ast.Module(body=body, type_ignores=[]), path, "exec"), mod.__dict__)
    patch(mod)                                        # Runner._test and main's own bound names
    for node in tail:
        exec(compile(ast.Module(body=node.body, type_ignores=[]), path, "exec"), mod.__dict__)


if __name__ == "__main__":
    _opts = parse_args(sys.argv[1:])
    run_main(_opts[1], _opts[2], _opts[0], _opts.link_precision, _opts.train_precision)
