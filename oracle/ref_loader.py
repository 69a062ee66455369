"""TEST INFRASTRUCTURE ONLY -- loads the UNMODIFIED reference (eladb3/SViT) from /root/reference.

Used only by tests/golden/make_golden.py (run in the build container, where the
reference tree is mounted read-only) to produce the committed golden fixtures.
Nothing in svit_b200/ imports this file. /root/reference does not exist on the GPU box.

Recipe (SURVEY.md 8c): the reference package cannot be imported as-is here because
fvcore / iopath / av are not installed.  We pre-seed empty package shells whose
__path__ points into the reference tree (so slowfast/__init__.py side effects are
skipped but sub-module imports resolve to the original files) and shim three tiny
things: fvcore.common.registry.Registry, slowfast.utils.logging.get_logger and the
two config readers of slowfast/utils/misc.py:406-423.
"""
import importlib
import logging
import os
import sys
import types

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _find_root():
    """SVIT_REFERENCE_ROOT, then /root/reference (build container), then <repo>/baseline/_ref (a driver-side install of
    the unmodified reference package, git-ignored) -- the first that holds slowfast/models."""
    cands = [os.environ.get("SVIT_REFERENCE_ROOT"), "/root/reference", os.path.join(_REPO, "baseline", "_ref")]
    for c in cands:
        if c and os.path.isdir(os.path.join(c, "slowfast", "models")):
            return c
    return cands[1]


REF_ROOT = _find_root()


def available() -> bool:
    return os.path.isdir(os.path.join(REF_ROOT, "slowfast", "models"))


class _Registry(dict):
    def __init__(self, name):
        super().__init__()
        self._name = name

    def register(self, obj=None):
        if obj is None:
            def deco(o):
                self[o.__name__] = o
                return o
            return deco
        self[obj.__name__] = obj
        return obj


def _shell(name, path):
    m = types.ModuleType(name)
    m.__path__ = [path]
    sys.modules[name] = m
    return m


def load():
    """Returns a namespace with the reference's attention / model / box_ops modules."""
    if not available():
        raise RuntimeError(f"reference tree not found at {REF_ROOT}")
    if "slowfast.models.video_model_builder" not in sys.modules:
        sf = os.path.join(REF_ROOT, "slowfast")
        _shell("slowfast", sf)
        _shell("slowfast.models", os.path.join(sf, "models"))
        _shell("slowfast.utils", os.path.join(sf, "utils"))
        # fvcore.common.registry.Registry shim
        fv = types.ModuleType("fvcore"); fvc = types.ModuleType("fvcore.common")
        fvr = types.ModuleType("fvcore.common.registry"); fvr.Registry = _Registry
        sys.modules.update({"fvcore": fv, "fvcore.common": fvc, "fvcore.common.registry": fvr})
        # slowfast.utils.logging shim
        lg = types.ModuleType("slowfast.utils.logging"); lg.get_logger = logging.getLogger
        sys.modules["slowfast.utils.logging"] = lg
        sys.modules["slowfast.utils"].logging = lg
        # slowfast.utils.misc shim (only the two readers the model ctor needs, misc.py:406-423)
        misc = types.ModuleType("slowfast.utils.misc")

        def get_num_classes(cfg):
            return cfg.MODEL.NUM_CLASSES

        def get_lambdas_dict(cfg):
            d = {"loss_ce": 1, "boxes_l1_loss": 5 * cfg.SVIT.LAMBDA_NODES,
                 "boxes_bce_loss": cfg.SVIT.LAMBDA_NODES, "boxes_giou_loss": 2 * cfg.SVIT.LAMBDA_NODES,
                 "loss_contact_state": cfg.SVIT.LAMBDA_EDGES}
            if cfg.TRAIN.FORWARD_VIDEO_FRAMES:
                d["video_image_boxes_l1_loss"] = cfg.SVIT.LAMBDA_CON
            return d
        misc.get_num_classes = get_num_classes
        misc.get_lambdas_dict = get_lambdas_dict
        sys.modules["slowfast.utils.misc"] = misc
        sys.modules["slowfast.utils"].misc = misc
    ns = types.SimpleNamespace()
    ns.attention = importlib.import_module("slowfast.models.attention")
    ns.builder = importlib.import_module("slowfast.models.video_model_builder")
    ns.stem = importlib.import_module("slowfast.models.stem_helper")
    ns.common = importlib.import_module("slowfast.models.common")
    ns.box_ops = importlib.import_module("slowfast.utils.box_ops")
    return ns
