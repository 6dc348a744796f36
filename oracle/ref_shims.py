"""Import the UNMODIFIED reference (Yxxxb/LAVT-RS) on CPU -- TEST INFRASTRUCTURE ONLY.

The reference does not import as shipped (SURVEY.md section 8c): ``timm``, ``mmcv``, ``mmseg`` and its
``bert/`` directory are absent and ``MultiModalSwinTransformer3D.__init__`` reads an undefined global
``sr_ratio``.  Everything is fixed from OUTSIDE with stub modules; no reference file is edited or copied.
Used only where a checkout of the reference is present, in ``oracle/_ref`` (not tracked) or at
``$LAVT_REFERENCE_ROOT``: to pin ``oracle/lavt_oracle.py`` and to generate ``tests/golden/*``
(oracle/make_golden.py).  Without it the tests that import the reference skip.
"""
from __future__ import annotations

import os
import sys
import types

import torch
import torch.nn as nn

REFERENCE_ROOT = os.environ.get("LAVT_REFERENCE_ROOT", os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref"))


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "lib"))


_installed = False


def install_shims() -> None:
    global _installed
    if _installed:
        return
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    # transformers must be imported BEFORE a fake timm appears in sys.modules
    from transformers import BertConfig, BertModel

    layers = types.ModuleType("timm.models.layers")

    class DropPath(nn.Module):
        """Stochastic depth with timm semantics (identity in eval)."""

        def __init__(self, drop_prob=0.0):
            super().__init__()
            self.drop_prob = drop_prob

        def forward(self, x):
            if self.drop_prob == 0.0 or not self.training:
                return x
            keep = 1.0 - self.drop_prob
            mask = x.new_empty((x.shape[0],) + (1,) * (x.ndim - 1)).bernoulli_(keep)
            return x * mask / keep

    layers.DropPath = DropPath
    layers.trunc_normal_ = nn.init.trunc_normal_
    layers.to_2tuple = lambda v: v if isinstance(v, tuple) else (v, v)
    timm = types.ModuleType("timm")
    timm_models = types.ModuleType("timm.models")
    timm.models, timm_models.layers = timm_models, layers
    sys.modules.update({"timm": timm, "timm.models": timm_models, "timm.models.layers": layers})

    for name in ("mmcv", "mmcv.fileio", "mmcv.parallel", "mmcv.utils", "mmcv.runner", "mmseg", "mmseg.utils"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["mmcv.fileio"].FileClient = object
    sys.modules["mmcv.fileio"].load = lambda *a, **k: None
    sys.modules["mmcv.parallel"].is_module_wrapper = lambda m: False
    sys.modules["mmcv.utils"].mkdir_or_exist = lambda p: None
    sys.modules["mmcv.runner"].get_dist_info = lambda: (0, 1)
    sys.modules["mmseg.utils"].get_root_logger = lambda *a, **k: None

    class _OfflineBert(BertModel):
        @classmethod
        def from_pretrained(cls, name, *a, **k):  # no weights offline: seeded random BERT-base
            torch.manual_seed(1234)
            return cls(BertConfig())

    bert_pkg = types.ModuleType("bert")
    bert_mod = types.ModuleType("bert.modeling_bert")
    bert_mod.BertModel = _OfflineBert
    bert_pkg.modeling_bert = bert_mod
    sys.modules.update({"bert": bert_pkg, "bert.modeling_bert": bert_mod})

    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import lib.video_swin_transformer as vst  # noqa: E402  (reference module)

    vst.sr_ratio = [1]  # undefined-name workaround (lib/video_swin_transformer.py:726); value unused
    _installed = True


def reference_args(argv):
    install_shims()
    saved = sys.modules.pop("args", None)
    try:
        import importlib.util
        spec = importlib.util.spec_from_file_location("_lavt_ref_args", os.path.join(REFERENCE_ROOT, "args.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod.get_parser().parse_args(argv)
    finally:
        if saved is not None:
            sys.modules["args"] = saved


def build_reference(model: str = "lavt_video", swin_type: str = "base", window12: bool = False, extra=(), seed: int = 0):
    """Reference nn.Module (eval, CPU fp32) built exactly as train.py does (lib/segmentation.py builders)."""
    install_shims()
    from lib import segmentation  # reference module
    argv = ["--model", model, "--swin_type", swin_type, *extra]
    if window12:
        argv.append("--window12")
    args = reference_args(argv)
    torch.manual_seed(seed)
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        net = segmentation.__dict__[model](pretrained="", args=args)
    net.eval()  # the reference's backbone.train() override returns None, so do not chain
    return net, args


SEP_T_PWAM_FLAGS = ("--sep_t_pwam", "--conv3d_kernel_size_t", "3-3-3", "--conv3d_kernel_size_s", "1-1-1",
                    "--w_t3x3_s1x1", "--mm_t3x3_s1x1")      # the reference README's video configuration (README.md:185)


def build_reference_backbone_small(embed_dim=128, depths=(2, 2, 2, 2), num_heads=(4, 8, 16, 32), window=(8, 7, 7),
                                   mha=(1, 1, 1, 1), seed=0, extra=(), out_indices=(0, 1, 2, 3)):
    """A shallow reference video backbone + decoder for fast parity runs (same classes, fewer blocks)."""
    install_shims()
    from lib.video_swin_transformer import MultiModalSwinTransformer3D
    from lib.mask_predictor import SimpleDecoding
    args = reference_args(["--model", "lavt_video", *extra])
    torch.manual_seed(seed)
    bb = MultiModalSwinTransformer3D(patch_size=(1, 4, 4), embed_dim=embed_dim, depths=list(depths), num_heads=list(num_heads),
                                     window_size=window, drop_path_rate=0.0, patch_norm=True, out_indices=tuple(out_indices),
                                     use_checkpoint=False, num_heads_fusion=list(mha), fusion_drop=0.0, args=args)
    bb.init_weights()
    dec = SimpleDecoding(8 * embed_dim, args)
    bb.eval()
    dec.eval()
    return bb, dec, args


def build_reference_image_backbone_small(embed_dim=128, depths=(2, 2, 2, 2), num_heads=(4, 8, 16, 32), window=7,
                                         mha=(1, 1, 1, 1), seed=0, extra=()):
    """A shallow reference 2-D (image) backbone + decoder: lib/backbone.py MultiModalSwinTransformer."""
    install_shims()
    from lib.backbone import MultiModalSwinTransformer
    from lib.mask_predictor import SimpleDecoding
    args = reference_args(["--model", "lavt_one", *extra])
    torch.manual_seed(seed)
    bb = MultiModalSwinTransformer(embed_dim=embed_dim, depths=list(depths), num_heads=list(num_heads), window_size=window,
                                   ape=False, drop_path_rate=0.0, patch_norm=True, out_indices=(0, 1, 2, 3),
                                   use_checkpoint=False, num_heads_fusion=list(mha), fusion_drop=0.0, args=args)
    bb.init_weights()
    dec = SimpleDecoding(8 * embed_dim, args)
    bb.eval()
    dec.eval()
    return bb, dec, args
