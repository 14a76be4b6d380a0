#!/usr/bin/env python
"""TEST / BENCH INFRASTRUCTURE -- stage the reference's own Python files of the hot path into the git-ignored
``oracle/_ref/py/`` so that bench.py's ``frames.reference_stack`` leg and the golden-vector generator
(tests/golden/make_reference_golden.py) can run the REFERENCE classes (``MSDeformAttnFunction``, ``MSDeformAttn``,
``DeformableTransformerEncoderLayer`` / ``DecoderLayer`` / ``DeformableReidHead``, the CondInst head of ddetrs.py)
unchanged.  Tests never need it: what they compare against is stored under tests/golden/.

    python -m oracle.refstage            # copies; no-op (exit 0) when no reference checkout is present

Same status as ``oracle/_ref/libmsda_refcuda.so`` (the reference's CUDA kernels compiled where they lie): the copies are
byte-identical to the reference, are never committed, and nothing under ``uninext_b200/`` imports them. What is copied,
verbatim:

    ops/functions/{__init__,ms_deform_attn_func}.py       (a1/a2: the autograd boundary)
    ops/modules/{__init__,ms_deform_attn}.py              (a9)
    deformable_transformer.py, deformable_transformer_dino.py   (a10/a11/a12 + reference-point helpers, f-3)
    ../ddetrs.py                                          (f-4: dynamic_mask_with_coords, aligned_bilinear, ...)

What is WRITTEN here (not copied) so those files import without the rest of UNINEXT: stub modules for imports that are
off the hot path -- ``util/misc.py`` (``inverse_sigmoid`` only), ``vlfusion.py`` / ``fuse_helper.py`` (the
vision-language fusion classes, never instantiated), the few detectron2 names ddetrs.py imports at module level.
"""
from __future__ import annotations

import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DEST = os.path.join(HERE, "_ref", "py")
PKG = os.path.join(DEST, "uninext_ref")
SRC = "/root/reference/projects/UNINEXT/uninext/models/deformable_detr"

COPIES = [
    "ops/functions/__init__.py",
    "ops/functions/ms_deform_attn_func.py",
    "ops/modules/__init__.py",
    "ops/modules/ms_deform_attn.py",
    "deformable_transformer.py",
    "deformable_transformer_dino.py",
    "../ddetrs.py",                                        # CondInst dynamic mask head (f-4)
]

STUBS = {
    "__init__.py": "",
    "util/__init__.py": "",
    "util/misc.py": (
        '"""Stub written by oracle/refstage.py: the helpers the staged files import from util/misc.py."""\n'
        "import torch\n\n\n"
        "def inverse_sigmoid(x, eps=1e-5):\n"
        "    x = x.clamp(min=0, max=1)\n"
        "    return torch.log(x.clamp(min=eps) / (1 - x).clamp(min=eps))\n\n\n"
        "class NestedTensor:\n    pass\n\n\n"
        "def interpolate(*a, **k):\n    return torch.nn.functional.interpolate(*a, **k)\n\n\n"
        "def nested_tensor_from_tensor_list(*a, **k):\n    raise NotImplementedError\n"),
    "models/conv_with_kaiming_uniform.py": (
        '"""Stub written by oracle/refstage.py (mask-feature convolutions are off the hot path)."""\n\n\n'
        "def conv_with_kaiming_uniform(*a, **k):\n    raise NotImplementedError\n"),
    "../detectron2/__init__.py": '"""Stub package written by oracle/refstage.py: names ddetrs.py imports at module level."""\n',
    "../detectron2/structures.py": "class Instances:\n    pass\n",
    "../detectron2/data/__init__.py": "",
    "../detectron2/data/datasets/__init__.py": "",
    "../detectron2/data/datasets/builtin_meta.py": "COCO_CATEGORIES = []\n",
    "models/__init__.py": "",
    "models/deformable_detr/__init__.py": "",
    "models/deformable_detr/ops/__init__.py": "",
    "models/deformable_detr/vlfusion.py": (
        '"""Stub written by oracle/refstage.py (vision-language fusion is off the hot path)."""\n'
        "import torch\n\n\n"
        "class VLFuse(torch.nn.Module):\n    pass\n\n\n"
        "class BertEncoderLayer(torch.nn.Module):\n    pass\n"),
    "models/deformable_detr/fuse_helper.py": (
        '"""Stub written by oracle/refstage.py (vision-language fusion is off the hot path)."""\n'
        "import torch\n\n\n"
        "class BiMultiHeadAttention(torch.nn.Module):\n    pass\n"),
}


def staged() -> bool:
    return all(os.path.exists(os.path.join(PKG, "models/deformable_detr", c)) for c in COPIES)


def stage(force: bool = False) -> bool:
    """Returns True when oracle/_ref/py is usable afterwards."""
    if not os.path.isdir(SRC):
        return staged()
    if staged() and not force:
        fresh = all(os.path.getmtime(os.path.join(PKG, "models/deformable_detr", c)) >= os.path.getmtime(os.path.join(SRC, c))
                    for c in COPIES)
        if fresh:
            return True
    for rel, text in STUBS.items():
        path = os.path.join(PKG, rel)
        os.makedirs(os.path.dirname(path), exist_ok=True)
        with open(path, "w") as fh:
            fh.write(text)
    for rel in COPIES:
        dst = os.path.join(PKG, "models/deformable_detr", rel)
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        shutil.copyfile(os.path.join(SRC, rel), dst)
    return True


def import_reference():
    """-> (func_module, attn_module, transformer_module, dino_module): the staged reference files, imported on top of
    the drop-in (``import MultiScaleDeformableAttention`` resolves to uninext_b200/dropin)."""
    import importlib
    import warnings

    import uninext_b200
    uninext_b200.install_dropin()
    if DEST not in sys.path:
        sys.path.insert(0, DEST)
    base = "uninext_ref.models.deformable_detr"
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")        # torch.cuda.amp.custom_fwd deprecation in the reference decorators
        return tuple(importlib.import_module(f"{base}.{m}") for m in
                     ("ops.functions.ms_deform_attn_func", "ops.modules.ms_deform_attn", "deformable_transformer",
                      "deformable_transformer_dino"))


def import_ddetrs():
    """The staged uninext/models/ddetrs.py (CondInst mask branch) with its off-path imports stubbed."""
    import importlib
    import warnings
    import_reference()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return importlib.import_module("uninext_ref.models.ddetrs")


if __name__ == "__main__":
    ok = stage(force="--force" in sys.argv)
    print(f"oracle/_ref/py {'ready' if ok else 'NOT staged (no reference checkout)'}")
