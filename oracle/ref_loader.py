"""Import the *real* reference head (TEST / BASELINE INFRASTRUCTURE, never the product).

Users: ``oracle/gen_golden.py``, the CPU reference arm of ``bench.py`` (``--impl reference`` /
``cpu_baseline``) and the drop-in learner tests.  The reference is the unmodified tree of the original
TEAM project, found at ``$TEAM_REFERENCE_ROOT`` or at ``<repo>/oracle/_ref`` - a git-ignored copy that
``__graft_entry__.build()`` makes from ``$TEAM_REFERENCE_ROOT``, so that it travels with the working tree
to a machine that does not have it.  Three third-party modules the reference imports are absent from
the image and are stubbed (SURVEY.md App. D): ``timm`` (imported, never used:
utils/inc_net.py:6), ``matplotlib`` (utils/state_distance.py:5, models/proof.py:15)
and ``open_clip`` (utils/inc_net.py:17-19) -> a fake CLIP that is the identity on
pre-computed 512-d features, which is exactly the boundary of the hot path.
"""
from __future__ import annotations

import contextlib
import io
import os
import sys
import types

import torch
import torch.nn as nn
import torch.nn.functional as F

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _resolve_root() -> str:
    cands = [os.environ.get("TEAM_REFERENCE_ROOT"), os.path.join(_REPO, "oracle", "_ref")]
    for c in cands:
        if c and os.path.isdir(os.path.join(c, "utils")) and os.path.isdir(os.path.join(c, "models")):
            return c
    return cands[1]


REF_ROOT = _resolve_root()


class FakeCLIP(nn.Module):
    def __init__(self):
        super().__init__()
        self.logit_scale = nn.Parameter(torch.ones([]) * 2.6592600369327783)
        self.out_dim = 512

    def encode_image(self, x, normalize=False):
        return F.normalize(x, dim=-1) if normalize else x

    def encode_text(self, x, normalize=False):
        return F.normalize(x, dim=-1) if normalize else x


def available() -> bool:
    return os.path.isdir(os.path.join(REF_ROOT, "utils"))


def install_stubs():
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    for m in ("timm", "matplotlib", "matplotlib.pyplot"):
        if m not in sys.modules:
            sys.modules[m] = types.ModuleType(m)
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    oc = types.ModuleType("open_clip")
    oc.create_model_and_transforms = lambda *a, **k: (FakeCLIP(), None, None)
    oc.get_tokenizer = lambda *a, **k: (lambda texts: texts)
    sys.modules["open_clip"] = oc


def build_reference_net(params, img_prototypes=None, prompts_per_task=10):
    """Construct the reference Proof_Net through its own API for T tasks and overwrite
    its parameters with ``params`` (names = reference state_dict names)."""
    install_stubs()
    from utils.inc_net import Proof_Net  # noqa: E402  (reference module)
    T = 0
    while f"projs_img.{T}.MLP.0.weight" in params:
        T += 1
    args = {"convnet_type": "clip", "model_name": "proof", "device": [torch.device("cpu")],
            "projection_type": "pure_mlp", "context_prompt_length_per_task": prompts_per_task}
    with contextlib.redirect_stdout(io.StringIO()):
        net = Proof_Net(args, False)
        for t in range(T):
            net.update_prototype(2 * (t + 1))
            net.update_context_prompt()
            net.extend_task()
    sd = net.state_dict()
    missing = [k for k in params if k not in sd]
    assert not missing, f"synthetic params not in reference state_dict: {missing}"
    with torch.no_grad():
        for k, v in params.items():
            sd[k].copy_(v)
    if img_prototypes is not None:
        net.img_prototypes = img_prototypes.clone()
    net.freeze_projection_weight_new()
    net.eval()
    return net
