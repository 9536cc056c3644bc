"""Drives the UNMODIFIED reference learner (models/proof.py `Learner.incremental_train`) on synthetic features
(TEST INFRASTRUCTURE, never the product).

Used twice with the same seeds:
  * `oracle/gen_golden.py` (build container, CPU): the reference learner with the reference `Proof_Net` and
    `AdaptiveStateDistanceMatrix` -> `tests/golden/learner_2tasks.npz`;
  * `tests/test_gpu_learner_dropin.py` (reference tree = `$TEAM_REFERENCE_ROOT` or `oracle/_ref`): the same learner code with the two
    classes swapped for `team_b200.inc_net.Proof_Net` / `AdaptiveStateDistanceMatrix` - the two import lines
    `models/proof.py:8` and `:202` (INTEGRATION.md) - on `cuda:0`.
SURVEY App. D: CLIP is the identity on pre-computed 512-d features ("images" ARE feature rows), the tokenizer maps a
prompt string to a deterministic 512-d row, the DataManager serves class-clustered features with life-stage ids.
Dropout is switched off (p = 0) in both runs: the reference's Philox stream is not reproducible by construction.
"""
from __future__ import annotations

import contextlib
import io
import zlib

import numpy as np
import torch
import torch.nn as nn
from torch.utils.data import Dataset

from . import ref_loader

D = 512
STATES = (1, 3, 4)


def _row(seed: int) -> torch.Tensor:
    return torch.randn(D, generator=torch.Generator().manual_seed(seed))


class FakeData:
    """Class-clustered 512-d features with a life-stage id per sample; class c lives around centre_c, its stage s around
    centre_c + 0.5 stage_s."""

    def __init__(self, n_classes=4, n_train=24, n_test=8, seed=1234):
        g = torch.Generator().manual_seed(seed)
        self.labels = [f"insect_{c}" for c in range(n_classes)]
        self.centres = torch.randn(n_classes, D, generator=g)
        stage_dir = {s: torch.randn(D, generator=g) for s in STATES}
        self.x, self.y, self.s = {}, {}, {}
        for split, n in (("train", n_train), ("test", n_test)):
            xs, ys, ss = [], [], []
            for c in range(n_classes):
                st = torch.tensor(STATES)[torch.randint(0, len(STATES), (n,), generator=g)]
                if c % 2 == 1:
                    st = torch.where(st == 3, torch.tensor(4), st)        # odd classes: two life stages only
                x = self.centres[c] + 0.5 * torch.stack([stage_dir[int(v)] for v in st]) + 0.6 * torch.randn(n, D, generator=g)
                xs.append(x); ys.append(torch.full((n,), c)); ss.append(st)
            self.x[split] = torch.cat(xs).float()
            self.y[split] = torch.cat(ys).numpy().astype(np.int64)
            self.s[split] = torch.cat(ss).numpy().astype(np.int64)

    def text_row(self, prompt: str) -> torch.Tensor:
        """Tokenizer + (identity) text tower: the class centre of the label named in the prompt plus string-keyed noise."""
        v = 0.3 * _row(zlib.crc32(prompt.encode()))
        for c, name in enumerate(self.labels):
            if name in prompt:
                v = v + self.centres[c]
        return v


class _Plain(Dataset):
    def __init__(self, data, ids, targets):
        self.data, self.ids, self.targets = data, ids, targets

    def __len__(self):
        return len(self.ids)

    def __getitem__(self, i):
        split, j = self.ids[i]
        return i, self.data.x[split][j], int(self.targets[i])


class _Multi(_Plain):
    def __getitem__(self, i):
        split, j = self.ids[i]
        return i, {"image": self.data.x[split][j], "stage_id": int(self.data.s[split][j])}, int(self.targets[i])


class FakeDataManager:
    """The slice of utils/data_manager.py:DataManager the learner touches (models/proof.py:282-307,366-367,
    models/base.py:121-136,261-281): sample handles are (split, row) pairs stored as structured numpy rows."""

    def __init__(self, data: FakeData, increment=2):
        self.data, self.increment = data, increment
        self._class_to_label = list(data.labels)
        self._data_to_prompt = ["a photo of a {}."]

    def get_task_size(self, task):
        return self.increment

    def _select(self, indices, source):
        ids, tg = [], []
        for c in indices:
            rows = np.where(self.data.y[source] == c)[0]
            ids += [(0 if source == "train" else 1, int(r)) for r in rows]
            tg += [int(c)] * len(rows)
        return ids, tg

    def _build(self, cls, indices, source, appendent, ret_data):
        ids, tg = self._select(indices, source)
        if appendent is not None and len(appendent) != 0:
            ad, at = appendent
            ids += [tuple(int(v) for v in r) for r in np.asarray(ad).reshape(-1, 2)]
            tg += [int(v) for v in np.asarray(at).reshape(-1)]
        named = [("train" if a == 0 else "test", b) for a, b in ids]
        ds = cls(self.data, named, np.asarray(tg, dtype=np.int64))
        if ret_data:
            return np.asarray(ids, dtype=np.int64).reshape(-1, 2), np.asarray(tg, dtype=np.int64), ds
        return ds

    def get_dataset(self, indices, source, mode, appendent=None, ret_data=False, m_rate=None):
        return self._build(_Plain, indices, source, appendent, ret_data)

    def get_multimodal_dataset(self, indices, source, mode, appendent=None, ret_data=False):
        return self._build(_Multi, indices, source, appendent, ret_data)


def _reseed_by_name(module: nn.Module, seed: int):
    """Identical parameters in both runs whatever the order the two implementations construct their sub-modules in:
    every 2-d parameter is redrawn from a generator keyed by its state_dict name, with the scale of its initialiser."""
    with torch.no_grad():
        for name, p in module.named_parameters():
            if p.dim() < 2:
                continue
            g = torch.Generator().manual_seed(seed + zlib.crc32(name.encode()) % 100003)
            std = float(p.detach().float().std()) or 0.02
            p.copy_((torch.randn(p.shape, generator=g) * std).to(p.device))


def run(device: torch.device, swap: bool, tasks: int = 2, epochs: int = 2, seed: int = 7, team_mode: str = "f32",
        swap_herding: bool = False, keep_dropout: bool = False):
    """Returns a dict of numpy arrays: accuracy after every task, prototypes, per-state prototypes, distance factors
    and the trained parameters."""
    ref_loader.install_stubs()
    import sys
    data = FakeData()
    # the fake tokenizer needs the data (string -> row); open_clip stub of ref_loader returns texts unchanged
    oc = sys.modules["open_clip"]
    oc.get_tokenizer = lambda *a, **k: (lambda texts: torch.stack([data.text_row(t) for t in texts]))
    import models.base as ref_base          # noqa: E402  (reference modules)
    import models.proof as ref_proof        # noqa: E402
    import utils.state_distance as ref_sd   # noqa: E402
    import utils.inc_net as ref_net         # noqa: E402
    from torch.utils.data import DataLoader as _DL
    loader0 = lambda *a, **k: _DL(*a, **{**k, "num_workers": 0})
    ref_proof.num_workers = 0
    ref_base.DataLoader = loader0
    orig = (ref_proof.Proof_Net, ref_sd.AdaptiveStateDistanceMatrix)
    orig_herd = ref_base.BaseLearner._construct_exemplar
    if swap_herding:                        # third optional line of INTEGRATION.md: exemplar herding on the GPU
        from team_b200 import exemplars
        ref_base.BaseLearner._construct_exemplar = exemplars.construct_exemplar
    if swap:                                # the two lines of INTEGRATION.md
        from team_b200 import inc_net as team_net
        ref_proof.Proof_Net = team_net.Proof_Net
        ref_sd.AdaptiveStateDistanceMatrix = team_net.AdaptiveStateDistanceMatrix
    else:
        ref_proof.Proof_Net = ref_net.Proof_Net
    args = {"prefix": "harness", "dataset": "iiminsects202", "memory_size": 8, "memory_per_class": 2, "fixed_memory": False,
            "shuffle": False, "init_cls": 2, "increment": 2, "model_name": "proof", "convnet_type": "clip",
            "device": [device], "seed": seed, "tuned_epoch": epochs, "batch_size": 16, "weight_decay": 0.05,
            "init_lr": 0.004, "min_lr": 1e-8, "optimizer": "adam", "projection_type": "pure_mlp",
            "context_prompt_length_per_task": 10, "team_mode": team_mode}
    out = {}
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            torch.manual_seed(seed)
            learner = ref_proof.Learner(args)
            learner._network.to(device)
            prior = learner.state_distance.distance_factors.detach().clone().cpu()
            _reseed_by_name(learner._network, seed)
            _reseed_by_name(learner.state_distance, seed + 1)
            with torch.no_grad():          # the prior factors (utils/state_distance.py:22-37) are not an initialiser: keep them
                learner.state_distance.distance_factors.copy_(prior.to(device))
            dm = FakeDataManager(data)
            accs = []
            for t in range(tasks):
                torch.manual_seed(seed + 100 * (t + 1))
                for m in learner._network.modules():       # dropout off in both runs (see module docstring)
                    if isinstance(m, nn.Dropout) and not keep_dropout:
                        m.p = 0.0
                learner.incremental_train(dm)
                accs.append(float(learner._compute_accuracy(learner._network, learner.test_loader)))
                learner.after_task()
        net = learner._network
        out["accuracy"] = np.asarray(accs, dtype=np.float64)
        out["img_prototypes"] = net.img_prototypes.detach().float().cpu().numpy()
        for c, dct in sorted(net.img_prototypes_by_state.items()):
            for s, v in sorted(dct.items()):
                out[f"by_state/{int(c)}/{int(s)}"] = v.detach().float().cpu().numpy()
        out["distance_factors"] = learner.state_distance.distance_factors.detach().float().cpu().numpy()
        out["memory_targets"] = np.asarray(learner._targets_memory, dtype=np.int64)
        out["memory_data"] = np.asarray(learner._data_memory, dtype=np.int64)
        for name, p in net.named_parameters():
            if name.startswith(("projs_", "sel_attn", "context_prompts")) or name == "state_embedder.state_embeddings.weight":
                v = p.detach().float().cpu().numpy()
                out["param/" + name] = v[::16] if v.ndim == 2 and v.shape[0] == 512 else v
    finally:
        ref_proof.Proof_Net, ref_sd.AdaptiveStateDistanceMatrix = orig
        ref_base.BaseLearner._construct_exemplar = orig_herd
    return out
