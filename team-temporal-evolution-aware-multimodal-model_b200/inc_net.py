"""Drop-in class surface of the reference's multimodal network for the TEAM learner
(SURVEY 8b): same class names, constructor arguments, parameter / ``state_dict`` names
(SURVEY App. B), method names, argument meaning and return conventions as

    utils/inc_net.py:342-617      Proof_Net
    convs/projections.py:7-87     Proj_Pure_MLP, MultiHeadAttention
    models/state_evolution.py     InsectLifecycleModel (state embedding + evolve_and_update)
    models/dynamic_modal_graph.py TemporalStateGCN / TemporalGCNBlock (parameter holders)
    utils/state_distance.py       AdaptiveStateDistanceMatrix
    convs/linears.py:31-61        CosineLinear

The modules below only HOLD parameters (so ``AdamW(net.parameters())``, ``requires_grad``
toggling, ``state_dict`` round trips and ``copy.deepcopy(net)`` keep working); every tensor
operation of the path is a call into ``libteam_b200.so`` through ``head`` / ``graph`` / ``ops``.
There is no torch fallback: on a machine without a B200 every method raises
``capi.TeamB200Error``.  The frozen CLIP towers are not part of the path: pass any object with
``encode_image / encode_text / logit_scale`` as ``convnet`` (the reference builds an open_clip
ViT-B/16, utils/inc_net.py:17-19).
"""
from __future__ import annotations

import copy
import math
from typing import Dict, List, Optional

import torch
import torch.nn as nn

from . import capi, feature_cache, graph, head, ops

FEATURE_DIM = capi.D


def _mode_of(args) -> int:
    m = (args or {}).get("team_mode", "f32") if isinstance(args, dict) else "f32"
    if m not in ("f32", "bf16"):
        raise ValueError(f"team_mode must be 'f32' or 'bf16', got {m!r}")
    return head.MODE_BF16 if m == "bf16" else head.MODE_F32


class Proj_Pure_MLP(nn.Module):
    """convs/projections.py:7-18: one Linear(512, 512) stored as ``MLP.0``."""

    def __init__(self, in_dim: int, hidden_dim: int, out_dim: int):
        super().__init__()
        if in_dim != FEATURE_DIM or out_dim != FEATURE_DIM:
            raise NotImplementedError("libteam_b200 is built for 512-d CLIP ViT-B/16 features")
        self.MLP = nn.Sequential(nn.Linear(in_dim, out_dim))

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return head.linear(x, self.MLP[0].weight, self.MLP[0].bias)


class MultiHeadAttention(nn.Module):
    """convs/projections.py:41-87 (n_head = 1).  Parameter holder: inside ``Proof_Net`` the block is
    evaluated by the fused kernels (shared rows projected once per step, fc folded into V)."""

    def __init__(self, n_head: int, d_model: int, d_k: int, d_v: int, dropout: float = 0.1):
        super().__init__()
        if n_head != 1 or d_model != FEATURE_DIM or d_k != FEATURE_DIM or d_v != FEATURE_DIM:
            raise NotImplementedError("sel_attn is single-head, 512-d (utils/inc_net.py:353)")
        self.n_head, self.d_k, self.d_v = n_head, d_k, d_v
        self.w_qs = nn.Linear(d_model, d_k, bias=False)
        self.w_ks = nn.Linear(d_model, d_k, bias=False)
        self.w_vs = nn.Linear(d_model, d_v, bias=False)
        nn.init.normal_(self.w_qs.weight, mean=0, std=math.sqrt(2.0 / (d_model + d_k)))
        nn.init.normal_(self.w_ks.weight, mean=0, std=math.sqrt(2.0 / (d_model + d_k)))
        nn.init.normal_(self.w_vs.weight, mean=0, std=math.sqrt(2.0 / (d_model + d_v)))
        self.layer_norm = nn.LayerNorm(d_model)
        self.fc = nn.Linear(d_v, d_model)
        nn.init.xavier_normal_(self.fc.weight)
        self.dropout = nn.Dropout(dropout)

    def forward(self, q, k, v):
        """Standalone call on arbitrary [B, L, 512] tokens (convs/projections.py:64-87): ``team_mha_fwd`` / ``team_mha_bwd``,
        differentiable.  Inside ``Proof_Net.forward_tri_modal`` the learner's eval / p = 0 path runs the factorised kernels
        instead.  Train mode with p > 0: both dropouts of the block (attention probabilities :28, fc output :62, :84) with the
        library's counter-based masks; seed = torch's seed, offset drawn from torch's CPU generator (so
        ``torch.manual_seed`` reproduces a run; the stream itself is not torch's)."""
        p, seed, offset = 0.0, 0, 0
        if self.training and self.dropout.p > 0:
            p = float(self.dropout.p)
            seed = torch.initial_seed()
            offset = int(torch.randint(0, 2 ** 62, (1,)).item()) * 2
        return head.mha(q, k, v, self.w_qs.weight, self.w_ks.weight, self.w_vs.weight, self.fc.weight, self.fc.bias,
                        self.layer_norm.weight, self.layer_norm.bias, mode=getattr(self, "team_mode", head.MODE_F32),
                        dropout_p=p, seed=seed, offset=offset)


class TemporalGCNBlock(nn.Module):
    """models/dynamic_modal_graph.py:268-292 - parameters only."""

    def __init__(self, hidden_dim: int):
        super().__init__()
        self.message_net = nn.Sequential(nn.Linear(hidden_dim * 2, hidden_dim), nn.LayerNorm(hidden_dim), nn.ReLU())
        self.update_net = nn.Sequential(nn.Linear(hidden_dim * 2, hidden_dim), nn.LayerNorm(hidden_dim), nn.ReLU())
        self.temporal_gate = nn.Sequential(nn.Linear(hidden_dim, 1), nn.Sigmoid())


class TemporalStateGCN(nn.Module):
    """models/dynamic_modal_graph.py:210-266; ``forward`` takes the reference's COO edge list."""

    def __init__(self, feature_dim: int, hidden_dim: int, num_layers: int = 2):
        super().__init__()
        self.feature_dim, self.hidden_dim = feature_dim, hidden_dim
        self.node_encoder = nn.Sequential(nn.Linear(feature_dim, hidden_dim), nn.LayerNorm(hidden_dim), nn.ReLU())
        self.time_encoder = nn.Sequential(nn.Linear(1, hidden_dim // 4), nn.LayerNorm(hidden_dim // 4), nn.ReLU())
        self.temporal_blocks = nn.ModuleList([TemporalGCNBlock(hidden_dim + hidden_dim // 4) for _ in range(num_layers)])
        self.output_proj = nn.Linear(hidden_dim + hidden_dim // 4, feature_dim)

    def forward(self, node_features, edge_index, edge_weights, time_steps):
        g = graph.graph_from_edge_list(node_features.shape[0], edge_index, edge_weights, time_steps)
        p = {f"g.{k}": v for k, v in self.named_parameters()}
        return graph.temporal_state_gcn(p, node_features, g, prefix="g")


class InsectLifecycleModel(nn.Module):
    """models/state_evolution.py:7-47, :239-367 - state embedding table + lifecycle graph evolution."""

    def __init__(self, feature_dim: int, hidden_dim: int, num_states: int = 10):
        super().__init__()
        self.feature_dim, self.hidden_dim, self.num_states = feature_dim, hidden_dim, num_states
        self.state_embeddings = nn.Embedding(num_states, feature_dim)
        self.state_type_names = {0: "egg", 1: "larva", 2: "pupa", 3: "nymph", 4: "adult", 5: "other"}
        self.class_lifecycle_types: Dict[int, str] = {}
        self.temporal_gcn = TemporalStateGCN(feature_dim=feature_dim, hidden_dim=hidden_dim)
        self.evolution_projector = nn.ModuleDict()
        self.evolution_detector = nn.Sequential(nn.Linear(feature_dim * 2, hidden_dim), nn.LayerNorm(hidden_dim),
                                                nn.ReLU(), nn.Linear(hidden_dim, 3), nn.Softmax(dim=1))

    def get_state_embeddings(self, state_ids):
        """models/state_evolution.py:45-47 on its own (differentiable).  Inside ``Proof_Net.encode_state`` /
        ``forward_tri_modal`` the lookup is fused: the 10-row table is projected once per step, then gathered."""
        return head.embedding(self.state_embeddings.weight, state_ids)

    def _detect_evolution_type(self, class_id, state_ids):
        t = graph.detect_evolution_type(list(state_ids))
        self.class_lifecycle_types[class_id] = t
        return t

    def evolve_and_update(self, class_prototypes_by_state, epoch=None, max_epoch=None):
        with torch.no_grad():
            return graph.evolve_and_update(dict(self.named_parameters()), class_prototypes_by_state,
                                           self.class_lifecycle_types, epoch, max_epoch, prefix="temporal_gcn")

    def integrate_with_state_distance(self, state_distance):
        return True          # the reference loops over an empty ModuleDict (SURVEY App. C-5)


class AdaptiveStateDistanceMatrix(nn.Module):
    """utils/state_distance.py:13-144."""

    def __init__(self, num_states: int = 10, feature_dim: int = 512, init_with_prior: bool = True,
                 update_interval: int = 10, decay_factor: float = 0.9):
        super().__init__()
        self.num_states, self.feature_dim = num_states, feature_dim
        init = graph.prior_distance_factors(num_states) if init_with_prior else torch.ones(num_states, num_states)
        self.distance_factors = nn.Parameter(init.clone())
        self.state_projector = nn.Sequential(nn.Linear(feature_dim, feature_dim // 2), nn.ReLU(),
                                             nn.Linear(feature_dim // 2, feature_dim // 4))
        self.update_history: List = []
        self.update_interval, self.decay_factor = update_interval, decay_factor
        self.update_counter = 0
        self.is_training = True

    def get_state_distance(self, state_i, state_j):
        return self.distance_factors[state_i, state_j]

    def get_distance_matrix(self):
        return graph.get_distance_matrix(self.distance_factors.data)

    def forward(self, state_features, state_ids):
        with torch.no_grad():
            cur, self.update_counter = graph.state_distance_forward(
                self.distance_factors.data, state_features, state_ids, self.update_counter,
                training=self.training and self.is_training, update_interval=self.update_interval,
                decay=self.decay_factor)
        return cur


class CosineLinear(nn.Module):
    """convs/linears.py:31-61 (nb_proxy = 1): ``{'logits': sigma * normalize(x) @ normalize(W).T}``."""

    def __init__(self, in_features: int, out_features: int, nb_proxy: int = 1, to_reduce: bool = False, sigma: bool = True):
        super().__init__()
        if nb_proxy != 1 or in_features != FEATURE_DIM:
            raise NotImplementedError("only nb_proxy = 1, 512-d CosineLinear is on the path")
        self.in_features, self.out_features = in_features, out_features
        self.weight = nn.Parameter(torch.empty(out_features, in_features))
        self.sigma = nn.Parameter(torch.ones(1)) if sigma else None
        stdv = 1.0 / math.sqrt(in_features)
        self.weight.data.uniform_(-stdv, stdv)

    def forward(self, input):
        with torch.no_grad():
            return {"logits": ops.cosine_logits(input, self.weight, self.sigma)}


class Proof_Net(nn.Module):
    """utils/inc_net.py:342-617.  ``args`` keys as in the reference (``device``, ``projection_type``,
    ``context_prompt_length_per_task``) plus the optional ``team_mode`` ('f32' parity mode | 'bf16')."""

    def __init__(self, args, pretrained, convnet=None, tokenizer=None, preprocess=None):
        super().__init__()
        self.args = args
        self.feature_dim = FEATURE_DIM
        self._device = args["device"][0]
        if convnet is None:
            try:
                import open_clip  # noqa: F401  (utils/inc_net.py:17-19)
            except Exception as e:
                raise NotImplementedError("no CLIP backbone: pass convnet=/tokenizer= (open_clip is not installed)") from e
            import open_clip
            convnet, _, preprocess = open_clip.create_model_and_transforms("ViT-B-16", pretrained="laion400m_e32")
            tokenizer = open_clip.get_tokenizer("ViT-B-16")
        self.convnet, self.tokenizer, self.preprocess = convnet, tokenizer, preprocess
        self.class_name = "SimpleClipNet"
        self.projs_img, self.projs_text, self.projs_state = nn.ModuleList(), nn.ModuleList(), nn.ModuleList()
        self.projtype = args.get("projection_type", "mlp")
        self.context_prompt_length_per_task = args.get("context_prompt_length_per_task", 3)
        self.sel_attn = MultiHeadAttention(1, FEATURE_DIM, FEATURE_DIM, FEATURE_DIM, dropout=0.1)
        self.img_prototypes = None
        self.context_prompts = nn.ParameterList()
        self.state_embedder = InsectLifecycleModel(feature_dim=FEATURE_DIM, hidden_dim=FEATURE_DIM // 2, num_states=10).to(self._device)
        self.state_evolution_graph = self.state_embedder          # same object, like the reference (:365)
        self.img_prototypes_by_state: Dict[int, Dict[int, torch.Tensor]] = {}
        self.evolution_embeddings = None
        self.team_mode = _mode_of(args)
        # frozen-tower feature cache (feature_cache.py; SURVEY 8f row 3): args["team_feature_cache"] = False switches it off
        self._towers = feature_cache.TowerCache(convnet) if args.get("team_feature_cache", True) else None

    def _img_feats(self, x):
        x = x.to(self._device)
        return self._towers.image(x) if self._towers is not None else self.convnet.encode_image(x)

    def _txt_feats(self, t):
        t = t.to(self._device) if torch.is_tensor(t) else t
        return self._towers.text(t) if self._towers is not None else self.convnet.encode_text(t)

    # ------------------------------------------------------------------ incremental bookkeeping
    def update_prototype(self, nb_classes):
        for c in range(nb_classes):
            self.img_prototypes_by_state.setdefault(c, {})
        if self.img_prototypes is not None:
            old = self.img_prototypes.to(self._device)
            self.img_prototypes = torch.cat([old.clone(), torch.zeros(nb_classes - len(old), FEATURE_DIM, device=self._device)])
        else:
            self.img_prototypes = torch.zeros(nb_classes, FEATURE_DIM, device=self._device)

    def update_context_prompt(self):
        for p in self.context_prompts:
            p.requires_grad = False
        self.context_prompts.append(nn.Parameter(torch.randn(self.context_prompt_length_per_task, FEATURE_DIM).to(self._device)))

    def get_context_prompts(self):
        return torch.cat([p for p in self.context_prompts], dim=0)

    def extend_item(self):
        if self.projtype == "pure_mlp":
            return Proj_Pure_MLP(FEATURE_DIM, FEATURE_DIM, FEATURE_DIM).to(self._device)
        raise NotImplementedError

    def extend_task(self):
        self.projs_img.append(self.extend_item())
        self.projs_text.append(self.extend_item())
        self.projs_state.append(self.extend_item())

    def freeze_projection_weight_new(self):
        n = len(self.projs_img)
        for lst in (self.projs_img, self.projs_text, self.projs_state):
            for i, proj in enumerate(lst):
                for p in proj.parameters():
                    p.requires_grad = (i == n - 1) if n > 1 else p.requires_grad
        for p in self.sel_attn.parameters():
            p.requires_grad = True
        for p in self.state_embedder.parameters():
            p.requires_grad = True

    # ------------------------------------------------------------------ the head
    def _pack(self) -> head.HeadParamPack:
        return head.HeadParamPack.from_state_dict(dict(self.named_parameters()))

    def _protos(self) -> torch.Tensor:
        if self.img_prototypes is None:
            raise capi.TeamB200Error("img_prototypes is unset: call update_prototype() first")
        self.img_prototypes = self.img_prototypes.to(self._device)
        return self.img_prototypes

    def extract_vector(self, x):
        """SimpleClipNet.extract_vector (utils/inc_net.py:324-325): the frozen tower's features (exemplar herding,
        models/base.py:213-238)."""
        return self.convnet.encode_image(x)

    def _dropout_active(self) -> bool:
        """The reference applies Dropout(0.1) to the attention probabilities and to the fc output in train mode
        (convs/projections.py:28,62,84; `.train()` at models/proof.py:398).  With dropout active, ``forward_tri_modal`` with
        per-sample text (the learner's form) runs the fused head with masks (``head.forward_tri_modal(dropout=...)``: one
        masked probability row per sample and table query, the same mask bits the token route draws); the class-text
        form and the PROOF fusion run the token-tensor route (encode_* with autograd -> the [B, L, 512] tokens the
        reference builds -> the stand-alone attention block with its dropout masks, team_mha_fwd / team_mha_bwd)."""
        return self.training and self.sel_attn.dropout.p > 0

    def encode_image(self, x, normalize: bool = False):
        feats = self._img_feats(x)
        return head.encode_grad(self._pack(), "image", feats, normalize=normalize, mode=self.team_mode)

    def encode_text(self, x, normalize: bool = False):
        feats = self._txt_feats(x)
        return head.encode_grad(self._pack(), "text", feats, normalize=normalize, mode=self.team_mode)

    def encode_state(self, state_ids, normalize: bool = False):
        return head.encode_grad(self._pack(), "state", state_ids.to(self._device), normalize=normalize, mode=self.team_mode)

    def encode_prototpyes(self, normalize: bool = False):        # (sic) utils/inc_net.py:417
        return head.encode_grad(self._pack(), "prototypes", self._protos(), normalize=normalize, mode=self.team_mode)

    def _wants_grad(self) -> bool:
        return torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())

    def forward_tri_modal(self, image, text, state_ids):
        """(image [B,512], text [B,1,512], state [B,512], proto [B,512], exp(logit_scale)); per-sample text
        (``len(text) == B``, the only form the learner uses, models/proof.py:421-425)."""
        img = self._img_feats(image)
        if isinstance(text, list):
            text = self.tokenizer(text)
        txt = self._txt_feats(text)
        if self._dropout_active():
            if txt.shape[0] != img.shape[0]:
                return self._tri_modal_tokens(img, txt, state_ids.to(self._device))
            # seed and offset drawn exactly as MultiHeadAttention.forward draws them: the same torch.manual_seed gives
            # the same masks (and the same consumption of torch's generator) on either route
            drop = (float(self.sel_attn.dropout.p), torch.initial_seed(), int(torch.randint(0, 2 ** 62, (1,)).item()) * 2)
            o = head.forward_tri_modal(self._pack(), img, txt, state_ids.to(self._device), self._protos(),
                                       mode=self.team_mode, dropout=drop)
            return o[0], o[1], o[2], o[3], self.convnet.logit_scale.exp()
        if txt.shape[0] != img.shape[0]:          # class texts shared by all samples: text output = mean over them
            if self._wants_grad():
                return self._tri_modal_tokens(img, txt, state_ids.to(self._device))
            with torch.no_grad():
                o = head.forward_tri_modal_class_text(self._pack(), img, txt, state_ids.to(self._device), self._protos(),
                                                      mode=self.team_mode)
            return o[0], o[1], o[2], o[3], self.convnet.logit_scale.exp()
        o = head.forward_tri_modal(self._pack(), img, txt, state_ids.to(self._device), self._protos(), mode=self.team_mode)
        return o[0], o[1], o[2], o[3], self.convnet.logit_scale.exp()

    def _tri_modal_tokens(self, img, txt, state_ids):
        """forward_tri_modal through the token tensor the reference builds (utils/inc_net.py:528-580): tokens = [image |
        text(s) | state | C prototypes | P prompts], sel_attn on them, slices / means as there.  Serves the class-text form
        with autograd (the fused forward-only kernel team_head_tri_classtext_fwd serves its no-grad case) and BOTH forms in
        train mode with dropout."""
        pack = self._pack()
        xi = head.encode_grad(pack, "image", img, normalize=True, mode=self.team_mode)
        xt = head.encode_grad(pack, "text", txt, normalize=True, mode=self.team_mode)
        xs = head.encode_grad(pack, "state", state_ids, normalize=True, mode=self.team_mode)
        xp = head.encode_grad(pack, "prototypes", self._protos(), normalize=True, mode=self.team_mode)
        B, Tn, Cn = xi.shape[0], xt.shape[0], xp.shape[0]
        per_sample = Tn == B                                 # utils/inc_net.py:544-547
        nt = 1 if per_sample else Tn
        text_tok = xt.view(B, 1, FEATURE_DIM) if per_sample else xt.view(1, Tn, FEATURE_DIM).expand(B, Tn, FEATURE_DIM)
        toks = torch.cat([xi.view(B, 1, FEATURE_DIM), text_tok,
                          xs.view(B, 1, FEATURE_DIM), xp.view(1, Cn, FEATURE_DIM).expand(B, Cn, FEATURE_DIM),
                          self.get_context_prompts().view(1, -1, FEATURE_DIM).expand(B, -1, FEATURE_DIM)], dim=1).contiguous()
        self.sel_attn.team_mode = self.team_mode
        f = self.sel_attn(toks, toks, toks)
        o_txt = f[:, 1:1 + nt]
        o_pro = f[:, 2 + nt:2 + nt + Cn]
        o_txt = head.mean_dim(o_txt.contiguous(), 1) if nt > 1 else o_txt
        o_pro = head.mean_dim(o_pro.contiguous(), 1) if Cn > 1 else o_pro
        return f[:, 0], o_txt, f[:, 1 + nt], o_pro, self.convnet.logit_scale.exp()

    def _proof_grad(self, xi, xt):
        """Differentiable PROOF fusion (utils/inc_net.py:447-462) on encoded rows: tokens = [image | Tn texts | C prototypes |
        P prompts], text / prototype outputs = means over the batch."""
        xp = self.encode_prototpyes(normalize=True)
        B, Tn, Cn = xi.shape[0], xt.shape[0], xp.shape[0]
        toks = torch.cat([xi.view(B, 1, FEATURE_DIM), xt.view(1, Tn, FEATURE_DIM).expand(B, Tn, FEATURE_DIM),
                          xp.view(1, Cn, FEATURE_DIM).expand(B, Cn, FEATURE_DIM),
                          self.get_context_prompts().view(1, -1, FEATURE_DIM).expand(B, -1, FEATURE_DIM)], dim=1).contiguous()
        self.sel_attn.team_mode = self.team_mode
        f = self.sel_attn(toks, toks, toks)
        o_txt = head.mean_dim(f[:, 1:1 + Tn].contiguous(), 0)
        o_pro = head.mean_dim(f[:, 1 + Tn:1 + Tn + Cn].contiguous(), 0)
        return f[:, 0], o_txt, self.convnet.logit_scale.exp(), o_pro

    def forward_for_classification(self, image, text_cls):
        """Learner.forward_for_classification (models/proof.py:519-536): cosine logits of the projected image
        against the projected class texts, no scale.  Returns (logits [B,C], argmax [B])."""
        img = self._img_feats(image)
        if isinstance(text_cls, list):
            text_cls = self.tokenizer(text_cls)
        tc = self._txt_feats(text_cls)
        with torch.no_grad():
            xi = head.encode(self._pack(), "image", img, normalize=True, mode=self.team_mode)
            ti = head.encode(self._pack(), "text", tc, normalize=True, mode=self.team_mode)
            return ops.cosine_logits(xi, ti, want_argmax=True)

    def forward(self, image, text):
        """PROOF fusion (utils/inc_net.py:436-463): (image [B,512], text [Tn,512] batch mean, exp(logit_scale),
        proto [C,512] batch mean).  Without autograd: one fused forward (team_head_proof_fwd); with autograd (a trainable
        parameter under enable_grad): the same function through the differentiable encode + standalone attention ops."""
        img = self._img_feats(image)
        if isinstance(text, list):
            text = self.tokenizer(text)
        txt = self._txt_feats(text)
        if self._wants_grad() or self._dropout_active():
            pack = self._pack()
            return self._proof_grad(head.encode_grad(pack, "image", img, normalize=True, mode=self.team_mode),
                                    head.encode_grad(pack, "text", txt, normalize=True, mode=self.team_mode))
        with torch.no_grad():
            o = head.forward_proof(self._pack(), img, txt, self._protos(), mode=self.team_mode)
        return o[0], o[1], self.convnet.logit_scale.exp(), o[2]

    def forward_transformer(self, image_features, text_features, transformer=False):
        """utils/inc_net.py:465-492: the same fusion on rows the caller already encoded (encode_image /
        encode_text with normalize=True); transformer=False returns the inputs and the encoded prototypes."""
        if not transformer:
            return image_features, text_features, self.convnet.logit_scale.exp(), self.encode_prototpyes(normalize=True)
        if self._wants_grad() or self._dropout_active():
            return self._proof_grad(image_features.to(self._device), text_features.to(self._device))
        with torch.no_grad():
            o = head.forward_proof(self._pack(), image_features.to(self._device), text_features.to(self._device),
                                   self._protos(), inputs_encoded=True, mode=self.team_mode)
        return o[0], o[1], self.convnet.logit_scale.exp(), o[2]

    # ------------------------------------------------------------------ prototypes / graph
    def evolve_state_prototypes(self):
        if not self.img_prototypes_by_state:
            return None
        with torch.no_grad():
            emb = graph.evolve_state_prototypes(dict(self.named_parameters()), self._protos(), self.img_prototypes_by_state,
                                                self.state_embedder.class_lifecycle_types)
        self.evolution_embeddings = emb
        return emb

    def _sync_class_prototypes(self):
        if self.img_prototypes is None:
            return
        graph.sync_class_prototypes(self._protos(), self.img_prototypes_by_state)


class SimpleVitNet(nn.Module):
    """utils/inc_net.py:261-296 for the SimpleCIL learner: cosine classifier over class-mean prototypes."""

    def __init__(self, args, pretrained, convnet=None):
        super().__init__()
        self.args, self.convnet, self.fc, self.feature_dim = args, convnet, None, FEATURE_DIM

    def update_fc(self, nb_classes, nextperiod_initialization=None):
        dev = self.args["device"][0]
        fc = CosineLinear(FEATURE_DIM, nb_classes).to(dev)
        if self.fc is not None:
            nb_output = self.fc.out_features
            weight = copy.deepcopy(self.fc.weight.data)
            fc.sigma.data = self.fc.sigma.data
            tail = nextperiod_initialization if nextperiod_initialization is not None else \
                torch.zeros(nb_classes - nb_output, FEATURE_DIM, device=dev)
            fc.weight = nn.Parameter(torch.cat([weight, tail]))
        self.fc = fc

    def extract_vector(self, x):
        return self.convnet(x) if callable(self.convnet) else x

    def forward(self, x):
        return self.fc(self.extract_vector(x))

    def replace_fc(self, features: torch.Tensor, labels: torch.Tensor, class_ids=None):
        """simplecil.Learner.replace_fc math (models/simplecil.py:48-55): fc.weight[c] = mean of the
        (un-normalised) features of class c, for the classes present in ``class_ids`` (default: all)."""
        n_cls = self.fc.out_features
        sums, counts = ops.keyed_sums(features, labels, num_classes=n_cls)
        if class_ids is not None:
            keep = torch.zeros(n_cls, dtype=torch.bool, device=counts.device)
            keep[torch.as_tensor(list(class_ids), device=counts.device)] = True
            counts = torch.where(keep, counts, torch.zeros_like(counts))
        ops.keyed_means(sums, counts, out=self.fc.weight.data)
        return self.fc.weight.data
