"""Drop-in `nn.Module` surface of the Macaron ODE-ViT (reference: models/macaron.py), backed by
libodevit.so's MACARON field.

    PatchEmbed :10-35        MLP :38-52        MultiheadSelfAttention :55-71
    ParallelAttentionMLP :78-123   ViT_ODEFunc :125-150   ViTMacaron :157-352

Same constructor kwargs, call signatures, `state_dict` keys and output dict as the reference.  The
vector field  x3 = x + 1/2 rs FFN(LN1 x) -> + rs MHA(LN2 .) -> + 1/2 rs FFN(LN3 .),  f = scaler * x3
(:106-123, :146-150) and the `odeint(...)` call (:323, :326) run in the C ABI (`ops.field_eval`,
`ops.ode_solve` with variant MACARON); sub-modules are parameter containers read at call time.
There is no CPU path.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib, ops
from .vit_ode import DEFAULT_PRECISION, _next_drop_seed, adaptive_solve_args


class PatchEmbed(nn.Module):
    """macaron.py:10-35 -- conv patchify (+ the optional `init_ivp` 5x5 conv branch, pooled)."""

    def __init__(self, img_size=32, patch_size=4, in_chans=3, embed_dim=192):
        super().__init__()
        assert img_size % patch_size == 0, "img_size must be divisible by patch_size"
        self.grid_size = img_size // patch_size
        self.num_patches = self.grid_size * self.grid_size
        self.proj = nn.Conv2d(in_chans, embed_dim, kernel_size=patch_size, stride=patch_size)
        self.init_ivp = nn.Conv2d(in_chans, embed_dim, kernel_size=5, stride=1)
        self.pooler = nn.AdaptiveAvgPool2d(1)

    def forward(self, x: torch.Tensor, learn_ivp: bool = False):
        pooled = None
        if learn_ivp:
            pooled = self.pooler(F.gelu(self.init_ivp(x))).flatten(2).squeeze(-1)
        tokens = self.proj(x).flatten(2).transpose(1, 2).contiguous()
        return tokens, pooled


class MLP(nn.Module):
    """macaron.py:38-52 -- fc1 + GELU (+ dropout); defined by the reference, unused by its block."""

    def __init__(self, dim: int, hidden_dim: int, drop: float = 0.0):
        super().__init__()
        self.fc1 = nn.Linear(dim, hidden_dim)
        self.act = nn.GELU()
        self.drop = nn.Dropout(drop)

    def forward(self, x):
        return self.drop(self.act(self.fc1(x)))


class MultiheadSelfAttention(nn.Module):
    """Parameter container for macaron.py:55-71: `nn.MultiheadAttention(bias=True, batch_first=True)`
    called with need_weights=False (no attention map leaves the block)."""

    def __init__(self, dim: int, num_heads: int, attn_drop: float = 0.0, proj_drop: float = 0.0, bias: bool = True):
        super().__init__()
        self.mha = nn.MultiheadAttention(embed_dim=dim, num_heads=num_heads, dropout=attn_drop, bias=bias,
                                         batch_first=True)
        self.proj_drop = nn.Dropout(proj_drop)


class ParallelAttentionMLP(nn.Module):
    """macaron.py:78-123 (the reference keeps the class name of the parallel block): half-FFN,
    attention, half-FFN with three LayerNorms, one SHARED ffn and a learnable `res_scale`."""

    def __init__(self, dim: int, num_heads: int, mlp_ratio: float = 4.0, attn_drop: float = 0.0,
                 proj_drop: float = 0.0, mlp_drop: float = 0.0, bias_init_scale: float = 1e-3):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim)
        self.norm2 = nn.LayerNorm(dim)
        self.norm3 = nn.LayerNorm(dim)
        hidden = int(dim * mlp_ratio)
        self.ffn = nn.Sequential(nn.Linear(dim, hidden), nn.GELU(), nn.Dropout(mlp_drop),
                                 nn.Linear(hidden, dim), nn.Dropout(mlp_drop))
        self.attn = MultiheadSelfAttention(dim=dim, num_heads=num_heads, attn_drop=attn_drop, proj_drop=proj_drop)
        for m in self.ffn.modules():     # :96-101 -- start close to the identity
            if isinstance(m, nn.Linear):
                nn.init.trunc_normal_(m.weight, std=1e-3)
                if m.bias is not None:
                    nn.init.zeros_(m.bias)
        self.res_scale = nn.Parameter(torch.ones(1) * 1.0)
        self.dim, self.num_heads = dim, num_heads
        self._drops = (attn_drop, proj_drop, mlp_drop)
        self.precision = DEFAULT_PRECISION

    def field_spec(self, scaler: float) -> ops.FieldSpec:
        # training-mode dropout (macaron.py:58-61, :88-94): attention map, after out_proj, after GELU and after ffn.3 of
        # both half steps (each with its own mask), re-drawn at every field evaluation
        attn_drop, proj_drop, mlp_drop = self._drops if self.training else (0.0, 0.0, 0.0)
        seed_kw = _next_drop_seed(self) if (attn_drop > 0 or proj_drop > 0 or mlp_drop > 0) else {}
        return ops.FieldSpec(dim=self.dim, heads=self.num_heads, hidden=self.ffn[0].weight.shape[0],
                             scaler=float(scaler), variant=_lib.FIELD_MACARON, precision=self.precision,
                             backward=getattr(self, "backward_mode", "auto"),
                             attn_drop=float(attn_drop), proj_drop=float(proj_drop), mlp_drop=float(mlp_drop),
                             **seed_kw)

    def field_weights(self) -> Dict[str, Optional[torch.Tensor]]:
        mha = self.attn.mha
        return {
            "norm_a_w": self.norm1.weight, "norm_a_b": self.norm1.bias,
            "norm_b_w": self.norm2.weight, "norm_b_b": self.norm2.bias,
            "norm_c_w": self.norm3.weight, "norm_c_b": self.norm3.bias,
            "in_proj_w": mha.in_proj_weight, "in_proj_b": mha.in_proj_bias,
            "out_proj_w": mha.out_proj.weight, "out_proj_b": mha.out_proj.bias,
            "fc1_w": self.ffn[0].weight, "fc1_b": self.ffn[0].bias,
            "fc2_w": self.ffn[3].weight, "fc2_b": self.ffn[3].bias,
            "res_scale": self.res_scale,
        }

    def forward(self, x: torch.Tensor, t: Optional[torch.Tensor] = None) -> torch.Tensor:
        x3, _ = ops.field_eval(x, self.field_spec(1.0), self.field_weights(), want_p=False)
        return x3


class ViT_ODEFunc(nn.Module):
    """macaron.py:125-150 -- f(t, x) = block(x, t) * scaler."""

    def __init__(self, dim: int, num_heads: int, mlp_ratio: float = 4.0, attn_drop: float = 0.0,
                 proj_drop: float = 0.0, mlp_drop: float = 0.0, emulate_depth: int = 12, time_interval: float = 12.0):
        super().__init__()
        self.dim = dim
        self.block = ParallelAttentionMLP(dim, num_heads, mlp_ratio, attn_drop, proj_drop, mlp_drop)
        self.scaler = float(emulate_depth) if time_interval == 1.0 else 1.0

    def forward(self, t: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
        dx, _ = ops.field_eval(x, self.block.field_spec(self.scaler), self.block.field_weights(), want_p=False)
        return dx


class ViTMacaron(nn.Module):
    """macaron.py:157-352 with the `odeint(...)` call replaced by one `odevit_solve_fwd` (variant
    MACARON) and its autograd by `odevit_solve_bwd`."""

    AVG_DISTANCES_CONSECUTIVE_HIDDEN_STATES_VIT = torch.tensor(
        [19.9335, 12.61485625, 13.10309922, 14.70024375, 15.15418125, 17.1821, 14.34054062,
         18.23386562, 23.4014875, 14.24714063, 29.36258125, 171.6232875])

    def __init__(self, img_size: int = 32, patch_size: int = 4, in_chans: int = 3, num_classes: int = 100,
                 embed_dim: int = 192, num_heads: int = 3, mlp_ratio: float = 4.0, attn_drop: float = 0.0,
                 proj_drop: float = 0.0, mlp_drop: float = 0.0, emulate_depth: int = 12,
                 time_interval: float = 12.0, num_eval_steps: int = 48, solver: str = "rk4",
                 add_distillation_token: bool = False, predict_outher_space: bool = False,
                 outher_embedding_dimension: int = 768, learn_ivp: bool = False):
        super().__init__()
        self.patch_embed = PatchEmbed(img_size, patch_size, in_chans, embed_dim)
        num_patches = self.patch_embed.num_patches
        num_extra_tokens = 1
        self.learn_ivp = learn_ivp
        self.add_distillation_token = add_distillation_token
        if learn_ivp:
            self._ivp_projector = nn.Linear(2 * embed_dim, embed_dim)
        if add_distillation_token:
            num_extra_tokens += 1
            self.dist_token = nn.Parameter(torch.zeros(1, 1, embed_dim))
            self.dist_head = nn.Linear(embed_dim, num_classes)
            self.norm_dist = nn.LayerNorm(embed_dim)
        self.cls_token = nn.Parameter(torch.zeros(1, 1, embed_dim))
        self.pos_embed = nn.Parameter(torch.zeros(1, num_extra_tokens + num_patches, embed_dim))
        self.pos_drop = nn.Dropout(p=0.0)
        self.embedding_dim = embed_dim
        if predict_outher_space:
            # the reference calls init_space_predictor(embed_dim, outher_dim) on a one-argument method
            # (:218-219 vs :274-275) and fails with a TypeError; same here
            self.outher_embed = self.init_space_predictor(embed_dim, outher_embedding_dimension)
        self.odefunc = ViT_ODEFunc(dim=embed_dim, num_heads=num_heads, mlp_ratio=mlp_ratio, attn_drop=attn_drop,
                                   proj_drop=proj_drop, mlp_drop=mlp_drop, emulate_depth=emulate_depth,
                                   time_interval=time_interval)
        self.norm_head = nn.LayerNorm(embed_dim)
        self.head = nn.Linear(embed_dim, num_classes)
        self.solver = solver
        self.time_interval = time_interval
        self.num_eval_steps = num_eval_steps
        self.t_grid = torch.linspace(0.0, time_interval, num_eval_steps)
        # None, or {"rtol", "atol"[, "first_step", "max_num_steps", "differentiable"]}: forward integrates over t_grid
        # with the per-image adaptive Dormand-Prince solve (inference only unless "differentiable" is True; a plain
        # attribute like `precision`, not a config key)
        self.adaptive_solve = None
        self._init_weights()

    # -- precision switch (not in the reference) -------------------------------------------------
    @property
    def precision(self) -> str:
        return self.odefunc.block.precision

    @precision.setter
    def precision(self, value: str) -> None:
        if value not in _lib.PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(_lib.PRECISIONS)}")
        self.odefunc.block.precision = value

    @property
    def device(self):
        return next(self.parameters()).device

    def get_proportional_control_points_with_temperature(self, temperature, num_eval_steps: Optional[int] = None):
        """:244-259 -- softmax-proportional checkpoints, WITHOUT the last-index clamp of the other model."""
        x = self.AVG_DISTANCES_CONSECUTIVE_HIDDEN_STATES_VIT / temperature
        e = torch.exp(x - torch.max(x))
        w = e / torch.sum(e)
        if num_eval_steps is not None:
            steps = torch.round(w * num_eval_steps)
        else:
            steps = torch.round(w * self.num_eval_steps).int()
        return torch.cumsum(steps, dim=0).long()

    def _init_weights(self):
        nn.init.trunc_normal_(self.pos_embed, std=0.02)
        nn.init.trunc_normal_(self.cls_token, std=0.02)
        if self.add_distillation_token:
            nn.init.trunc_normal_(self.dist_token, std=0.02)
        if self.head.bias is not None:
            nn.init.zeros_(self.head.bias)

    def init_space_predictor(self, outher_embedding_dimension):
        self.space_predictor = nn.Linear(self.embedding_dim, outher_embedding_dimension)

    def embed(self, x: torch.Tensor) -> torch.Tensor:
        """:278-300 -- [cls | (dist) | patches] + positional embedding."""
        x, ivp = self.patch_embed(x, self.learn_ivp)
        B, N, _ = x.shape
        cls = self.cls_token.expand(B, -1, -1)
        if self.learn_ivp:
            cls = F.gelu(self._ivp_projector(torch.cat([cls, ivp.unsqueeze(1)], dim=-1)))
        if self.add_distillation_token:
            x = torch.cat([cls, self.dist_token.expand(B, -1, -1), x], dim=1)
            extra = 2
        else:
            x = torch.cat([cls, x], dim=1)
            extra = 1
        x = x + self.pos_embed[:, :(N + extra)]
        return self.pos_drop(x)

    def forward(self, pixel_values: torch.Tensor, labels: Optional[torch.Tensor] = None,
                output_hidden_states: bool = False, output_control_points: bool = False,
                t_grid: Optional[torch.Tensor] = None, temperature: Optional[float] = 100.0):
        """:302-352."""
        block = self.odefunc.block
        if self.adaptive_solve is not None:
            cfg = adaptive_solve_args(self, {})
        tokens = self.embed(pixel_values)
        if t_grid is None:
            num_eval_steps, t = self.num_eval_steps, self.t_grid
        else:
            num_eval_steps, t = len(t_grid), t_grid
        idx = None
        if output_control_points:
            idx = self.get_proportional_control_points_with_temperature(temperature=temperature,
                                                                        num_eval_steps=num_eval_steps)
            if int(idx.max()) >= num_eval_steps or int(idx.min()) < -num_eval_steps:
                raise IndexError(f"control point index {int(idx.max())} is out of bounds for a trajectory of "
                                 f"{num_eval_steps} states (the reference's states[control_points] fails alike)")
            idx = idx % num_eval_steps
        if self.adaptive_solve is not None:
            res = ops.ode_solve_adaptive(tokens, t, block.field_spec(self.odefunc.scaler), block.field_weights(),
                                         cfg["rtol"], cfg["atol"], first_step=cfg.get("first_step"),
                                         max_num_steps=cfg.get("max_num_steps", ops.DOPRI5_MAX_NUM_STEPS),
                                         differentiable=cfg.get("differentiable", False),
                                         capturable=cfg.get("capturable", False))
            if idx is not None:
                res["rows"] = res["states"][idx]
        else:
            res = ops.ode_solve(tokens, t, block.field_spec(self.odefunc.scaler), self.solver, block.field_weights(),
                                row_index=idx.tolist() if idx is not None else ())
        states, final = res["states"], res["final"]
        out = {"logits": self.head(self.norm_head(final[:, 0]))}
        if self.adaptive_solve is not None:
            out["nfe"] = res["nfe"]
        if self.add_distillation_token:
            out["logits_dist"] = self.dist_head(self.norm_dist(final[:, 1]))
        if labels is not None:
            out["loss"] = F.cross_entropy(out["logits"], labels)
        if output_hidden_states:
            out["states"] = states
        if output_control_points:
            out["control_points"] = res["rows"]
        return out
