"""Drop-in `nn.Module` surface of the ODE-ViT hot path, backed by libodevit.so.

Mirrors (constructor kwargs, call signatures, `state_dict` keys, output-dict keys, side
attributes) of the reference's `models/ode_transformer_gpt.py`:

    CenterNorm :66-83            MLP :185-200            MultiheadSelfAttention :203-232
    ParallelAttentionMLP :240-277   ViT_ODEFunc :280-330   PatchEmbed :86-182
    ViTNeuralODE :338-645

What differs is where the arithmetic runs.  `ParallelAttentionMLP.forward`,
`ViT_ODEFunc.forward` and the `odeint(...)` call inside `ViTNeuralODE.forward` enqueue the
fused sm_100a kernels through the C ABI (`ops.field_eval`, `ops.ode_solve`); the sub-modules
(`CenterNorm`, `MLP`, `MultiheadSelfAttention`) are parameter containers that keep the
reference's `state_dict` layout -- the kernels read their parameters at call time, so modules
and parameters may be re-assigned after construction exactly as the reference's training
scripts do (main_classification_ode_distillation.py:86-100).

There is no CPU path: a CPU tensor raises `OdevitError`.

Two switches that the reference does not have (plain attributes, not ctor kwargs, so hydra
configs keep working): `model.precision` in {"fp32", "bf16"} (default "fp32": results within
1e-4 of the reference; "bf16" = tensor-core operands, within 2e-2) and `model.time_mod`
(optional ScaleShift modulation, models/time_emb.py, off like in the reference).
"""
from __future__ import annotations

import math
import os
from typing import Dict, Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib, ops
from ._lib import OdevitError

DEFAULT_PRECISION = os.environ.get("ODEVIT_PRECISION", "fp32")


class CenterNorm(nn.Module):
    """Parameter container for ode_transformer_gpt.py:66-83: D/(D-1)*(x-mean)*w + b (no variance,
    `eps` accepted and unused).  On the hot path the centring is a kernel prologue and the affine
    part is folded into the projection weights (csrc/rows.cu::fold_w1_kernel)."""

    def __init__(self, normalized_shape, eps=1e-6):
        super().__init__()
        self.weight = nn.Parameter(torch.ones(normalized_shape))
        self.bias = nn.Parameter(torch.zeros(normalized_shape))
        self.scale = normalized_shape / (normalized_shape - 1.0)

    def forward(self, x):
        # Not on the hot path (the reference only calls it through the block); kept so the module
        # is usable stand-alone, e.g. `norm_dist`.
        return self.weight * (self.scale * (x - x.mean(-1, keepdim=True))) + self.bias


class MLP(nn.Module):
    """Parameter container for ode_transformer_gpt.py:185-200 (fc1/fc2 without bias, erf-GELU)."""

    def __init__(self, dim: int, hidden_dim: int, drop: float = 0.0):
        super().__init__()
        self.fc1 = nn.Linear(dim, hidden_dim, bias=False)
        self.act = nn.GELU()
        self.fc2 = nn.Linear(hidden_dim, dim, bias=False)
        self.drop = nn.Dropout(drop)


class MultiheadSelfAttention(nn.Module):
    """Parameter container for ode_transformer_gpt.py:203-232.  Holds a real
    `nn.MultiheadAttention(bias=False, batch_first=True)` so `mha.in_proj_weight` /
    `mha.out_proj.weight` have the reference's names, shapes and initialisation."""

    def __init__(self, dim: int, num_heads: int, attn_drop: float = 0.0, proj_drop: float = 0.0,
                 bias: bool = False):
        super().__init__()
        self.mha = nn.MultiheadAttention(embed_dim=dim, num_heads=num_heads, dropout=attn_drop,
                                         bias=bias, batch_first=True)
        self.proj_drop = nn.Dropout(proj_drop)


class L2SelfAttention(nn.Module):
    """Parameter container for ode_transformer_gpt.py:12-63: separate q/k/v/out Linears WITH bias;
    weights exp(-||q_i - k_j||^2 / sqrt(d)) normalised by (row sum + 1e-8).  The arithmetic runs in
    libodevit.so (variant PARALLEL_L2)."""

    def __init__(self, dim: int, num_heads: int, attn_drop: float = 0.0, proj_drop: float = 0.0):
        super().__init__()
        self.num_heads = num_heads
        self.head_dim = dim // num_heads
        self.scale = self.head_dim ** -0.5
        self.q_proj = nn.Linear(dim, dim)
        self.k_proj = nn.Linear(dim, dim)
        self.v_proj = nn.Linear(dim, dim)
        self.out_proj = nn.Linear(dim, dim)
        self.attn_drop = nn.Dropout(attn_drop)
        self.proj_drop = nn.Dropout(proj_drop)


def _next_drop_seed(block: nn.Module) -> dict:
    """FieldSpec seed arguments of this call.  Eager calls draw a 64-bit host seed from PyTorch's CPU generator
    (`torch.manual_seed` reproduces a step, as in the reference).  While a CUDA graph is being captured -- or when
    `block.device_seed` is set, which GraphedTrainStep does before its warm-up -- the seed lives in device memory
    (ops.DropState) and a 1-thread kernel advances it, so every replay of the captured step draws new masks.
    `block.last_drop_seed` keeps what was used (int or int64[1] CUDA tensor): tests restate the masks from it."""
    if getattr(block, "device_seed", False) or torch.cuda.is_current_stream_capturing():
        dev = next(block.parameters()).device
        st = getattr(block, "_drop_state", None)
        if st is None or st.state.device != dev:
            st = ops.DropState(dev)
            block._drop_state = st
        block.last_drop_seed = st.next_seed()
        return dict(seed_dev=block.last_drop_seed)
    block.last_drop_seed = ops.draw_seed()
    return dict(seed=block.last_drop_seed)


class ParallelAttentionMLP(nn.Module):
    """ode_transformer_gpt.py:240-277 -- returns F(x) + G(x) = MLP(CN_mlp x) + MHA(CN_attn x) and
    stores the attention map of this evaluation in `self.attentions`."""

    def __init__(self, dim: int, num_heads: int, mlp_ratio: float = 4.0, attn_drop: float = 0.0,
                 proj_drop: float = 0.0, mlp_drop: float = 0.0, use_l2: bool = False):
        super().__init__()
        self.norm_attn = CenterNorm(dim)
        self.norm_mlp = CenterNorm(dim)
        self.use_l2 = use_l2
        if use_l2:      # :259-262
            self.attn = L2SelfAttention(dim=dim, num_heads=num_heads, attn_drop=attn_drop, proj_drop=proj_drop)
        else:
            self.attn = MultiheadSelfAttention(dim=dim, num_heads=num_heads, attn_drop=attn_drop,
                                               proj_drop=proj_drop)
        self.mlp = MLP(dim=dim, hidden_dim=int(dim * mlp_ratio), drop=mlp_drop)
        self.dim, self.num_heads = dim, num_heads
        self._drops = (attn_drop, proj_drop, mlp_drop)
        self.precision = DEFAULT_PRECISION
        self.time_mod: Optional[Dict[str, torch.Tensor]] = None

    # -- what the kernels consume --------------------------------------------------------------
    def field_spec(self, scaler: float) -> ops.FieldSpec:
        hidden = self.mlp.fc1.weight.shape[0]
        # dropout is live in training mode only; every call draws a fresh seed, and inside a solve the
        # masks are re-drawn at every field evaluation from (seed, evaluation index) -- SURVEY 2.3 quirk 16
        attn_drop, proj_drop, mlp_drop = self._drops if self.training else (0.0, 0.0, 0.0)
        seed_kw = _next_drop_seed(self) if (attn_drop > 0 or proj_drop > 0 or mlp_drop > 0) else {}
        return ops.FieldSpec(dim=self.dim, heads=self.num_heads, hidden=hidden, scaler=float(scaler),
                             variant=_lib.FIELD_PARALLEL_L2 if self.use_l2 else _lib.FIELD_PARALLEL,
                             precision=self.precision,
                             backward=getattr(self, "backward_mode", "auto"),
                             attn_drop=float(attn_drop), proj_drop=float(proj_drop), mlp_drop=float(mlp_drop),
                             **seed_kw)

    def field_weights(self) -> Dict[str, Optional[torch.Tensor]]:
        """odevit_weights field name -> parameter, read at call time (SURVEY 7.3-7)."""
        if self.use_l2:
            a = self.attn   # the ABI takes [Wq; Wk; Wv] stacked like nn.MultiheadAttention's packed weight
            in_w = torch.cat([a.q_proj.weight, a.k_proj.weight, a.v_proj.weight], 0)
            in_b = torch.cat([a.q_proj.bias, a.k_proj.bias, a.v_proj.bias], 0)
            out_w, out_b = a.out_proj.weight, a.out_proj.bias
        else:
            mha = self.attn.mha
            in_w, in_b, out_w, out_b = mha.in_proj_weight, mha.in_proj_bias, mha.out_proj.weight, mha.out_proj.bias
        w = {
            "norm_a_w": self.norm_attn.weight, "norm_a_b": self.norm_attn.bias,
            "norm_b_w": self.norm_mlp.weight, "norm_b_b": self.norm_mlp.bias,
            "in_proj_w": in_w, "in_proj_b": in_b,
            "out_proj_w": out_w, "out_proj_b": out_b,
            "fc1_w": self.mlp.fc1.weight, "fc1_b": self.mlp.fc1.bias,
            "fc2_w": self.mlp.fc2.weight, "fc2_b": self.mlp.fc2.bias,
        }
        if self.time_mod:
            for k in _lib.MOD_FIELDS:
                if self.time_mod.get(k) is not None:
                    w[k] = self.time_mod[k]
        return w

    def forward(self, x: torch.Tensor, t: Optional[torch.Tensor] = None) -> torch.Tensor:
        dx, self.attentions = ops.field_eval(x, self.field_spec(1.0), self.field_weights(), want_p=True)
        return dx


class ViT_ODEFunc(nn.Module):
    """ode_transformer_gpt.py:280-330 -- f(t, x) = scaler * block(x); appends the detached
    attention map of every evaluation to `self.attention_trajectory`."""

    def __init__(self, dim: int, num_heads: int, mlp_ratio: float = 4.0, attn_drop: float = 0.0,
                 proj_drop: float = 0.0, mlp_drop: float = 0.0, emulate_depth: int = 12,
                 time_interval: float = 12.0, l2_attention: bool = True):
        super().__init__()
        self.dim = dim
        self.block = ParallelAttentionMLP(dim, num_heads, mlp_ratio, attn_drop, proj_drop, mlp_drop,
                                          use_l2=l2_attention)
        self.scaler = float(emulate_depth) if time_interval == 1.0 else 1.0

    def forward(self, t: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
        dx, p = ops.field_eval(x, self.block.field_spec(self.scaler), self.block.field_weights(), want_p=True)
        self.block.attentions = p
        if not hasattr(self, "attention_trajectory"):
            self.attention_trajectory = []
        self.attention_trajectory.append(p.detach())
        return dx


def odeint(func: ViT_ODEFunc, y0: torch.Tensor, t: torch.Tensor, *, method: str = "rk4",
           rtol=None, atol=None, options=None, record_attention: bool = True):
    """`torchdiffeq.odeint(func, y0, t, method=...)` as the reference calls it
    (ode_transformer_gpt.py:571-578), for the fused vector field only: the whole fixed grid runs in
    libodevit.so.  Returns the trajectory `[len(t), *y0.shape]`; like the reference's call it
    leaves `func.block.attentions` (last evaluation, differentiable) and extends
    `func.attention_trajectory` (every evaluation, detached) unless `record_attention=False`.
    rtol / atol are ignored by fixed-grid methods; `options` (step_size ...) is not supported."""
    if not (hasattr(func, "block") and hasattr(func.block, "field_spec") and hasattr(func, "scaler")):
        raise TypeError("odevit_b200.odeint integrates odevit_b200 vector-field modules only "
                        "(there is no generic / CPU solver in this package)")
    if hasattr(func.block, "res_scale"):   # the Macaron block
        record_attention = False   # macaron.py:60-65: need_weights=False, the block exposes no map
    if options:
        raise NotImplementedError("odeint options (step_size, ...) are not used by the reference and not built")
    res = ops.ode_solve(y0, t, func.block.field_spec(func.scaler), method, func.block.field_weights(),
                        want_p_last=record_attention, p_traj_first=0 if record_attention else None)
    if record_attention:
        if res["p_last"] is not None:
            func.block.attentions = res["p_last"]
        if not hasattr(func, "attention_trajectory"):
            func.attention_trajectory = []
        if res["p_traj"] is not None:
            func.attention_trajectory.extend(res["p_traj"].unbind(0))
    return res["states"]


def _check_field_module(func, who: str) -> None:
    if not (hasattr(func, "block") and hasattr(func.block, "field_spec") and hasattr(func, "scaler")):
        raise TypeError(f"odevit_b200.{who} integrates odevit_b200 vector-field modules only "
                        "(there is no generic / CPU solver in this package)")


def odeint_adaptive(func, y0: torch.Tensor, t: torch.Tensor, *, rtol: float = 1e-7, atol: float = 1e-9,
                    options: Optional[dict] = None, return_stats: bool = False, differentiable: bool = False,
                    capturable: bool = False, record_attention: bool = False):
    """`torchdiffeq.odeint(func, y0, t, method="dopri5", rtol, atol, options)` for the fused vector field, with the
    step size controlled PER IMAGE (ops.ode_solve_adaptive): image b's error norm, steps and dense output depend on
    image b alone, where torchdiffeq takes one norm over the batch.  `t` strictly increasing; options: `first_step`,
    `max_num_steps` (attempted steps per image over the whole solve, not per output interval).  `record_attention`
    leaves `func.block.attentions` as `odeint` does: image b's row is the map of b's own last field evaluation (k7 = f(y1)
    of its last accepted step), differentiable with `differentiable`; `func.attention_trajectory` (every evaluation's
    map) is not built and stays as it is (a MACARON field exposes no map: ignored there, as in `odeint`).  Not with
    `capturable`.  Inference only unless `differentiable`: then the trajectory is differentiable with respect to y0 and the
    field's weights, with each image's accepted steps frozen (not the continuous adjoint, and not autograd through an
    unrolled torchdiffeq solve).  `capturable`: the on-chip, non-synchronising form that a CUDA graph can capture
    (ops.ode_solve_adaptive; stats then also hold `status` and `rounds` is a 0-d device tensor).  Returns the trajectory
    [len(t), *y0.shape], or (trajectory, stats) with stats = dict(nfe, accepted, rejected: int32 [B] device tensors,
    rounds: int) when `return_stats`."""
    _check_field_module(func, "odeint_adaptive")
    options = dict(options or {})
    unknown = set(options) - {"first_step", "max_num_steps"}
    if unknown:
        raise ValueError(f"unsupported dopri5 options {sorted(unknown)}; first_step and max_num_steps are built")
    if hasattr(func.block, "res_scale"):   # the Macaron block
        record_attention = False
    res = ops.ode_solve_adaptive(y0, t, func.block.field_spec(func.scaler), func.block.field_weights(), rtol, atol,
                                 first_step=options.get("first_step"),
                                 max_num_steps=options.get("max_num_steps", ops.DOPRI5_MAX_NUM_STEPS),
                                 differentiable=differentiable, capturable=capturable, want_p_last=record_attention)
    if record_attention:
        func.block.attentions = res["p_last"]
    if return_stats:
        return res["states"], {k: res[k] for k in ("nfe", "accepted", "rejected", "rounds", "status") if k in res}
    return res["states"]


def adaptive_solve_args(model: nn.Module, output_flags: Dict[str, bool]) -> dict:
    """Checks a model's `adaptive_solve` request (a dict with rtol, atol and optionally first_step, max_num_steps,
    differentiable, capturable, attention_outputs) and the forward's arguments against what the adaptive solve can give.
    `output_attentions` is honoured only when the request opts in with "attention_outputs": True -- the outputs cost one
    extra field evaluation and one small kernel per evaluation, and a request without the key keeps refusing them."""
    cfg = dict(model.adaptive_solve)
    unknown = set(cfg) - {"rtol", "atol", "first_step", "max_num_steps", "differentiable", "capturable",
                          "attention_outputs"}
    if unknown or "rtol" not in cfg or "atol" not in cfg:
        raise ValueError(f"adaptive_solve takes rtol, atol [, first_step, max_num_steps, differentiable, capturable, "
                         f"attention_outputs], got {sorted(model.adaptive_solve)}")
    if output_flags.get("output_attention_trajectory"):
        raise ValueError("output_attention_trajectory is not built with adaptive_solve (the per-image list of every "
                         "evaluation's map); output_attentions is, with \"attention_outputs\": True")
    if output_flags.get("output_attentions"):
        if not cfg.get("attention_outputs", False):
            raise ValueError("output_attentions with adaptive_solve needs \"attention_outputs\": True in it (each image's "
                             "last-evaluation map and JaSMin window: one extra field evaluation and a small kernel per "
                             "evaluation)")
        if cfg.get("capturable", False):
            raise ValueError("output_attentions is not built with adaptive_solve's capturable=True (the on-chip adaptive "
                             "solve exports no maps); the default path gives it")
    if (not cfg.get("differentiable", False) and torch.is_grad_enabled()
            and any(p.requires_grad for p in model.parameters())):
        raise RuntimeError("adaptive_solve is inference-only (no backward is built): run the model under torch.no_grad()")
    return cfg


class PatchEmbed(nn.Module):
    """ode_transformer_gpt.py:86-182 -- conv patchify, [cls | (dist) | patches | registers], learned
    positional embedding over all tokens or over cls+patches only.  (Row f1 of SURVEY section 8:
    outside the hot path; plain cuDNN/aten here.)"""

    def __init__(self, img_size=32, patch_size=4, in_chans=3, embed_dim=192, add_distillation_token=False,
                 register_tokens: int = 4, pos_embed_register_tokens: bool = True):
        super().__init__()
        assert img_size % patch_size == 0, "img_size must be divisible by patch_size"
        self.grid_size = img_size // patch_size
        self.num_patches = self.grid_size * self.grid_size
        self.pos_embed_register_tokens = pos_embed_register_tokens
        self.proj = nn.Conv2d(in_chans, embed_dim, kernel_size=patch_size, stride=patch_size)
        self.add_distillation_token = add_distillation_token
        if add_distillation_token:
            self.dist_token = nn.Parameter(torch.zeros(1, 1, embed_dim))
        self.cls_token = nn.Parameter(torch.zeros(1, 1, embed_dim))
        self.register_tokens = nn.Parameter(torch.randn(register_tokens, embed_dim))
        self.num_register_tokens = register_tokens
        self.pos_embed = nn.Parameter(torch.zeros(1, self.num_patches + 1 + register_tokens, embed_dim))
        self.pos_drop = nn.Dropout(p=0.0)
        nn.init.trunc_normal_(self.cls_token, std=0.02)
        nn.init.trunc_normal_(self.register_tokens, std=0.02)
        nn.init.trunc_normal_(self.pos_embed, std=0.02)
        if add_distillation_token:
            nn.init.trunc_normal_(self.dist_token, std=0.02)

    def forward(self, x: torch.Tensor, learn_ivp: bool = False) -> torch.Tensor:
        p = self.proj.kernel_size[0]
        if (getattr(self, "precision", "fp32") == "bf16" and x.is_cuda and x.dtype == torch.float32
                and x.shape[-1] % p == 0 and x.shape[-2] % p == 0 and not learn_ivp and self.pos_drop.p == 0.0
                and self.proj.out_channels % 4 == 0 and getattr(self, "fused_assembly", True)):
            # bf16 mode: im2col + ONE tcgen05 GEMM whose epilogue writes the patch rows of the token tensor with bias and
            # positional rows added; cls / dist / register rows by one small kernel (ops.token_assembly, row (f)1)
            n_pos = self.num_patches + 1 + (self.num_register_tokens if self.pos_embed_register_tokens else 0)
            return ops.token_assembly(x, self.proj.weight, self.proj.bias, self.cls_token,
                                      self.dist_token if self.add_distillation_token else None,
                                      self.register_tokens if self.num_register_tokens else None, self.pos_embed, p, n_pos)
        if (getattr(self, "precision", "fp32") == "bf16" and x.is_cuda and x.dtype == torch.float32
                and x.shape[-1] % p == 0 and x.shape[-2] % p == 0):
            # bf16 mode: im2col + tcgen05 GEMM (ops.patch_project) instead of cuDNN's TF32 convolution
            x = ops.patch_project(x, self.proj.weight, self.proj.bias, p)
        else:
            x = self.proj(x).flatten(2).transpose(1, 2)
        B = x.shape[0]
        parts = [self.cls_token.expand(B, -1, -1)]
        if self.add_distillation_token:
            parts.append(self.dist_token.expand(B, -1, -1))
        parts += [x, self.register_tokens.expand(B, -1, -1)]
        x = torch.cat(parts, dim=1)
        n_pos = self.num_patches + 1 + (self.num_register_tokens if self.pos_embed_register_tokens else 0)
        pe = self.pos_embed[:, :n_pos].to(x.device)
        if n_pos == x.shape[1]:
            x = x + pe
        else:
            x = torch.cat([x[:, :n_pos] + pe, x[:, n_pos:]], dim=1)
        return self.pos_drop(x)


class ViTNeuralODE(nn.Module):
    """ode_transformer_gpt.py:338-645 with the `odeint(...)` call (:571-578) replaced by one
    `odevit_solve_fwd` (and its autograd by `odevit_solve_bwd`)."""

    AVG_DISTANCES_CONSECUTIVE_HIDDEN_STATES_VIT = torch.tensor(
        [19.99450625, 12.949505, 5.35348687, 4.86699219, 4.81463781, 4.52093875,
         5.21054063, 5.69734125, 6.1311925, 6.05176188, 6.4614325, 53.514895])

    def __init__(self, img_size: int = 32, patch_size: int = 4, in_chans: int = 3, num_classes: int = 100,
                 embed_dim: int = 192, num_heads: int = 3, mlp_ratio: float = 4.0, attn_drop: float = 0.0,
                 proj_drop: float = 0.0, mlp_drop: float = 0.0, emulate_depth: int = 12,
                 time_interval: float = 12.0, num_eval_steps: int = 24, solver: str = "rk4",
                 add_distillation_token: bool = False, l2_attention: bool = False,
                 outher_embedding_dimension: int = 768, register_tokens: int = 4,
                 pos_embed_register_tokens: bool = False):
        super().__init__()
        self.patch_embed = PatchEmbed(img_size, patch_size, in_chans, embed_dim, add_distillation_token,
                                      register_tokens=register_tokens,
                                      pos_embed_register_tokens=pos_embed_register_tokens)
        self.emulate_depth = emulate_depth
        self.l2_attention = l2_attention
        self.add_distillation_token = add_distillation_token
        self.odefunc = ViT_ODEFunc(dim=embed_dim, num_heads=num_heads, mlp_ratio=mlp_ratio, attn_drop=attn_drop,
                                   proj_drop=proj_drop, mlp_drop=mlp_drop, emulate_depth=emulate_depth,
                                   time_interval=time_interval, l2_attention=l2_attention)
        self.head = nn.Linear(embed_dim, num_classes)
        self.solver = solver
        if add_distillation_token:
            self.dist_head = nn.Linear(embed_dim, num_classes)
            self.norm_dist = CenterNorm(embed_dim)
        self.embed_dim = embed_dim
        self.time_interval = time_interval
        self.num_eval_steps = num_eval_steps
        self.t_grid = torch.linspace(0.0, time_interval, num_eval_steps)  # plain attribute, not a buffer
        # None, or {"rtol", "atol"[, "first_step", "max_num_steps", "differentiable", "capturable", "attention_outputs"]}:
        # forward integrates over t_grid with the per-image adaptive Dormand-Prince solve (inference only unless
        # "differentiable" is True; output_attentions only with "attention_outputs": True; a plain attribute like
        # `precision`, not a config key)
        self.adaptive_solve = None
        self.patch_embed.precision = self.odefunc.block.precision
        self.apply(self._spectral_init)

    # -- precision switch (not in the reference) -------------------------------------------------
    @property
    def precision(self) -> str:
        return self.odefunc.block.precision

    @precision.setter
    def precision(self, value: str) -> None:
        if value not in _lib.PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(_lib.PRECISIONS)}")
        self.odefunc.block.precision = value
        self.patch_embed.precision = value

    @property
    def device(self):
        return next(self.parameters()).device

    def _spectral_init(self, m):
        """:494-513 -- xavier-normal then division by the top singular value (sigma_max = 1)."""
        if isinstance(m, nn.Linear):
            nn.init.xavier_normal_(m.weight)
            if m.bias is not None:
                nn.init.constant_(m.bias, 0)
            m.weight.data = m.weight.data / torch.svd(m.weight)[1][0]
        elif isinstance(m, nn.Conv2d):
            nn.init.xavier_normal_(m.weight)
            m.weight.data = m.weight.data / torch.svd(m.weight.data.reshape(m.weight.shape[0], -1))[1][0]
        elif isinstance(m, (nn.LayerNorm, CenterNorm, nn.BatchNorm2d)):
            nn.init.constant_(m.bias, 0)
            nn.init.constant_(m.weight, 1.0)

    # -- post-solve reductions (SURVEY section 8 row (a)8 / (f)2: stay PyTorch this round) -------
    def g_k(self, p, k=1):
        """:419-427"""
        s, _ = torch.sort(p, dim=-1, descending=True)
        x_k = s[..., k - 1]
        x_k1 = s[..., k] if k < p.size(-1) else torch.zeros_like(x_k)
        return x_k * (1 - x_k + x_k1)

    def jasmin_loss(self, attn_maps, k=0, reduction="mean"):
        """:429-456"""
        if isinstance(attn_maps, torch.Tensor):
            attn_maps = [attn_maps]
        losses = []
        for P in attn_maps:
            P = torch.clamp(P, min=1e-12, max=1.0)
            P = P / (P.sum(dim=-1, keepdim=True) + 1e-12)
            g1 = self.g_k(P, k=1)
            if k == 0:
                loss = torch.log(g1 + 1e-12)
            else:
                loss = torch.log(g1 / (self.g_k(P, k=k) + 1e-12) + 1e-12)
            losses.append(loss.max(dim=-1).values.mean(dim=1).mean())
        losses = torch.stack(losses)
        return losses.mean() if reduction == "mean" else losses.sum()

    def finite_difference_second_derivative_sequence(self, f_t, delta_t=1e-4):
        """:458-468"""
        return (f_t[2:] - 2 * f_t[1:-1] + f_t[:-2]) / (delta_t ** 2)

    def get_proportional_control_points_with_temperature(self, temperature, num_eval_steps: Optional[int] = None):
        """:470-488 (the last index is forced to num_eval_steps-1; num_eval_steps=None fails there too)."""
        x = self.AVG_DISTANCES_CONSECUTIVE_HIDDEN_STATES_VIT / temperature
        e = torch.exp(x - torch.max(x))
        w = e / torch.sum(e)
        if num_eval_steps is not None:
            steps = torch.round(w * num_eval_steps)
        else:
            steps = torch.round(w * self.num_eval_steps).int()
        checkpoints = torch.cumsum(steps, dim=0).long()
        checkpoints[-1] = num_eval_steps - 1
        return checkpoints

    def compute_upper_bound_by_second_derivative(self, R, L):
        """:515-527"""
        Wq, Wk, Wv = self.odefunc.block.attn.mha.in_proj_weight.reshape(3, self.embed_dim, self.embed_dim)
        factor1 = R ** 2 * torch.norm(Wv, p=2)
        factor2 = R * torch.linalg.norm(Wk @ Wq.mT) + (Wk.shape[-1]) ** 0.5
        factor3 = (self.num_eval_steps ** 2) * (Wq.shape[-1] ** 0.5)
        return (math.e ** L - 1) / (2 * L * self.num_eval_steps) * (factor1 * factor2) / factor3

    @torch.no_grad()
    def compute_upper_bound_by_fininte_difference(self, x, L, N, fd_max=None):
        """:529-543.  `fd_max` [B,N]: the maxima of |s[j+2] - 2 s[j+1] + s[j]| when the solve formed them itself
        (trajectory-free inference, x is None then)."""
        first = (math.e ** L - 1) / (2 * L * N)
        if x is None:
            delta_t = 1 / N
            per_seq = fd_max / (delta_t * delta_t)
        else:
            if x.shape[0] < 3:
                raise RuntimeError("finite-difference bound needs a trajectory of at least 3 states "
                                   "(the reference's max() over an empty tensor fails the same way)")
            per_seq = ops.fd_curvature(x, 1 / N)           # one pass over [T,B,N,D] (odevit_fd_curvature)
        per_batch = per_seq.max(-1)[0]
        g = first * per_batch.max()
        # the reference returns a Python float here (:541), i.e. one host sync per forward; inside a CUDA-graph
        # capture (odevit_b200.graphs) a sync is illegal and the 0-d tensor is returned instead
        g = g if torch.cuda.is_current_stream_capturing() else g.item()
        return dict(global_upper_bound=g, batched_upper_bound=first * per_batch,
                    batched_upper_bound_per_seq=first * per_seq)

    def init_space_predictor(self, outher_embedding_dimension):
        self.space_predictor = nn.Linear(self.embed_dim, outher_embedding_dimension)

    # -- forward -----------------------------------------------------------------------------------
    def forward(self, pixel_values: torch.Tensor, labels: Optional[torch.Tensor] = None,
                output_hidden_states: bool = False, output_control_points: bool = False,
                output_attentions: bool = False, output_attention_trajectory: bool = False,
                t_grid: Optional[torch.Tensor] = None, temperature: Optional[float] = 30, jasmin_k: int = 10):
        """:548-645.  Same output dict; the attention maps are exported only for the evaluations a
        caller can observe (last one for `attentions`, the JaSMin window, all on request)."""
        block = self.odefunc.block
        R = self.patch_embed.num_register_tokens
        if self.adaptive_solve is not None:
            cfg = adaptive_solve_args(self, {"output_attentions": output_attentions,
                                             "output_attention_trajectory": output_attention_trajectory})
        tokens = self.patch_embed(pixel_values)
        if t_grid is None:
            num_eval_steps, t = self.num_eval_steps, self.t_grid
        else:
            num_eval_steps, t = len(t_grid), t_grid
        if self.adaptive_solve is not None:
            return self._forward_adaptive(tokens, t, num_eval_steps, cfg, labels, output_hidden_states,
                                          output_control_points, output_attentions, temperature, jasmin_k)
        stages = _lib.STAGES.get(self.solver)
        if stages is None:
            raise ValueError(f"unsupported solver {self.solver!r}")
        n_evals = (num_eval_steps - 1) * stages

        idx = None
        if output_control_points:
            idx = self.get_proportional_control_points_with_temperature(temperature=temperature,
                                                                        num_eval_steps=num_eval_steps)
        p_first, jas = None, None
        window = int(self.num_eval_steps * 0.85)                            # :614-618
        if output_attention_trajectory:
            p_first = 0
        elif output_attentions and window > 0:
            # only the JaSMin statistic of the window's maps is consumed: formed inside the attention kernel, the
            # maps themselves (0.85 T x B x H x N x N fp32) are never written
            jas = (max(0, n_evals - window), int(jasmin_k))
        spec, weights = block.field_spec(self.odefunc.scaler), block.field_weights()
        # Inference that does not ask for `states`: no [T,B,N,D] tensor at all (36 x 8192 x 207 x 768 fp32 would be
        # 188 GB) -- the finite-difference bound is formed inside the solve, the control-point rows are written
        # directly.  Not for shapes the on-chip-state kernel takes (its trajectory rows cost one bulk copy each) and
        # not when a backward pass can follow (the reverse sweep reads the trajectory).
        track = torch.is_grad_enabled() and (tokens.requires_grad or any(
            v is not None and v.requires_grad for v in weights.values()))
        lean = (not output_hidden_states and not output_attention_trajectory and not track and num_eval_steps >= 3
                and not ops.solve_uses_resident(spec, tokens.shape[0], tokens.shape[1], self.solver, num_eval_steps))
        if lean:
            # "auto": only when the trajectory would take a large share of the free memory -- the in-epilogue bound
            # costs ~3 % more time than one pass over a materialised trajectory (measured, S3.8M shape, batch 1024), while
            # allocating and touching a multi-GB trajectory per call has its own cost: the switch sits at 5 % of free memory
            mode = getattr(self, "trajectory_free_inference", os.environ.get("ODEVIT_TRAJECTORY_FREE", "auto"))
            if mode in (False, "0", "off"):
                lean = False
            elif mode == "auto":
                need = 4 * num_eval_steps * tokens.numel()
                lean = need > 0.05 * torch.cuda.mem_get_info(tokens.device)[0]
        if lean:
            res = ops.ode_solve_lean(tokens, t, spec, self.solver, weights,
                                     row_index=idx.tolist() if idx is not None else (), want_p_last=True, jasmin=jas)
        else:
            res = ops.ode_solve(tokens, t, spec, self.solver, weights,
                                row_index=idx.tolist() if idx is not None else (),
                                want_p_last=True, p_traj_first=p_first, jasmin=jas)
        states, final = res["states"], res["final"]
        block.attentions = res["p_last"]

        fused_head = (final.is_cuda and type(self.head) is nn.Linear and final.dtype == torch.float32
                      and getattr(self, "fused_head", True))
        if fused_head:
            # head + smoothed cross-entropy in one launch each way (ops.head_ce, row (f)1)
            logits, loss = ops.head_ce(final, self.head.weight, self.head.bias, labels, 0.05)
        else:
            logits, loss = self.head(final[:, 0]), None
        out = {
            "logits": logits,
            "second_derivative_upper_bound": self.compute_upper_bound_by_second_derivative(R=jasmin_k, L=1 / 2),
            "finite_difference_upper_bound": self.compute_upper_bound_by_fininte_difference(
                states.detach() if states is not None else None, 0.5, 1 / self.num_eval_steps,
                fd_max=res.get("fd_max")),
        }
        p_traj = res["p_traj"]
        if output_attention_trajectory:
            # quirk 12: the reference slices dims 2,3 of the stacked [E,B,H,N,N] tensor (heads, query rows)
            stacked = p_traj if p_traj is not None else tokens.new_empty(0, tokens.shape[0], block.num_heads,
                                                                         tokens.shape[1], tokens.shape[1])
            out["attention_trajectory"] = stacked[:, :, :-R, :-R]
        if output_attentions:
            p_last = res["p_last"]
            out["attentions"] = p_last[:, :, :-R, :-R]
            out["attentions_register_tokens"] = p_last[:, :, -R:, :]
            # :614-618 -- the reference sorts every row of every map of the window; here the per-(evaluation, image,
            # head) row maxima come out of the solve (in-kernel, or odevit_jasmin_rowmax on exported maps), and the
            # means over heads / images / maps are taken here
            jt = res["jas_traj"]
            if jt is None and p_traj is not None and p_traj.shape[0] and window > 0:
                jt = ops.jasmin_rowmax(p_traj[-window:], jasmin_k)
            if jt is None:
                out["jasmin_loss"] = self.jasmin_loss([], k=jasmin_k, reduction="mean")
            else:
                out["jasmin_loss"] = jt.mean(dim=2).mean(dim=1).mean()
        if self.add_distillation_token:
            out["logits_dist"] = self.dist_head(final[:, 1])
        if labels is not None:
            out["loss"] = loss if fused_head else F.cross_entropy(out["logits"], labels, label_smoothing=0.05)
        if output_hidden_states:
            out["states"] = states
        if output_control_points:
            out["control_points"] = res["rows"][:, :, :-R]
        self.odefunc.attention_trajectory = []   # :641-643
        return out

    def _forward_adaptive(self, tokens, t, num_eval_steps, cfg, labels, output_hidden_states, output_control_points,
                          output_attentions, temperature, jasmin_k):
        """forward() with `adaptive_solve` set: the trajectory over t comes from the dense output of the per-image
        adaptive solve; the finite-difference bound is taken on it; `nfe` [B] is added to the output.  With
        output_attentions, `attentions` / `attentions_register_tokens` slice each image's last-evaluation map and
        `jasmin_loss` is taken over each image's own window (ops.ode_solve_adaptive's want_p_last / jasmin)."""
        R = self.patch_embed.num_register_tokens
        window = int(self.num_eval_steps * 0.85)                            # :614-618
        res = ops.ode_solve_adaptive(tokens, t, self.odefunc.block.field_spec(self.odefunc.scaler),
                                     self.odefunc.block.field_weights(), cfg["rtol"], cfg["atol"],
                                     first_step=cfg.get("first_step"),
                                     max_num_steps=cfg.get("max_num_steps", ops.DOPRI5_MAX_NUM_STEPS),
                                     differentiable=cfg.get("differentiable", False),
                                     capturable=cfg.get("capturable", False), want_p_last=output_attentions,
                                     jasmin=(window, int(jasmin_k)) if (output_attentions and window > 0) else None)
        states, final = res["states"], res["final"]
        logits = self.head(final[:, 0])
        out = {
            "logits": logits,
            "second_derivative_upper_bound": self.compute_upper_bound_by_second_derivative(R=jasmin_k, L=1 / 2),
            "finite_difference_upper_bound": self.compute_upper_bound_by_fininte_difference(
                states.detach(), 0.5, 1 / self.num_eval_steps),
            "nfe": res["nfe"],
        }
        if output_attentions:
            # per image: its own last evaluation's map, and the JaSMin statistic over its own last min(W, nfe_b)
            # evaluations, averaged over heads and window slots, then over images (the reference's formula when
            # every image has the same evaluations)
            p_last = res["p_last"]
            self.odefunc.block.attentions = p_last
            out["attentions"] = p_last[:, :, :-R, :-R]
            out["attentions_register_tokens"] = p_last[:, :, -R:, :]
            if window > 0:
                out["jasmin_loss"] = ops.adaptive_jasmin_mean(res["jas_ring"], res["jas_count"]).mean()
            else:
                out["jasmin_loss"] = self.jasmin_loss([], k=jasmin_k, reduction="mean")
        if self.add_distillation_token:
            out["logits_dist"] = self.dist_head(final[:, 1])
        if labels is not None:
            out["loss"] = F.cross_entropy(logits, labels, label_smoothing=0.05)
        if output_hidden_states:
            out["states"] = states
        if output_control_points:
            idx = self.get_proportional_control_points_with_temperature(temperature=temperature,
                                                                        num_eval_steps=num_eval_steps)
            out["control_points"] = states[idx][:, :, :-R]
        self.odefunc.attention_trajectory = []
        return out
