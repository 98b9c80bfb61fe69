"""odevit_b200 -- B200-native (sm_100a) implementation of ODE-ViT's hot path: the vector field
f(t, x) evaluated by a fixed-step solver over the integration grid, behind the reference's
nn.Module surface.  See DESIGN.md; the C ABI is include/odevit.h (csrc/libodevit.so)."""
from ._lib import OdevitError, LIB_PATH, launch_count, reset_launch_count  # noqa: F401
from .ops import FieldSpec, NotConvergedError, field_eval, ode_solve, ode_solve_adaptive  # noqa: F401
from .vit_ode import (CenterNorm, L2SelfAttention, MLP, MultiheadSelfAttention, ParallelAttentionMLP,  # noqa: F401
                      PatchEmbed, ViT_ODEFunc, ViTNeuralODE, odeint, odeint_adaptive)
from .macaron import ViTMacaron  # noqa: F401
from . import macaron, time_emb  # noqa: F401
from .teacher import ViTTeacher  # noqa: F401
from . import loss_trainer  # noqa: F401
from .loss_trainer import ImageDistilTrainer  # noqa: F401
from .time_emb import (LearnedSinusoidalPosEmb, ScaleShift, SinusoidalPosEmb, TimeEmbedding,  # noqa: F401
                       attach_time_modulation)

__all__ = ["OdevitError", "LIB_PATH", "FieldSpec", "field_eval", "ode_solve", "ode_solve_adaptive", "odeint_adaptive",
           "NotConvergedError", "CenterNorm", "MLP",
           "MultiheadSelfAttention", "ParallelAttentionMLP", "PatchEmbed", "ViT_ODEFunc", "ViTNeuralODE",
           "odeint", "launch_count", "reset_launch_count", "L2SelfAttention", "ViTMacaron", "macaron", "time_emb",
           "ViTTeacher", "ImageDistilTrainer", "loss_trainer", "SinusoidalPosEmb", "LearnedSinusoidalPosEmb", "TimeEmbedding", "ScaleShift", "attach_time_modulation"]
