"""PyTorch-facing operators over the C ABI: one vector-field evaluation and the fixed-grid solve,
each as a `torch.autograd.Function` whose forward/backward enqueue libodevit.so kernels on the
current CUDA stream.  PyTorch is plumbing here (device memory, streams, autograd graph edges).

Replaces, for CUDA tensors:
  * `ViT_ODEFunc.forward(t, x)`                         models/ode_transformer_gpt.py:317-330
  * `torchdiffeq.odeint(func, y0, t, method=...)`        models/ode_transformer_gpt.py:571-578
  * `torchdiffeq.odeint(..., method="dopri5")` with the error norm taken per image (ode_solve_adaptive)
  * autograd through all three (backprop-through-solver)  train.py:57-67; the adaptive solve's with its accepted
    steps frozen
"""
from __future__ import annotations

import ctypes
import os
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import OdevitError

_vp = ctypes.c_void_p


@dataclass(frozen=True)
class FieldSpec:
    """Static description of the vector field (everything but the batch)."""
    dim: int
    heads: int
    hidden: int
    scaler: float
    variant: int = _lib.FIELD_PARALLEL
    precision: str = "bf16"
    backward: str = "auto"   # "tape" | "recompute" | "auto" (tape when it fits TAPE_BUDGET_FRACTION of free HBM)
    # training-mode dropout (0 = off); masks come from a counter-based generator keyed by `seed`
    attn_drop: float = 0.0
    proj_drop: float = 0.0
    mlp_drop: float = 0.0
    seed: int = 0
    # a device-resident seed (int64[1] CUDA tensor, see `DropState`) read at kernel time instead of `seed`: what makes
    # dropout work under CUDA-graph replay (the captured launches hold the address, not the value)
    seed_dev: Optional[torch.Tensor] = None

    def desc(self, batch: int, tokens: int) -> _lib.Desc:
        d = _lib.Desc()
        d.abi_version = _lib.ABI_VERSION
        d.batch, d.tokens, d.dim, d.heads, d.hidden = batch, tokens, self.dim, self.heads, self.hidden
        d.variant = self.variant
        d.precision = _lib.PRECISIONS[self.precision]
        d.scaler = float(self.scaler)
        d.attn_drop, d.proj_drop, d.mlp_drop = float(self.attn_drop), float(self.proj_drop), float(self.mlp_drop)
        d.drop_seed_lo, d.drop_seed_hi = self.seed & 0xFFFFFFFF, (self.seed >> 32) & 0xFFFFFFFF
        d.drop_seed_dev = self.seed_dev.data_ptr() if (self.seed_dev is not None and self.has_dropout) else None
        return d

    @property
    def has_dropout(self) -> bool:
        return self.attn_drop > 0 or self.proj_drop > 0 or self.mlp_drop > 0


def _dp_rank() -> int:
    try:
        import torch.distributed as dist
        return dist.get_rank() if (dist.is_available() and dist.is_initialized()) else 0
    except Exception:  # noqa: BLE001
        return 0


def draw_seed() -> int:
    """A fresh 64-bit mask seed from PyTorch's default CPU generator (so `torch.manual_seed` makes
    dropout reproducible, as it does in the reference), mixed with the data-parallel rank: replicas that
    seeded identically still draw different masks (rank 0 is unchanged)."""
    hi, lo = torch.randint(0, 2 ** 31 - 1, (2,)).tolist()
    return ((int(hi) << 32) | int(lo)) ^ ((_dp_rank() * 0x9E3779B97F4A7C15) & 0x7FFFFFFFFFFFFFFF)


class DropState:
    """Device-resident dropout seed of one vector-field module: int64[3] = (base seed, step counter, seed of the
    current step).  `next_seed()` advances it with a 1-thread kernel (`odevit_drop_state_advance`) and returns a
    device copy of the new step seed: the forward AND the backward launches of that step read the copy, later steps
    get their own.  Everything is a device operation on fixed addresses, so a step captured in a CUDA graph draws
    fresh masks at every replay (PyTorch's own Philox capture works the same way).  The base seed comes from
    `draw_seed()` (hence `torch.manual_seed`) mixed with the data-parallel rank: replicas draw different masks."""

    def __init__(self, device: torch.device):
        self.state = torch.tensor([draw_seed() & 0x7FFFFFFFFFFFFFFF, 0, 0], dtype=torch.int64, device=device)

    def next_seed(self) -> torch.Tensor:
        with torch.cuda.device(self.state.device):
            st = _lib.lib().odevit_drop_state_advance(_vp(self.state.data_ptr()), _stream())
        _lib.check(st, "odevit_drop_state_advance")
        return self.state[2:3].clone()


# ---------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------
def _require_cuda(t: torch.Tensor, what: str) -> torch.Tensor:
    if not t.is_cuda:
        raise OdevitError(f"{what} is on {t.device}: odevit_b200 runs on CUDA devices only (no CPU fallback)")
    if t.dtype != torch.float32:
        raise OdevitError(f"{what} must be float32, got {t.dtype}")
    return t.contiguous()


def _ptr(t: Optional[torch.Tensor]):
    return _vp(t.data_ptr()) if t is not None else None


_WS_CACHE: Dict[Tuple[int, int, int, bool], torch.Tensor] = {}


def _workspace(desc: _lib.Desc, kind: int, method: int, device: torch.device):
    """A cached, 1024-byte aligned device workspace per (device, kind, STREAM, deterministic mode).

    Keyed by the current stream so that (a) two streams never share scratch memory and (b) a CUDA-graph capture
    -- which runs on its own capture stream -- allocates its workspace from the graph's private pool: the graph
    then owns the buffer its kernels have baked in, and nothing an eager call does later (a larger batch, another
    method) can free or reuse it under a replay.  A buffer that must grow is replaced, never resized in place;
    `GraphedTrainStep` additionally pins the buffers that were live when it captured."""
    det = _sync_deterministic()   # (the deterministic mode's backward layouts carry partial-sum scratch)
    n = _lib.lib().odevit_workspace_bytes(ctypes.byref(desc), kind, method)
    if n == 0:
        _lib.check(-1, "odevit_workspace_bytes")
    dev = device.index if device.index is not None else torch.cuda.current_device()
    key = (dev, kind, int(torch.cuda.current_stream(device).cuda_stream), det)
    buf = _WS_CACHE.get(key)
    if buf is None or buf.numel() < n + 1024:
        buf = torch.empty(int(n * 1.05) + 2048, dtype=torch.uint8, device=device)
        _WS_CACHE[key] = buf
    base = buf.data_ptr()
    aligned = (base + 1023) & ~1023
    return buf, _vp(aligned), buf.numel() - (aligned - base)


def live_workspaces() -> List[torch.Tensor]:
    """The workspace buffers currently cached (a captured graph keeps these alive: see graphs.py)."""
    return list(_WS_CACHE.values())


def free_workspaces() -> None:
    _WS_CACHE.clear()


TAPE_BUDGET_FRACTION = float(os.environ.get("ODEVIT_TAPE_FRACTION", "0.5"))
_TAPE_FITS: Dict[Tuple[Optional[int], int], bool] = {}


def _alloc_tape(desc: _lib.Desc, method: int, n_grid: int, mode: str, device: torch.device):
    """The forward's record of per-evaluation intermediates for the reverse sweep (what autograd's saved
    tensors are in the reference), or None -> the reverse sweep recomputes each step."""
    if mode == "recompute" or n_grid < 2:
        return None
    return _tape_buffer(int(_lib.lib().odevit_tape_bytes(ctypes.byref(desc), method, n_grid)), mode, device)


def _tape_buffer(n: int, mode: str, device: torch.device):
    """A tape of n bytes under the backward mode `mode` ("tape" | "recompute" | "auto": when it fits
    TAPE_BUDGET_FRACTION of the free memory), or None."""
    if mode == "recompute" or n == 0:
        return None
    if mode == "auto":
        key = (device.index, n)
        ok = _TAPE_FITS.get(key)
        if ok is None:   # decided once per (device, size): the driver query is not free
            free, _total = torch.cuda.mem_get_info(device)
            reusable = torch.cuda.memory_reserved(device) - torch.cuda.memory_allocated(device)
            ok = _TAPE_FITS[key] = bool(n <= TAPE_BUDGET_FRACTION * (free + reusable))
        if not ok:
            return None
    try:
        return torch.empty(n + 1024, dtype=torch.uint8, device=device)
    except torch.OutOfMemoryError:
        if mode == "tape":
            raise
        _TAPE_FITS[(device.index, n)] = False
        return None


def _aligned(buf: Optional[torch.Tensor]):
    if buf is None:
        return None, 0
    base = buf.data_ptr()
    al = (base + 1023) & ~1023
    return _vp(al), buf.numel() - (al - base)


_DETERMINISTIC = [False]   # what the library was last told


def _sync_deterministic() -> bool:
    """Mirror torch.are_deterministic_algorithms_enabled() into the library (odevit_set_deterministic), calling the
    setter only when the value changes.  On, the backward kernels sum their reductions in a fixed order instead of
    through atomics: identical inputs give bitwise-identical gradients (same build, GPU model and SM count)."""
    on = torch.are_deterministic_algorithms_enabled()
    if on != _DETERMINISTIC[0]:
        _lib.check(_lib.lib().odevit_set_deterministic(int(on)), "odevit_set_deterministic")
        _DETERMINISTIC[0] = on
    return on


def _stream() -> _vp:
    # every library call takes its stream from here: the place to bring the deterministic mode up to date
    _sync_deterministic()
    return _vp(torch.cuda.current_stream().cuda_stream)


def _pack_weights(names: Sequence[str], tensors: Sequence[torch.Tensor]):
    w = _lib.Weights()
    keep = []
    for n, t in zip(names, tensors):
        if t is None:
            continue
        t = _require_cuda(t.detach(), f"weight {n}")
        keep.append(t)
        setattr(w, n, t.data_ptr())
    return w, keep


def _alloc_grads(names: Sequence[str], tensors: Sequence[torch.Tensor], needs: Sequence[bool]):
    """Zero-filled gradient accumulators: ONE flat buffer (one memset) carved into per-weight views."""
    g = _lib.WeightGrads()
    want = [(t is not None and need and n not in _lib.MOD_FIELDS) for n, t, need in zip(names, tensors, needs)]
    sizes = [((t.numel() + 63) // 64) * 64 if w else 0 for t, w in zip(tensors, want)]   # 256-byte aligned views
    out: List[Optional[torch.Tensor]] = [None] * len(want)
    if not any(want):
        return g, out
    dev = next(t for t, w in zip(tensors, want) if w).device
    flat = torch.zeros(sum(sizes), dtype=torch.float32, device=dev)
    off = 0
    for i, (n, t, w) in enumerate(zip(names, tensors, want)):
        if not w:
            continue
        gt = flat[off:off + t.numel()].view(t.shape)
        off += sizes[i]
        setattr(g, n, gt.data_ptr())
        out[i] = gt
    return g, out


# ---------------------------------------------------------------------------------------------
# one field evaluation
# ---------------------------------------------------------------------------------------------
class _FieldEval(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, spec: FieldSpec, want_p: bool, names: Tuple[str, ...], *weights):
        x = _require_cuda(x, "x")
        B, N, D = x.shape
        desc = spec.desc(B, N)
        w, keep = _pack_weights(names, weights)
        dx = torch.empty_like(x)
        p = torch.empty(B, spec.heads, N, N, device=x.device, dtype=torch.float32) if want_p else None
        buf, ws, ws_bytes = _workspace(desc, _lib.WS_FIELD, _lib.EULER, x.device)
        with torch.cuda.device(x.device):
            st = _lib.lib().odevit_field_fwd(ctypes.byref(desc), ctypes.byref(w), _ptr(x), _ptr(dx), _ptr(p),
                                             ws, ws_bytes, _stream())
        _lib.check(st, "odevit_field_fwd")
        ctx.spec, ctx.names, ctx.want_p = spec, names, want_p
        ctx.save_for_backward(x, *[t for t in weights])
        ctx.set_materialize_grads(False)
        if want_p:
            return dx, p
        return dx, x.new_empty(0)

    @staticmethod
    def backward(ctx, g_dx, g_p):
        x, *weights = ctx.saved_tensors
        spec, names = ctx.spec, ctx.names
        B, N, D = x.shape
        desc = spec.desc(B, N)
        w, keep = _pack_weights(names, weights)
        needs = ctx.needs_input_grad[4:]
        gw, gts = _alloc_grads(names, weights, needs)
        if g_dx is None:
            g_dx = torch.zeros_like(x)
        g_dx = _require_cuda(g_dx, "g_dx")
        if g_p is not None and (not ctx.want_p or g_p.numel() == 0):
            g_p = None
        if g_p is not None:
            g_p = _require_cuda(g_p, "g_p")
        g_x = torch.empty_like(x)
        buf, ws, ws_bytes = _workspace(desc, _lib.WS_SOLVE_BWD, _lib.EULER, x.device)
        with torch.cuda.device(x.device):
            st = _lib.lib().odevit_field_bwd(ctypes.byref(desc), ctypes.byref(w), _ptr(x), _ptr(g_dx), _ptr(g_p),
                                             _ptr(g_x), ctypes.byref(gw), ws, ws_bytes, _stream())
        _lib.check(st, "odevit_field_bwd")
        return (g_x if ctx.needs_input_grad[0] else None, None, None, None, *gts)


def field_eval(x: torch.Tensor, spec: FieldSpec, weights: Dict[str, Optional[torch.Tensor]],
               want_p: bool = True):
    """dx, P = f(x).  `weights` maps the odevit_weights field names to fp32 CUDA tensors."""
    names = tuple(k for k, v in weights.items() if v is not None)
    dx, p = _FieldEval.apply(x, spec, want_p, names, *[weights[k] for k in names])
    return dx, (p if want_p else None)


# ---------------------------------------------------------------------------------------------
# the fixed-grid solve
# ---------------------------------------------------------------------------------------------
_ROW_INDEX_CACHE: Dict[Tuple[Tuple[int, ...], torch.device], torch.Tensor] = {}


def _row_index_tensor(row_index: Tuple[int, ...], device: torch.device) -> torch.Tensor:
    """Device copy of a control-point index list, made once: indexing with a Python list uploads it on every
    call (a pageable host-to-device copy: a stall in eager mode, illegal inside a CUDA-graph capture)."""
    key = (row_index, device)
    t = _ROW_INDEX_CACHE.get(key)
    if t is None:
        t = torch.tensor(row_index, dtype=torch.long, device=device)
        _ROW_INDEX_CACHE[key] = t
    return t


def _solve_grid_outputs(x0: torch.Tensor, t: torch.Tensor, spec: FieldSpec, method: str, want_p_last: bool,
                        jas: Optional[Tuple[int, int]]):
    """What both fixed-grid solves pass the same way: (T, the host grid as a C array, the evaluation count, p_last
    [B,H,N,N] | None, (jas_traj [E,B,H] | None, its first evaluation, k))."""
    B, N, _ = x0.shape
    T = int(t.numel())
    t_c = (ctypes.c_float * T)(*t.detach().to("cpu", torch.float32).contiguous().tolist())
    n_evals = (T - 1) * _lib.STAGES[method]
    p_last = (torch.empty(B, spec.heads, N, N, device=x0.device, dtype=torch.float32)
              if (want_p_last and n_evals > 0) else None)
    jas_traj, jas_first, jas_k = None, 0, 0
    if jas is not None and n_evals > 0:
        jas_first, jas_k = max(0, min(int(jas[0]), n_evals)), int(jas[1])
        if n_evals - jas_first > 0:
            jas_traj = torch.empty(n_evals - jas_first, B, spec.heads, device=x0.device, dtype=torch.float32)
    return T, t_c, n_evals, p_last, (jas_traj, jas_first, jas_k)


class _OdeSolve(torch.autograd.Function):
    """(states, final, rows, p_last, p_traj) = solve(x0).

    * `states` [T,B,N,D]: what `odeint` returns;
    * `final` [B,N,D]: states[-1] as its own output, so a loss on the final state does not make
      autograd materialise a dense [T,B,N,D] cotangent;
    * `rows` [Q,B,N,D]: states[row_index] (the control points), same reason;
    * `p_last` [B,H,N,N]: attention map of the last field evaluation (`block.attentions`);
    * `p_traj` [E,B,H,N,N]: maps of the last E evaluations (`attention_trajectory`, detached).
    """

    @staticmethod
    def forward(ctx, x0, spec: FieldSpec, method: str, t_host: torch.Tensor, row_index: Tuple[int, ...],
                want_p_last: bool, p_traj_first: Optional[int], jas: Optional[Tuple[int, int]],
                names: Tuple[str, ...], track: bool, *weights):
        x0 = _require_cuda(x0, "x0")
        B, N, D = x0.shape
        desc = spec.desc(B, N)
        w, keep = _pack_weights(names, weights)
        T, t_c, n_evals, p_last, (jas_traj, jas_first, jas_k) = _solve_grid_outputs(x0, t_host, spec, method,
                                                                                   want_p_last, jas)
        states = torch.empty(T, B, N, D, device=x0.device, dtype=torch.float32)
        final = torch.empty(B, N, D, device=x0.device, dtype=torch.float32)
        p_traj = None
        first = 0
        if p_traj_first is not None and n_evals > 0:
            first = max(0, min(int(p_traj_first), n_evals))
            if n_evals - first > 0:
                p_traj = torch.empty(n_evals - first, B, spec.heads, N, N, device=x0.device, dtype=torch.float32)
        buf, ws, ws_bytes = _workspace(desc, _lib.WS_SOLVE_FWD, _lib.METHODS[method], x0.device)
        # `track`: a backward pass can follow (grad mode on and something requires grad); decided by the
        # caller, because inside forward() grad mode is always off and needs_input_grad ignores no_grad()
        tape = _alloc_tape(desc, _lib.METHODS[method], T, spec.backward, x0.device) if track else None
        tape_p, tape_n = _aligned(tape)
        with torch.cuda.device(x0.device):
            st = _lib.lib().odevit_solve_fwd(ctypes.byref(desc), ctypes.byref(w), _lib.METHODS[method], _ptr(x0),
                                             t_c, T, _ptr(states), _ptr(final), _ptr(p_last), _ptr(p_traj), first,
                                             _ptr(jas_traj), jas_first, jas_k, tape_p, tape_n, ws, ws_bytes, _stream())
        _lib.check(st, "odevit_solve_fwd")
        ctx.tape = tape
        rows = states.index_select(0, _row_index_tensor(tuple(row_index), states.device)) if len(row_index) else x0.new_empty(0)
        ctx.spec, ctx.method, ctx.names, ctx.row_index = spec, method, names, tuple(row_index)
        ctx.t_c, ctx.T = t_c, T
        ctx.has_p_last = p_last is not None
        ctx.save_for_backward(states, *weights)
        ctx.set_materialize_grads(False)
        empty = x0.new_empty(0)
        out_p_traj = p_traj if p_traj is not None else empty
        out_jas = jas_traj if jas_traj is not None else x0.new_empty(0)
        ctx.mark_non_differentiable(out_p_traj, out_jas)
        return states, final, rows, (p_last if p_last is not None else empty), out_p_traj, out_jas

    @staticmethod
    def backward(ctx, g_states, g_final, g_rows, g_p_last, _g_p_traj, _g_jas):
        states, *weights = ctx.saved_tensors
        spec, method, names = ctx.spec, ctx.method, ctx.names
        T, B, N, D = states.shape
        desc = spec.desc(B, N)
        w, keep = _pack_weights(names, weights)
        needs = ctx.needs_input_grad[10:]
        gw, gts = _alloc_grads(names, weights, needs)
        parts, index = [], []
        if g_final is not None:
            parts.append(_require_cuda(g_final, "g_final").unsqueeze(0))
            index.append(T - 1)
        if g_rows is not None and g_rows.numel() and len(ctx.row_index):
            parts.append(_require_cuda(g_rows, "g_rows"))
            index.extend(ctx.row_index)
        g_rows_all = torch.cat(parts, 0).contiguous() if parts else None
        idx_c = (ctypes.c_int32 * max(1, len(index)))(*index)
        if g_states is not None:
            g_states = _require_cuda(g_states, "g_states")
        if g_p_last is not None and (not ctx.has_p_last or g_p_last.numel() == 0):
            g_p_last = None
        if g_p_last is not None:
            g_p_last = _require_cuda(g_p_last, "g_p_last")
        g_x0 = torch.empty(B, N, D, device=states.device, dtype=torch.float32)
        buf, ws, ws_bytes = _workspace(desc, _lib.WS_SOLVE_BWD, _lib.METHODS[method], states.device)
        tape_p, tape_n = _aligned(ctx.tape)
        with torch.cuda.device(states.device):
            st = _lib.lib().odevit_solve_bwd(ctypes.byref(desc), ctypes.byref(w), _lib.METHODS[method], ctx.t_c, T,
                                             _ptr(states), _ptr(g_states), _ptr(g_rows_all), idx_c, len(index),
                                             _ptr(g_p_last), _ptr(g_x0), ctypes.byref(gw), tape_p, tape_n,
                                             ws, ws_bytes, _stream())
        _lib.check(st, "odevit_solve_bwd")
        ctx.tape = None
        return (g_x0 if ctx.needs_input_grad[0] else None, None, None, None, None, None, None, None, None, None, *gts)


def ode_solve(x0: torch.Tensor, t: torch.Tensor, spec: FieldSpec, method: str,
              weights: Dict[str, Optional[torch.Tensor]], row_index: Sequence[int] = (),
              want_p_last: bool = False, p_traj_first: Optional[int] = None,
              jasmin: Optional[Tuple[int, int]] = None):
    """Fixed-grid solve of dx/dt = f(x) over the grid `t` (euler | midpoint | rk4 = 3/8 rule).
    `jasmin=(first_eval, k)`: the JaSMin statistic [E,B,H] of the maps of evaluations >= first_eval, without
    exporting them (`jas_traj`).

    Returns dict(states, final, rows, p_last, p_traj, jas_traj); see `_OdeSolve`."""
    if method not in _lib.METHODS:
        raise ValueError(f"unsupported solver {method!r}; fixed-grid euler | midpoint | rk4 are built")
    if t.ndim != 1 or t.numel() < 1:
        raise ValueError("t must be one dimensional")
    names = tuple(k for k, v in weights.items() if v is not None)
    track = torch.is_grad_enabled() and (x0.requires_grad or any(weights[k].requires_grad for k in names))
    states, final, rows, p_last, p_traj, jas_traj = _OdeSolve.apply(
        x0, spec, method, t, tuple(int(i) for i in row_index), want_p_last, p_traj_first, jasmin, names, track,
        *[weights[k] for k in names])
    return {"states": states, "final": final, "rows": rows if len(row_index) else None,
            "p_last": p_last if p_last.numel() else None, "p_traj": p_traj if p_traj.numel() else None,
            "jas_traj": jas_traj if jas_traj.numel() else None}


class _ExtractMass(torch.autograd.Function):
    """odevit_extract_mass_fwd / _bwd: the L1-attention-loss front-end (loss_trainer.py:80-117) as one launch each way."""

    @staticmethod
    def forward(ctx, rows, threshold: float, smooth: bool, scale_factor: float, want_mask: bool):
        rows = _require_cuda(rows, "attn_rows")
        B, H, n = rows.shape
        mean = torch.empty(B, n, device=rows.device, dtype=torch.float32)
        heads = torch.empty(B, H, n, device=rows.device, dtype=torch.float32)
        mask = torch.empty(B, n, device=rows.device, dtype=torch.float32) if want_mask else None
        with torch.cuda.device(rows.device):
            st = _lib.lib().odevit_extract_mass_fwd(_ptr(rows), B, H, n, float(threshold), int(bool(smooth)), float(scale_factor),
                                                    _ptr(mean), _ptr(heads), _ptr(mask), _stream())
        _lib.check(st, "odevit_extract_mass_fwd")
        ctx.save_for_backward(rows)
        ctx.cfg = (float(threshold), int(bool(smooth)), float(scale_factor))
        ctx.set_materialize_grads(False)
        if mask is None:
            mask = rows.new_empty(0)
        ctx.mark_non_differentiable(mask)
        return mean, heads, mask

    @staticmethod
    def backward(ctx, g_mean, g_heads, _g_mask):
        (rows,) = ctx.saved_tensors
        if g_mean is None and g_heads is None:
            return None, None, None, None, None
        B, H, n = rows.shape
        g_mean = _require_cuda(g_mean, "g_mean") if g_mean is not None else None
        g_heads = _require_cuda(g_heads, "g_heads") if g_heads is not None else None
        g_rows = torch.empty_like(rows)
        thr, smooth, scale = ctx.cfg
        with torch.cuda.device(rows.device):
            st = _lib.lib().odevit_extract_mass_bwd(_ptr(rows), B, H, n, thr, smooth, scale, _ptr(g_mean), _ptr(g_heads),
                                                    _ptr(g_rows), _stream())
        _lib.check(st, "odevit_extract_mass_bwd")
        return g_rows, None, None, None, None


def extract_mass(attn_rows: torch.Tensor, threshold: float = 0.8, smooth: bool = True, scale_factor: float = 40.0,
                 return_mask: bool = False):
    """loss_trainer.py:80-117 on a CUDA tensor [B, heads, n = side^2]: (mean over heads [B,side,side], per head
    [B,heads,side,side], mean mask [B,side,side] | None), differentiable (csrc/mass.cu)."""
    B, H, n = attn_rows.shape
    side = int(n ** 0.5 + 0.5)
    mean, heads, mask = _ExtractMass.apply(attn_rows.contiguous().float(), threshold, smooth, scale_factor, return_mask)
    return mean.view(B, side, side), heads.view(B, H, side, side), (mask.view(B, side, side) if return_mask else None)


def solve_uses_resident(spec: FieldSpec, batch: int, tokens: int, method: str, n_grid: int) -> bool:
    """True when the inference solve of this shape runs in the on-chip-state kernel (odevit_solve_uses_resident)."""
    desc = spec.desc(batch, tokens)
    return bool(_lib.lib().odevit_solve_uses_resident(ctypes.byref(desc), _lib.METHODS[method], int(n_grid)))


@torch.no_grad()
def ode_solve_lean(x0: torch.Tensor, t: torch.Tensor, spec: FieldSpec, method: str,
                   weights: Dict[str, Optional[torch.Tensor]], row_index: Sequence[int] = (),
                   want_p_last: bool = False, jasmin: Optional[Tuple[int, int]] = None):
    """Inference solve WITHOUT the [T,B,N,D] trajectory (odevit_solve_fwd_lean): the reference materialises `states`
    for every call but returns them only on request (ode_transformer_gpt.py:628-630); what it always needs from them
    is the finite-difference bound (:529-543), formed here inside the solve, and the control-point rows (:632-639),
    written straight into `rows`.  No autograd (the reverse sweep needs the trajectory).

    Returns dict(final [B,N,D], rows [Q,B,N,D] | None, fd_max [B,N] = max_j,d |s[j+2] - 2 s[j+1] + s[j]|,
    p_last, jas_traj)."""
    if method not in _lib.METHODS:
        raise ValueError(f"unsupported solver {method!r}; fixed-grid euler | midpoint | rk4 are built")
    names = tuple(k for k, v in weights.items() if v is not None)
    x0 = _require_cuda(x0.detach(), "x0")
    B, N, D = x0.shape
    desc = spec.desc(B, N)
    w, keep = _pack_weights(names, [weights[k].detach() for k in names])
    T, t_c, n_evals, p_last, (jas_traj, jas_first, jas_k) = _solve_grid_outputs(x0, t, spec, method, want_p_last, jasmin)
    final = torch.empty(B, N, D, device=x0.device, dtype=torch.float32)
    row_index = [int(i) for i in row_index]
    rows = torch.empty(len(row_index), B, N, D, device=x0.device, dtype=torch.float32) if row_index else None
    idx_c = (ctypes.c_int32 * max(1, len(row_index)))(*row_index)
    fd_max = torch.empty(B, N, device=x0.device, dtype=torch.float32)
    buf, ws, ws_bytes = _workspace(desc, _lib.WS_SOLVE_FWD, _lib.METHODS[method], x0.device)
    with torch.cuda.device(x0.device):
        st = _lib.lib().odevit_solve_fwd_lean(ctypes.byref(desc), ctypes.byref(w), _lib.METHODS[method], _ptr(x0), t_c, T,
                                              _ptr(final), _ptr(rows), idx_c, len(row_index), _ptr(fd_max), _ptr(p_last),
                                              _ptr(jas_traj), jas_first, jas_k, ws, ws_bytes, _stream())
    _lib.check(st, "odevit_solve_fwd_lean")
    return {"states": None, "final": final, "rows": rows, "fd_max": fd_max, "p_last": p_last, "p_traj": None,
            "jas_traj": jas_traj}


class NotConvergedError(OdevitError):
    """The adaptive solve stopped: an image exceeded max_num_steps, met a non-finite error ratio or a dt that no longer
    advances t (the message names the image)."""


DOPRI5_MAX_NUM_STEPS = 2 ** 31 - 1   # torchdiffeq's default


ADAPTIVE_STEP_CAP = 1024   # first size of the accepted-step record of a differentiable adaptive solve (grown 4x on demand)


def _adaptive_attn_outputs(x0, spec: FieldSpec, want_p_last: bool, jasmin: Optional[Tuple[int, int]]):
    """The attention outputs of an adaptive solve: (p_last [B,H,N,N] | None, (jas_ring [W,B,H], jas_count [B] int32, W,
    k) | None) for jasmin = (W, k)."""
    B, N, _ = x0.shape
    if (want_p_last or jasmin is not None) and spec.variant == _lib.FIELD_MACARON:
        raise OdevitError("MACARON exposes no attention map (macaron.py:60-65): no p_last / JaSMin window")
    p_last = torch.empty(B, spec.heads, N, N, device=x0.device, dtype=torch.float32) if want_p_last else None
    jas = None
    if jasmin is not None:
        W, k = int(jasmin[0]), int(jasmin[1])
        if W < 1:
            raise ValueError(f"jasmin window must be >= 1, got {W}")
        jas = (torch.empty(W, B, spec.heads, device=x0.device, dtype=torch.float32),
               torch.empty(B, device=x0.device, dtype=torch.int32), W, k)
    return p_last, jas


def _adaptive_call(x0, t_c, T: int, spec: FieldSpec, names, weights, rtol: float, atol: float, fs: float,
                   max_num_steps: int, record=None, attn=None):
    """One odevit_solve_adaptive call, or odevit_solve_adaptive_record with record = (cap, t0, dt, out), or, with
    attn = (p_last | None, jas | None) from _adaptive_attn_outputs, odevit_solve_adaptive_attn (record optional).
    Returns (status, states [T,B,N,D], counts [3,B] int32 = nfe, accepted, rejected)."""
    B, N, D = x0.shape
    desc = spec.desc(B, N)
    w, keep = _pack_weights(names, weights)
    states = torch.empty(T, B, N, D, device=x0.device, dtype=torch.float32)
    counts = torch.zeros(3, B, device=x0.device, dtype=torch.int32)
    buf, ws, ws_bytes = _workspace(desc, _lib.WS_SOLVE_ADAPTIVE, 0, x0.device)
    with torch.cuda.device(x0.device):
        if attn is not None:
            p_last, jas = attn
            cap, t0, dt, out = record if record is not None else (0, None, None, None)
            ring, jcount, W, k = jas if jas is not None else (None, None, 0, 0)
            st = _lib.lib().odevit_solve_adaptive_attn(ctypes.byref(desc), ctypes.byref(w), _ptr(x0), t_c, T,
                                                       float(rtol), float(atol), fs, int(max_num_steps), _ptr(states),
                                                       _ptr(counts[0]), _ptr(counts[1]), _ptr(counts[2]), int(cap),
                                                       _ptr(t0), _ptr(dt), _ptr(out), _ptr(p_last), int(k), int(W),
                                                       _ptr(ring), _ptr(jcount), ws, ws_bytes, _stream())
        elif record is None:
            st = _lib.lib().odevit_solve_adaptive(ctypes.byref(desc), ctypes.byref(w), _ptr(x0), t_c, T, float(rtol),
                                                  float(atol), fs, int(max_num_steps), _ptr(states), _ptr(counts[0]),
                                                  _ptr(counts[1]), _ptr(counts[2]), ws, ws_bytes, _stream())
        else:
            cap, t0, dt, out = record
            st = _lib.lib().odevit_solve_adaptive_record(ctypes.byref(desc), ctypes.byref(w), _ptr(x0), t_c, T,
                                                         float(rtol), float(atol), fs, int(max_num_steps), _ptr(states),
                                                         _ptr(counts[0]), _ptr(counts[1]), _ptr(counts[2]), int(cap),
                                                         _vp(t0.data_ptr()), _vp(dt.data_ptr()), _vp(out.data_ptr()),
                                                         ws, ws_bytes, _stream())
    return st, states, counts


_ADAPTIVE_STATUS = {1: "max_num_steps ({max_steps}) exceeded before t_out[-1]", 2: "non-finite error ratio",
                    3: "underflow in dt (t + dt == t)"}


def _adaptive_resident_call(x0, t_c, T: int, spec: FieldSpec, names, weights, rtol: float, atol: float, fs: float,
                            max_num_steps: int):
    """One odevit_solve_adaptive_resident call (enqueued only: no synchronisation).
    Returns (states [T,B,N,D], counts [4,B] int32 = nfe, accepted, rejected, status)."""
    B, N, D = x0.shape
    desc = spec.desc(B, N)
    w, keep = _pack_weights(names, weights)
    states = torch.empty(T, B, N, D, device=x0.device, dtype=torch.float32)
    counts = torch.empty(4, B, device=x0.device, dtype=torch.int32)
    buf, ws, ws_bytes = _workspace(desc, _lib.WS_SOLVE_ADAPTIVE_RESIDENT, 0, x0.device)
    with torch.cuda.device(x0.device):
        st = _lib.lib().odevit_solve_adaptive_resident(ctypes.byref(desc), ctypes.byref(w), _ptr(x0), t_c, T,
                                                       float(rtol), float(atol), fs, int(max_num_steps), _ptr(states),
                                                       _ptr(counts[0]), _ptr(counts[1]), _ptr(counts[2]),
                                                       _ptr(counts[3]), ws, ws_bytes, _stream())
    _lib.check(st, "odevit_solve_adaptive_resident")
    return states, counts


def _adaptive_check(st: int, what: str) -> None:
    if st == _lib.ERR_NOT_CONVERGED:
        raise NotConvergedError(_lib.lib().odevit_last_error_string().decode("utf-8", "replace"))
    _lib.check(st, what)


class _AdaptiveSolve(torch.autograd.Function):
    """(states, counts, p_last, jas_ring, jas_count) = the adaptive solve of x0; its backward is
    odevit_solve_adaptive_bwd (odevit_solve_adaptive_bwd_attn with a cotangent of p_last) over the accepted steps the
    forward recorded (frozen: the step sizes, the output times' positions in them and the rejected attempts carry no
    gradient).  p_last, jas_ring, jas_count are empty unless asked for (want_p_last, jasmin); the window is not
    differentiable."""

    @staticmethod
    def forward(ctx, x0, spec: FieldSpec, t_c, T: int, rtol: float, atol: float, fs: float, max_num_steps: int,
                want_p_last: bool, jasmin: Optional[Tuple[int, int]], names: Tuple[str, ...], *weights):
        B = x0.shape[0]
        cap = max(1, min(int(max_num_steps), int(ADAPTIVE_STEP_CAP)))
        while True:
            rec = (cap, torch.empty(cap, B, device=x0.device, dtype=torch.float64),
                   torch.empty(cap, B, device=x0.device, dtype=torch.float64),
                   torch.empty(cap, B, device=x0.device, dtype=torch.int32))
            attn = _adaptive_attn_outputs(x0, spec, want_p_last, jasmin) if (want_p_last or jasmin) else None
            st, states, counts = _adaptive_call(x0, t_c, T, spec, names, weights, rtol, atol, fs, max_num_steps, rec,
                                                attn)
            # a full record: the solve is deterministic, so a larger one gives the same result
            if st == _lib.ERR_WORKSPACE and cap < max_num_steps and b"step record" in _lib.lib().odevit_last_error_string():
                cap = min(4 * cap, int(max_num_steps))
                continue
            break
        _adaptive_check(st, "odevit_solve_adaptive_record")
        ctx.spec, ctx.names, ctx.t_c, ctx.T, ctx.cap = spec, names, t_c, T, cap
        ctx.n_steps = counts[1].cpu().tolist()   # (the solve has synchronised already)
        ctx.save_for_backward(x0, rec[1], rec[2], rec[3], *weights)
        empty = x0.new_empty(0)
        p_last, jas = attn if attn is not None else (None, None)
        ctx.has_p_last = p_last is not None
        ring, jcount = (jas[0], jas[1]) if jas is not None else (empty, empty.int())
        ctx.mark_non_differentiable(counts, ring, jcount)
        ctx.set_materialize_grads(False)
        return states, counts, (p_last if p_last is not None else empty), ring, jcount

    @staticmethod
    def backward(ctx, g_states, _g_counts, g_p_last, _g_ring, _g_jcount):
        x0, step_t0, step_dt, step_out, *weights = ctx.saved_tensors
        spec, names = ctx.spec, ctx.names
        B, N, D = x0.shape
        if g_p_last is not None and (not ctx.has_p_last or g_p_last.numel() == 0):
            g_p_last = None
        if g_states is None and g_p_last is None:
            return (None,) * (11 + len(weights))
        gw, gts = _alloc_grads(names, weights, ctx.needs_input_grad[11:])
        if g_states is None:
            g_states = torch.zeros(ctx.T, B, N, D, device=x0.device, dtype=torch.float32)
        g_states = _require_cuda(g_states, "g_states")
        desc = spec.desc(B, N)
        w, keep = _pack_weights(names, weights)
        S = max(ctx.n_steps)
        ckpt = torch.empty(S + 1, B, N, D, device=x0.device, dtype=torch.float32)
        tape = _tape_buffer(int(_lib.lib().odevit_adaptive_tape_bytes(ctypes.byref(desc), S)), spec.backward, x0.device)
        tape_p, tape_n = _aligned(tape)
        g_x0 = torch.empty_like(x0)
        n_c = (ctypes.c_int32 * B)(*ctx.n_steps)
        buf, ws, ws_bytes = _workspace(desc, _lib.WS_SOLVE_ADAPTIVE_BWD, 0, x0.device)
        with torch.cuda.device(x0.device):
            if g_p_last is None:
                st = _lib.lib().odevit_solve_adaptive_bwd(ctypes.byref(desc), ctypes.byref(w), _ptr(x0), ctx.t_c, ctx.T,
                                                          _vp(step_t0.data_ptr()), _vp(step_dt.data_ptr()),
                                                          _vp(step_out.data_ptr()), ctx.cap, n_c, _ptr(g_states),
                                                          _ptr(g_x0), ctypes.byref(gw), _ptr(ckpt), tape_p, tape_n, ws,
                                                          ws_bytes, _stream())
            else:
                g_p_last = _require_cuda(g_p_last, "g_p_last")
                st = _lib.lib().odevit_solve_adaptive_bwd_attn(ctypes.byref(desc), ctypes.byref(w), _ptr(x0), ctx.t_c,
                                                               ctx.T, _vp(step_t0.data_ptr()), _vp(step_dt.data_ptr()),
                                                               _vp(step_out.data_ptr()), ctx.cap, n_c, _ptr(g_states),
                                                               _ptr(g_p_last), _ptr(g_x0), ctypes.byref(gw),
                                                               _ptr(ckpt), tape_p, tape_n, ws, ws_bytes, _stream())
        _lib.check(st, "odevit_solve_adaptive_bwd")
        return (g_x0 if ctx.needs_input_grad[0] else None,) + (None,) * 10 + tuple(gts)


def ode_solve_adaptive(x0: torch.Tensor, t: torch.Tensor, spec: FieldSpec, weights: Dict[str, Optional[torch.Tensor]],
                       rtol: float, atol: float, first_step: Optional[float] = None,
                       max_num_steps: int = DOPRI5_MAX_NUM_STEPS, differentiable: bool = False,
                       capturable: bool = False, want_p_last: bool = False,
                       jasmin: Optional[Tuple[int, int]] = None):
    """Adaptive Dormand-Prince 5(4) solve with per-image step control (odevit_solve_adaptive).

    torchdiffeq's dopri5 run on every image on its own: the error norm, the accept / reject decisions, the step sizes
    and the dense output of image b depend on image b alone (torchdiffeq takes one norm over the whole batch).  `t`
    must be strictly increasing; `max_num_steps` bounds the attempted steps per image over the whole solve (torchdiffeq
    counts them per output interval).  Synchronises with the device once per round (one attempted step of every image).

    differentiable=False: inference only, a gradient request raises.  differentiable=True: when grad mode is on and x0
    or a weight requires grad, `states` is differentiable with respect to them, with each image's accepted steps frozen
    (discretise-then-optimise: odevit_solve_adaptive_record / odevit_solve_adaptive_bwd).  Gradients with respect to
    `t` are not built.

    capturable=True: the same algorithm inside the on-chip-state kernel (odevit_solve_adaptive_resident): one launch, no
    synchronisation, so the call can be captured into a CUDA graph; a replay decides the step sequence on the device
    again.  Failures are reported per image in `status` [B] (0 ok, 1 max_num_steps, 2 non-finite error ratio, 3 dt
    underflow; a failed image's rows from the first output it did not reach are NaN).  Outside a capture `status` is
    read once after the launch and the lowest failed image raises NotConvergedError; inside a capture nothing is checked.
    Covers the PARALLEL field in bf16 at on-chip shapes (head dim 64, dim <= 192, <= 128 tokens, len(t) <= 129), inference
    only: anything else raises, it never falls back to the synchronising solve.  This is a different contract, not a
    faster setting: the default path is the forward of the differentiable solve and raises at the first failure.

    want_p_last: also `p_last` [B,H,N,N], the attention map of each image's LAST field evaluation (k7 = f(y1) of its last
    accepted step, torchdiffeq's `block.attentions`), differentiable with differentiable=True.
    jasmin=(W, k): also the JaSMin window of every image's own last min(W, nfe_b) evaluations (f(x0), the initial-step
    probe and the 6 stages of every attempted step count, rejected ones included): `jas_ring` [W,B,H], image b's window
    in slots [0, min(W, jas_count[b])) (evaluation e in slot e mod W), and `jas_count` [B] (= nfe); not differentiable.
    Neither is built with capturable=True, nor for the MACARON field (it exposes no map).

    Returns dict(states [len(t),B,N,D] (row i = solution at t[i]), final [B,N,D], nfe [B], accepted [B], rejected [B]
    (int32, device), rounds (int: rounds with at least one image still stepping = max_b accepted + rejected; with
    capturable=True a 0-d device tensor), with capturable=True status [B] (int32, device), and the requested attention
    outputs)."""
    names = tuple(k for k, v in weights.items() if v is not None)
    if capturable and (want_p_last or jasmin is not None):
        raise OdevitError("attention outputs (p_last, the JaSMin window) are not built for capturable=True: the on-chip "
                          "adaptive solve exports no maps")
    if capturable:
        return _ode_solve_adaptive_capturable(x0, t, spec, weights, names, rtol, atol, first_step, max_num_steps,
                                              differentiable)
    track = torch.is_grad_enabled() and (x0.requires_grad or any(weights[k].requires_grad for k in names))
    if track and not differentiable:
        raise OdevitError("the adaptive solve is inference-only (no backward is built): run it under torch.no_grad() "
                          "or detach x0 and the weights")
    if spec.has_dropout:
        if differentiable:
            raise OdevitError("the adaptive solve has no dropout: the field's dropout must be 0")
        raise OdevitError("the adaptive solve is inference-only: the field's dropout must be 0 (call .eval())")
    t_host = t.detach().to("cpu", torch.float32).contiguous()
    T = int(t_host.numel())
    t_c = (ctypes.c_float * max(1, T))(*t_host.tolist())
    fs = 0.0 if first_step is None else float(first_step)
    if first_step is not None and not fs > 0:
        raise ValueError(f"first_step must be > 0, got {first_step}")
    jasmin = (int(jasmin[0]), int(jasmin[1])) if jasmin is not None else None
    res = {}
    if track:
        x0 = _require_cuda(x0, "x0")
        states, counts, p_last, ring, jcount = _AdaptiveSolve.apply(
            x0, spec, t_c, T, float(rtol), float(atol), fs, int(max_num_steps), bool(want_p_last), jasmin, names,
            *[weights[k] for k in names])
        if want_p_last:
            res["p_last"] = p_last
        if jasmin is not None:
            res["jas_ring"], res["jas_count"] = ring, jcount
    else:
        x0 = _require_cuda(x0.detach(), "x0")
        attn = _adaptive_attn_outputs(x0, spec, want_p_last, jasmin) if (want_p_last or jasmin is not None) else None
        st, states, counts = _adaptive_call(x0, t_c, T, spec, names, [weights[k].detach() for k in names], rtol, atol,
                                            fs, max_num_steps, attn=attn)
        _adaptive_check(st, "odevit_solve_adaptive")
        if want_p_last:
            res["p_last"] = attn[0]
        if jasmin is not None:
            res["jas_ring"], res["jas_count"] = attn[1][0], attn[1][1]
    rounds = int((counts[1] + counts[2]).max().item())
    res.update({"states": states, "final": states[-1], "nfe": counts[0], "accepted": counts[1], "rejected": counts[2],
                "rounds": rounds})
    return res


def adaptive_jasmin_mean(jas_ring: torch.Tensor, jas_count: torch.Tensor) -> torch.Tensor:
    """Per image b: the mean of the JaSMin statistic over the heads and the min(W, jas_count[b]) slots of b's window
    (ode_solve_adaptive(jasmin=(W, k))): [B], on the device, without a synchronisation."""
    W = jas_ring.shape[0]
    n = jas_count.clamp(max=W).to(jas_ring.dtype)
    valid = torch.arange(W, device=jas_ring.device)[:, None] < jas_count[None, :]
    return (jas_ring.mean(dim=2) * valid).sum(dim=0) / n


def _ode_solve_adaptive_capturable(x0, t, spec: FieldSpec, weights, names, rtol, atol, first_step, max_num_steps,
                                   differentiable):
    if differentiable:
        raise OdevitError("capturable=True is inference-only: it cannot be combined with differentiable=True")
    if torch.is_grad_enabled() and (x0.requires_grad or any(weights[k].requires_grad for k in names)):
        raise OdevitError("the capturable adaptive solve is inference-only: run it under torch.no_grad() or detach x0 "
                          "and the weights")
    if spec.has_dropout:
        raise OdevitError("the capturable adaptive solve is inference-only: the field's dropout must be 0 (call .eval())")
    t_host = t.detach().to("cpu", torch.float32).contiguous()
    T = int(t_host.numel())
    t_c = (ctypes.c_float * max(1, T))(*t_host.tolist())
    fs = 0.0 if first_step is None else float(first_step)
    if first_step is not None and not fs > 0:
        raise ValueError(f"first_step must be > 0, got {first_step}")
    x0 = _require_cuda(x0.detach(), "x0")
    states, counts = _adaptive_resident_call(x0, t_c, T, spec, names, [weights[k].detach() for k in names], rtol,
                                             atol, fs, max_num_steps)
    if not torch.cuda.is_current_stream_capturing():
        status = counts[3].cpu()
        bad = torch.nonzero(status).flatten()
        if bad.numel():
            b = int(bad[0])
            raise NotConvergedError(f"image {b}: " + _ADAPTIVE_STATUS.get(int(status[b]), "status %d" % int(status[b]))
                                    .format(max_steps=int(max_num_steps)))
    return {"states": states, "final": states[-1], "nfe": counts[0], "accepted": counts[1], "rejected": counts[2],
            "status": counts[3], "rounds": (counts[1] + counts[2]).max()}


def fd_curvature(states: torch.Tensor, delta_t: float) -> torch.Tensor:
    """per_seq [B,N] = max over time and features of |s[j+2] - 2 s[j+1] + s[j]| / delta_t^2, one pass
    over the trajectory (ode_transformer_gpt.py:458-468 + the norms/maxima of :529-543)."""
    states = _require_cuda(states.detach(), "states")
    T, B, N, D = states.shape
    out = torch.empty(B, N, device=states.device, dtype=torch.float32)
    with torch.cuda.device(states.device):
        st = _lib.lib().odevit_fd_curvature(_ptr(states), T, B, N, D, float(delta_t), _ptr(out), _stream())
    _lib.check(st, "odevit_fd_curvature")
    return out


class EncoderWeights:
    """The weights of a pre-LayerNorm encoder stack as the C ABI takes them (one odevit_weights per layer) plus
    the library's prepared (activation-typed) copies.  `layers` is a list of dicts with the fp32 CUDA tensors
    norm_a_w/b, norm_b_w/b, in_proj_w [3D,D], in_proj_b [3D], out_proj_w/b, fc1_w/b, fc2_w/b.  Call
    `invalidate()` after changing any of them (a frozen teacher never does)."""

    def __init__(self, layers: Sequence[Dict[str, torch.Tensor]]):
        self.n_layers = len(layers)
        self._keep = []
        self.array = (_lib.Weights * self.n_layers)()
        for i, lw in enumerate(layers):
            for n, t in lw.items():
                t = _require_cuda(t.detach(), f"layer {i} weight {n}").contiguous().float()
                self._keep.append(t)
                setattr(self.array[i], n, t.data_ptr())
        self.cache: Optional[torch.Tensor] = None
        self.cache_key = None

    def invalidate(self) -> None:
        self.cache_key = None


def encoder_forward(x0: torch.Tensor, weights: EncoderWeights, heads: int, hidden: int, ln_eps: float,
                    precision: str = "bf16", attention_maps: str = "last"):
    """hidden [L,B,N,D], maps = pre-LN encoder stack on x0 [B,N,D] (odevit_encoder_fwd): HF ViT's encoder, no grad.
    attention_maps: "none" | "last" ([B,H,N,N]) | "all" ([L,B,H,N,N])."""
    x0 = _require_cuda(x0.detach(), "x0").contiguous().float()
    B, N, D = x0.shape
    L = weights.n_layers
    desc = _lib.Desc(_lib.ABI_VERSION, B, N, D, heads, hidden, _lib.FIELD_MACARON, _lib.PRECISIONS[precision], 1.0)
    p_mode = {"none": 0, "last": 1, "all": 2}[attention_maps]
    hidden_out = torch.empty(L, B, N, D, device=x0.device, dtype=torch.float32)
    maps = None
    if p_mode == 1:
        maps = torch.empty(B, heads, N, N, device=x0.device, dtype=torch.float32)
    elif p_mode == 2:
        maps = torch.empty(L, B, heads, N, N, device=x0.device, dtype=torch.float32)
    with torch.cuda.device(x0.device):
        need = _lib.lib().odevit_encoder_cache_bytes(ctypes.byref(desc), L)
        if need == 0:
            _lib.check(-1, "odevit_encoder_cache_bytes")
        key = (D, heads, hidden, precision, x0.device)
        valid = int(weights.cache is not None and weights.cache_key == key)
        if weights.cache is None or weights.cache.numel() < need + 1024:
            weights.cache = torch.empty(need + 2048, dtype=torch.uint8, device=x0.device)
            valid = 0
        cbase = weights.cache.data_ptr()
        caligned = (cbase + 1023) & ~1023
        keep, ws, ws_bytes = _workspace(desc, _lib.WS_ENCODER_FWD, 0, x0.device)
        st = _lib.lib().odevit_encoder_fwd(ctypes.byref(desc), weights.array, L, float(ln_eps), _ptr(x0), _ptr(hidden_out),
                                           _ptr(maps), p_mode, _vp(caligned), weights.cache.numel() - (caligned - cbase), valid,
                                           ws, ws_bytes, _stream())
    _lib.check(st, "odevit_encoder_fwd")
    weights.cache_key = key
    return hidden_out, maps


def jasmin_rowmax(p_maps: torch.Tensor, k: int) -> torch.Tensor:
    """[..., N, N] attention maps -> [...] max over query rows of the JaSMin row value
    log(g_1 / (g_k + 1e-12) + 1e-12) (ode_transformer_gpt.py:419-456), one pass, no sort."""
    p_maps = _require_cuda(p_maps.detach(), "p_maps").contiguous()
    N = p_maps.shape[-1]
    if p_maps.shape[-2] != N:
        raise ValueError("attention maps must be square in their last two dimensions")
    lead = p_maps.shape[:-2]
    out = torch.empty(lead, device=p_maps.device, dtype=torch.float32)
    with torch.cuda.device(p_maps.device):
        st = _lib.lib().odevit_jasmin_rowmax(_ptr(p_maps), out.numel(), N, int(k), _ptr(out), _stream())
    _lib.check(st, "odevit_jasmin_rowmax")
    return out


# ---------------------------------------------------------------------------------------------
# patch projection (row (f1) of SURVEY section 8: the caller just before the hot path)
# ---------------------------------------------------------------------------------------------
def _gemm_bf16(M: int, N: int, K: int, mn_major: int, A: torch.Tensor, B: torch.Tensor, C: torch.Tensor,
               accumulate: int = 0) -> None:
    """C[M,N] (fp32) (+)= A . B^T on the tcgen05 GEMM (FFMA kernel for shapes it does not cover).  `accumulate` adds into C:
    the library then splits a long contraction over the idle SMs (weight-gradient shapes: few output tiles, K = every
    token of the batch) -- pass a zero-filled C."""
    L = _lib.lib()
    with torch.cuda.device(C.device):
        st = L.odevit_gemm_bf16(M, N, K, mn_major, _ptr(A), _ptr(B), _ptr(C), accumulate, 1, _stream())
        if st == -4:   # ODEVIT_ERR_UNSUPPORTED
            st = L.odevit_gemm_bf16(M, N, K, mn_major, _ptr(A), _ptr(B), _ptr(C), accumulate, 0, _stream())
    _lib.check(st, "odevit_gemm_bf16")


class _PatchProj(torch.autograd.Function):
    """`Conv2d(kernel = stride = patch)` (ode_transformer_gpt.py:137, :157) as im2col (one permuting
    cast) + one bf16 GEMM with fp32 accumulation; weight / input gradients are GEMMs of the same kernel."""

    @staticmethod
    def forward(ctx, x, weight, bias, patch: int):
        x = _require_cuda(x, "pixel_values")
        Bn, C, H, W = x.shape
        g_h, g_w = H // patch, W // patch
        M, K, D = Bn * g_h * g_w, C * patch * patch, weight.shape[0]
        a = torch.empty(Bn, g_h, g_w, C, patch, patch, dtype=torch.bfloat16, device=x.device)
        a.copy_(x.view(Bn, C, g_h, patch, g_w, patch).permute(0, 2, 4, 1, 3, 5))
        w = weight.detach().reshape(D, K).to(torch.bfloat16)
        out = torch.empty(M, D, dtype=torch.float32, device=x.device)
        _gemm_bf16(M, D, K, 0, a, w, out)
        if bias is not None:
            out += bias.detach()
        ctx.save_for_backward(a, w)
        ctx.shape = (Bn, C, H, W, patch, tuple(weight.shape), bias is not None)
        return out.view(Bn, g_h * g_w, D)

    @staticmethod
    def backward(ctx, g_out):
        a, w = ctx.saved_tensors
        Bn, C, H, W, patch, w_shape, has_bias = ctx.shape
        g_h, g_w = H // patch, W // patch
        M, K, D = Bn * g_h * g_w, C * patch * patch, w_shape[0]
        gy = g_out.reshape(M, D).to(torch.bfloat16).contiguous()
        g_x = g_w_ = g_b = None
        if ctx.needs_input_grad[1]:
            g_w_ = torch.zeros(D, K, dtype=torch.float32, device=gy.device)
            _gemm_bf16(D, K, M, 1, gy, a.view(M, K), g_w_, accumulate=1)   # dW[d,k] = sum_m gy[m,d] a[m,k], split over the SMs
            g_w_ = g_w_.view(w_shape)
        if has_bias and ctx.needs_input_grad[2]:
            g_b = g_out.reshape(M, D).sum(0)
        if ctx.needs_input_grad[0]:
            cols = torch.empty(M, K, dtype=torch.float32, device=gy.device)
            _gemm_bf16(M, K, D, 0, gy, w.t().contiguous(), cols)  # dA = gy @ W
            g_x = cols.view(Bn, g_h, g_w, C, patch, patch).permute(0, 3, 1, 4, 2, 5).reshape(Bn, C, H, W)
        return g_x, g_w_, g_b, None


def patch_project(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor], patch: int) -> torch.Tensor:
    """[B, C, H, W] -> [B, (H/p)(W/p), D] patch tokens (before cls / register / positional assembly)."""
    return _PatchProj.apply(x, weight, bias, patch)


class _TokenAssembly(torch.autograd.Function):
    """PatchEmbed.forward (ode_transformer_gpt.py:148-182) in two launches after the im2col cast: the patch GEMM writes
    its rows of x0 [B,N,D] with bias + positional rows added in the epilogue (odevit_tokens_fwd, EPI_TOKENS); the cls /
    distillation / register rows are broadcast by one small kernel.  Token order: cls, [dist], patches, registers; the
    positional rows go to the first `n_pos` tokens (the reference's slicing, including its offset with a dist token)."""

    @staticmethod
    def forward(ctx, x, weight, bias, cls, dist, reg, pos, patch: int, n_pos: int):
        x = _require_cuda(x, "pixel_values")
        Bn, C, H, W = x.shape
        g_h, g_w = H // patch, W // patch
        P, K, D = g_h * g_w, C * patch * patch, weight.shape[0]
        off = 1 + (1 if dist is not None else 0)
        R = reg.shape[0] if reg is not None else 0
        N = off + P + R
        dev = x.device
        a = torch.empty(Bn, g_h, g_w, C, patch, patch, dtype=torch.bfloat16, device=dev)
        a.copy_(x.view(Bn, C, g_h, patch, g_w, patch).permute(0, 2, 4, 1, 3, 5))
        w = weight.detach().reshape(D, K).to(torch.bfloat16)
        pe = pos.detach().reshape(-1, D)
        n_pos = min(int(n_pos), N, pe.shape[0])
        patch_add = torch.zeros(P, D, device=dev, dtype=torch.float32)
        if bias is not None:
            patch_add += bias.detach()
        hi = max(off, min(n_pos, off + P))
        patch_add[:hi - off] += pe[off:hi]
        rows = [cls.detach().reshape(1, D) + pe[0:1]]
        index = [0]
        if dist is not None:
            rows.append(dist.detach().reshape(1, D) + (pe[1:2] if n_pos > 1 else 0))
            index.append(1)
        if R:
            r = reg.detach().clone()
            lo = off + P
            if n_pos > lo:
                r[:n_pos - lo] += pe[lo:n_pos]
            rows.append(r)
            index.extend(range(lo, lo + R))
        special = torch.cat(rows, 0).contiguous().float()
        idx_t = _row_index_tensor(tuple(index), dev).to(torch.int32)
        x0 = torch.empty(Bn, N, D, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            st = _lib.lib().odevit_tokens_fwd(_ptr(a), _ptr(w), Bn, P, K, D, N, off, _ptr(patch_add), _ptr(special), _ptr(idx_t),
                                              len(index), _ptr(x0), _stream())
        _lib.check(st, "odevit_tokens_fwd")
        ctx.save_for_backward(a, w)
        ctx.meta = (Bn, C, H, W, patch, tuple(weight.shape), bias is not None, dist is not None, R, off, P, n_pos,
                    tuple(pos.shape), tuple(cls.shape))
        return x0

    @staticmethod
    def backward(ctx, g):
        a, w = ctx.saved_tensors
        Bn, C, H, W, patch, w_shape, has_bias, has_dist, R, off, P, n_pos, pos_shape, cls_shape = ctx.meta
        g = g.contiguous()
        D = w_shape[0]
        K = C * patch * patch
        M = Bn * P
        need = ctx.needs_input_grad
        g_x = g_w = g_b = g_cls = g_dist = g_reg = g_pos = None
        gp = g[:, off:off + P]
        if need[0] or need[1]:
            gy = gp.to(torch.bfloat16).reshape(M, D).contiguous()
            if need[1]:
                g_w = torch.zeros(D, K, dtype=torch.float32, device=g.device)
                _gemm_bf16(D, K, M, 1, gy, a.view(M, K), g_w, accumulate=1)   # (9 output tiles, K = B * P: split over the SMs)
                g_w = g_w.view(w_shape)
            if need[0]:
                cols = torch.empty(M, K, dtype=torch.float32, device=g.device)
                _gemm_bf16(M, K, D, 0, gy, w.t().contiguous(), cols)
                g_h, g_w_ = H // patch, W // patch
                g_x = cols.view(Bn, g_h, g_w_, C, patch, patch).permute(0, 3, 1, 4, 2, 5).reshape(Bn, C, H, W)
        col = g.sum(0) if (need[3] or need[4] or need[5] or need[6] or (has_bias and need[2])) else None     # [N, D]
        if has_bias and need[2]:
            g_b = col[off:off + P].sum(0)
        if need[3]:
            g_cls = col[0].reshape(cls_shape)
        if has_dist and need[4]:
            g_dist = col[1].reshape(cls_shape)
        if R and need[5]:
            g_reg = col[off + P:].clone()
        if need[6]:
            g_pos = torch.zeros(pos_shape, device=g.device, dtype=torch.float32)
            g_pos.view(-1, D)[:n_pos] = col[:n_pos]
        return g_x, g_w, g_b, g_cls, g_dist, g_reg, g_pos, None, None


def token_assembly(x, weight, bias, cls, dist, reg, pos, patch: int, n_pos: int) -> torch.Tensor:
    """[B,C,H,W] pixels -> x0 [B,N,D] tokens (cls, [dist], patches, registers) with positional rows, bf16 GEMM."""
    return _TokenAssembly.apply(x, weight, bias, cls, dist, reg, pos, patch, n_pos)


class _HeadCE(torch.autograd.Function):
    """logits = head(final[:, 0]) and F.cross_entropy(logits, labels, label_smoothing) (ode_transformer_gpt.py:588-589,
    :626) as one launch (odevit_head_ce_fwd); backward: d logits from the loss and / or a cotangent on the logits, d
    cls row, d head.weight / bias (odevit_head_ce_bwd)."""

    @staticmethod
    def forward(ctx, final, weight, bias, labels, eps: float):
        final = _require_cuda(final, "final")
        B, N, D = final.shape
        C = weight.shape[0]
        dev = final.device
        w = _require_cuda(weight.detach(), "head.weight")
        b = _require_cuda(bias.detach(), "head.bias") if bias is not None else None
        logits = torch.empty(B, C, device=dev, dtype=torch.float32)
        has_loss = labels is not None
        rows = torch.empty(B, device=dev, dtype=torch.float32) if has_loss else None
        lse = torch.empty(B, device=dev, dtype=torch.float32) if has_loss else None
        lab = labels.to(dev, torch.int64).contiguous() if has_loss else None
        with torch.cuda.device(dev):
            st = _lib.lib().odevit_head_ce_fwd(_ptr(final), N * D, _ptr(w), _ptr(b), _ptr(lab), B, C, D, float(eps), _ptr(logits),
                                               _ptr(rows), _ptr(lse), _stream())
        _lib.check(st, "odevit_head_ce_fwd")
        ctx.save_for_backward(final, w, lab if has_loss else final.new_empty(0), logits, lse if has_loss else final.new_empty(0))
        ctx.cfg = (float(eps), has_loss, bias is not None)
        ctx.set_materialize_grads(False)
        loss = rows.mean() if has_loss else final.new_zeros(())
        return logits, loss

    @staticmethod
    def backward(ctx, g_logits, g_loss):
        final, w, lab, logits, lse = ctx.saved_tensors
        eps, has_loss, has_bias = ctx.cfg
        B, N, D = final.shape
        C = w.shape[0]
        dev = final.device
        if not has_loss:
            g_loss = None
        if g_logits is None and g_loss is None:
            return None, None, None, None, None
        g_logits = _require_cuda(g_logits, "g_logits") if g_logits is not None else None
        g_loss = g_loss.reshape(1).float().contiguous() if g_loss is not None else None
        dz = torch.empty(B, C, device=dev, dtype=torch.float32)
        need = ctx.needs_input_grad
        g_final = torch.zeros_like(final) if need[0] else None
        g_w = torch.zeros_like(w) if need[1] else None
        g_b = torch.zeros(C, device=dev, dtype=torch.float32) if (has_bias and need[2]) else None
        if g_b is not None and g_w is None:
            g_w = torch.zeros_like(w)
        with torch.cuda.device(dev):
            st = _lib.lib().odevit_head_ce_bwd(_ptr(final), N * D, _ptr(w), _ptr(lab if has_loss else None), _ptr(logits),
                                               _ptr(lse if has_loss else None), _ptr(g_logits), _ptr(g_loss), B, C, D, eps,
                                               _ptr(dz), _ptr(g_final), N * D, _ptr(g_w), _ptr(g_b), _stream())
        _lib.check(st, "odevit_head_ce_bwd")
        return g_final, (g_w if need[1] else None), g_b, None, None


def head_ce(final: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor], labels: Optional[torch.Tensor],
            label_smoothing: float = 0.05):
    """(logits [B,C], loss 0-d | None) from the final state [B,N,D] (CLS row 0) and the head's parameters."""
    logits, loss = _HeadCE.apply(final, weight, bias, labels, label_smoothing)
    return logits, (loss if labels is not None else None)
