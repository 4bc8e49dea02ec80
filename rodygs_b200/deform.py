"""Time embedding + motion-basis MLP, state-dict compatible with the reference's
`MLPBasisNetwork` (/root/reference/src/model/rodygs_dynamic.py:243-327) and
`TimestepEmbedder` (:192-220).

Two implementations of SURVEY.md §8 row a1:

* `BasisMLP` - the product path: the packed parameters live in ONE flat fp32 buffer and
  `rdg_basis_mlp_fwd` / `rdg_basis_mlp_bwd` (csrc/basis_mlp.cu) evaluate the embedding,
  the timenet and the 16 heads for the query time and all T training times in one
  launch (two for the backward, deterministic).  No PyTorch fallback.
* `MotionBasisNetwork` - an `nn.Module` with the reference's parameter names, kept as
  the state-dict carrier (checkpoints load into it unchanged) and as the torch-autograd
  twin the tests compare the kernels with.  Its 16 per-basis heads, which the reference
  runs as a Python loop of 16 x 2 `nn.Linear` calls (:314-317), are two batched matmuls.

Their outputs feed the fused kernel (rodygs_b200.dynamic.render_dynamic).
"""
from __future__ import annotations

import math

import ctypes as C
from typing import Dict, Optional, Tuple

import torch
import torch.nn as nn


class TimestepEmbedder(nn.Module):
    """emb(t) = [t, sin(f_0 pi t), cos(f_0 pi t), sin(f_1 pi t), ...] (rodygs_dynamic.py:202-220)."""

    def __init__(self, emb_multires: int, input_dims: int = 1, log_sampling: bool = False):
        super().__init__()
        self.num_freqs = emb_multires
        if log_sampling:
            freqs = 2.0 ** torch.linspace(0.0, emb_multires - 1, emb_multires)
        else:
            freqs = torch.linspace(1.0, 2.0 ** (emb_multires - 1), emb_multires)
        self.register_buffer("freqs_pi", freqs * math.pi, persistent=False)

    def forward(self, t: torch.Tensor) -> torch.Tensor:
        t = torch.as_tensor(t, dtype=torch.float32, device=self.freqs_pi.device)
        ang = t.unsqueeze(-1) * self.freqs_pi                       # [..., F]
        sc = torch.stack((torch.sin(ang), torch.cos(ang)), dim=-1)  # [..., F, 2] -> interleaved sin, cos
        return torch.cat((t.unsqueeze(-1), sc.flatten(-2)), dim=-1)


class _Head(nn.Module):
    """Parameter container with the reference's names: basis_xyz.{k}.basis.{0,2}."""

    def __init__(self, width: int, out_dim: int, act: nn.Module):
        super().__init__()
        self.basis = nn.Sequential(nn.Linear(width, width // 2), act, nn.Linear(width // 2, out_dim))
        for m in self.basis.modules():
            if isinstance(m, nn.Linear):
                nn.init.normal_(m.weight, mean=0, std=1e-2)
                nn.init.constant_(m.bias, 0)


class MotionBasisNetwork(nn.Module):
    trans_dim = 3
    rot_dim = 4

    def __init__(self, netwidth: int = 128, num_basis: int = 16, t_emb_multires: int = 26,
                 t_log_sampling: bool = False, activation: str = "gelu"):
        super().__init__()
        self.num_basis = num_basis
        self.t_embed_dim = t_emb_multires * 2 + 1
        self.t_embedder = TimestepEmbedder(t_emb_multires, 1, t_log_sampling)
        self.activation = nn.GELU() if activation.lower() != "relu" else nn.ReLU(inplace=False)
        self.timenet = nn.Sequential(
            nn.Linear(self.t_embed_dim, netwidth), self.activation,
            nn.Linear(netwidth, netwidth), self.activation,
            nn.Linear(netwidth, netwidth // 2), self.activation)
        for m in self.timenet.modules():
            if isinstance(m, nn.Linear):
                nn.init.normal_(m.weight, mean=0, std=1e-2)
                nn.init.constant_(m.bias, 0)
        self.basis_xyz = nn.ModuleList([_Head(netwidth // 2, 7, self.activation) for _ in range(num_basis)])

    def bases(self, t_embs: torch.Tensor) -> torch.Tensor:
        """t_embs [..., 53] -> B [..., num_basis, 7]; equals `batch_inference` (:296-306)."""
        h = self.timenet(t_embs)
        w0 = torch.stack([hd.basis[0].weight for hd in self.basis_xyz])   # [K, w/2, w]
        b0 = torch.stack([hd.basis[0].bias for hd in self.basis_xyz])     # [K, w/2]
        w2 = torch.stack([hd.basis[2].weight for hd in self.basis_xyz])   # [K, 7, w/2]
        b2 = torch.stack([hd.basis[2].bias for hd in self.basis_xyz])     # [K, 7]
        u = self.activation(torch.einsum("...i,koi->...ko", h, w0) + b0)
        return torch.einsum("...ki,koi->...ko", u, w2) + b2

    def batch_embedding(self, timesteps: torch.Tensor) -> torch.Tensor:
        return self.t_embedder(timesteps)

    def batch_inference(self, t_embs: torch.Tensor) -> torch.Tensor:
        return self.bases(t_embs)

    def query_and_table(self, t: torch.Tensor, train_time_embs: torch.Tensor):
        """(B(t) [K,7], table [T,K,7]) from a single batched pass."""
        emb = torch.cat((self.t_embedder(t).reshape(1, -1), train_time_embs), dim=0)
        out = self.bases(emb)
        return out[0], out[1:]

    def forward(self, coeff: torch.Tensor, timestep: torch.Tensor):
        """Reference signature (:308-327): returns (translation, rotation) = coeff @ B(t)."""
        basis = self.bases(self.t_embedder(timestep))
        tot = torch.squeeze(torch.squeeze(coeff) @ basis)
        return tot[..., : self.trans_dim], tot[..., self.trans_dim:]


def packed_layout(emb_dim: int, width: int, num_basis: int, out_dim: int = 7):
    """Name -> (offset, shape) of the packed parameter buffer of `rdg_basis_mlp_*` (include/rodygs_b200.h);
    the four head blocks are the reference's `basis_xyz.{k}.basis.{0,2}.{weight,bias}` stacked over k."""
    h, q = width // 2, width // 4
    blocks = [("timenet.0.weight", (width, emb_dim)), ("timenet.0.bias", (width,)),
              ("timenet.2.weight", (width, width)), ("timenet.2.bias", (width,)),
              ("timenet.4.weight", (h, width)), ("timenet.4.bias", (h,)),
              ("heads.0.weight", (num_basis, q, h)), ("heads.0.bias", (num_basis, q)),
              ("heads.2.weight", (num_basis, out_dim, q)), ("heads.2.bias", (num_basis, out_dim))]
    out, off = {}, 0
    for name, shape in blocks:
        out[name] = (off, shape)
        off += math.prod(shape)
    return out, off


def pack_state_dict(state: Dict[str, torch.Tensor], emb_dim: int, width: int, num_basis: int, out_dim: int = 7) -> torch.Tensor:
    """Reference `MLPBasisNetwork.state_dict()` (or that of its gradients) -> packed fp32 vector."""
    layout, total = packed_layout(emb_dim, width, num_basis, out_dim)
    flat = torch.empty(total, dtype=torch.float32)
    for name, (off, shape) in layout.items():
        if name.startswith("heads."):
            li, kind = name.split(".")[1:]
            t = torch.stack([state[f"basis_xyz.{k}.basis.{li}.{kind}"] for k in range(num_basis)])
        else:
            t = state[name]
        assert tuple(t.shape) == tuple(shape), (name, tuple(t.shape), shape)
        flat[off:off + t.numel()] = t.detach().reshape(-1).to(torch.float32).cpu()
    return flat


def unpack_to_state_dict(flat: torch.Tensor, emb_dim: int, width: int, num_basis: int, out_dim: int = 7) -> Dict[str, torch.Tensor]:
    """Inverse of `pack_state_dict`: packed vector -> tensors under the reference's names."""
    layout, _ = packed_layout(emb_dim, width, num_basis, out_dim)
    out = {}
    for name, (off, shape) in layout.items():
        t = flat[off:off + math.prod(shape)].reshape(shape)
        if name.startswith("heads."):
            li, kind = name.split(".")[1:]
            for k in range(num_basis):
                out[f"basis_xyz.{k}.basis.{li}.{kind}"] = t[k]
        else:
            out[name] = t
    return out


class BasisMLP:
    """The motion-basis network on the CUDA path (`rdg_basis_mlp_fwd` / `_bwd`).

    `params` is one flat fp32 CUDA tensor (a leaf with `requires_grad`), `grad` its gradient buffer -
    the same convention as the trainer's flat Gaussian buffers, so one `rdg_adam` call steps the whole network
    (the reference registers it as a single Adam group, src/trainer/rodygs_dynamic.py:112-118).
    """

    def __init__(self, netwidth: int = 128, num_basis: int = 16, t_emb_multires: int = 26, t_log_sampling: bool = False,
                 activation: str = "gelu", device="cuda", out_dim: int = 7):
        from . import _lib
        self._lib = _lib
        _lib.load()                                   # raises if the CUDA library is not built: no fallback
        self.width, self.num_basis, self.out_dim = netwidth, num_basis, out_dim
        # everything but the device: what a checkpoint needs to build the same network again (SplatTrainStep.state_dict)
        self.init_args = {"netwidth": int(netwidth), "num_basis": int(num_basis), "t_emb_multires": int(t_emb_multires),
                          "t_log_sampling": bool(t_log_sampling), "activation": str(activation), "out_dim": int(out_dim)}
        self.emb_dim = 2 * t_emb_multires + 1
        self.activation = 1 if activation.lower() == "relu" else 0
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("BasisMLP runs on CUDA only (no CPU fallback)")
        self.layout, self.n_params = packed_layout(self.emb_dim, netwidth, num_basis, out_dim)
        assert self.n_params == _lib.load().rdg_basis_mlp_param_count(self.emb_dim, netwidth, num_basis, out_dim)
        self.saved_floats = int(_lib.load().rdg_basis_mlp_saved_floats(self.emb_dim, netwidth, num_basis))
        emb = TimestepEmbedder(t_emb_multires, 1, t_log_sampling)
        self.freqs_pi = emb.freqs_pi.to(self.device).contiguous()
        # reference init: every Linear weight ~ N(0, 1e-2), bias 0 (rodygs_dynamic.py:233-236, 271-274)
        flat = torch.zeros(self.n_params, dtype=torch.float32)
        for name, (off, shape) in self.layout.items():
            if name.endswith("weight"):
                flat[off:off + math.prod(shape)].normal_(0.0, 1e-2)
        self.params = flat.to(self.device).requires_grad_(True)
        self.grad = torch.zeros_like(self.params)
        self._saved: Optional[torch.Tensor] = None
        self._rows = 0
        self._ws: Optional[torch.Tensor] = None

    # -- checkpoints ---------------------------------------------------------------------------------------------
    def load_state_dict(self, state: Dict[str, torch.Tensor]):
        """Accepts `MLPBasisNetwork.state_dict()` of the reference (or of `MotionBasisNetwork`)."""
        with torch.no_grad():
            self.params.copy_(pack_state_dict(state, self.emb_dim, self.width, self.num_basis, self.out_dim))
        return self

    def state_dict(self) -> Dict[str, torch.Tensor]:
        return {k: v.clone() for k, v in unpack_to_state_dict(self.params.detach(), self.emb_dim, self.width,
                                                              self.num_basis, self.out_dim).items()}

    def grad_state_dict(self) -> Dict[str, torch.Tensor]:
        return unpack_to_state_dict(self.grad, self.emb_dim, self.width, self.num_basis, self.out_dim)

    # -- kernels -------------------------------------------------------------------------------------------------
    def _args(self, rows: int, emb, times, basis, saved, row0=None):
        L = self._lib
        return L.RdgBasisMlp(self.emb_dim, self.width, self.num_basis, self.out_dim, self.activation, rows,
                             L.ptr(self.params), L.ptr(emb), L.ptr(times), L.ptr(self.freqs_pi), L.ptr(basis), L.ptr(row0),
                             L.ptr(saved))

    def forward_rows(self, times: Optional[torch.Tensor] = None, emb: Optional[torch.Tensor] = None,
                     save: bool = True, out: Optional[torch.Tensor] = None,
                     out_row0: Optional[torch.Tensor] = None) -> torch.Tensor:
        """B for every row: `times` [rows] (embedding evaluated in the kernel) or `emb` [rows, emb_dim]
        (`batch_embedding` output). Returns [rows, num_basis, 7]; keeps the pre-activations for `backward_rows`.
        With `out_row0` [num_basis, 7] and `out` [rows - 1, num_basis, 7] (contiguous fp32 CUDA tensors, e.g. the
        trainer's B(t) and table slices) the kernel writes row 0 and rows 1.. straight into them and `out` is returned."""
        L = self._lib
        src = emb if emb is not None else times
        L.require_cuda(src)
        src = src.to(torch.float32).contiguous()
        if emb is not None:
            src = src.reshape(-1, self.emb_dim)
        else:
            src = src.reshape(-1)
        rows = src.shape[0]
        if out_row0 is not None:
            L.require_cuda(out, out_row0)
            assert out.is_contiguous() and out_row0.is_contiguous()
            assert out.numel() == (rows - 1) * self.num_basis * self.out_dim and out_row0.numel() == self.num_basis * self.out_dim
            basis = out
        else:
            basis = torch.empty(rows, self.num_basis, self.out_dim, device=self.device) if out is None else out
            assert basis.is_contiguous() and basis.numel() == rows * self.num_basis * self.out_dim
        saved = torch.empty(rows, self.saved_floats, device=self.device) if save else None
        a = self._args(rows, src if emb is not None else None, src if emb is None else None, basis, saved, out_row0)
        L.check(L.load().rdg_basis_mlp_fwd(C.byref(a), L.stream_ptr()))
        if save:
            self._saved, self._rows = saved, rows
        return basis

    def backward_rows(self, d_basis: torch.Tensor, accumulate: bool = False, saved: Optional[torch.Tensor] = None,
                      out: Optional[torch.Tensor] = None, d_row0: Optional[torch.Tensor] = None) -> torch.Tensor:
        """dL/dB [rows, num_basis, 7] -> packed parameter gradient (written to `self.grad` unless `out` is given).
        With `d_row0` [num_basis, 7], `d_basis` holds rows 1.. only (the trainer's dL/dB(t) and dL/dtable slices)."""
        L = self._lib
        saved = self._saved if saved is None else saved
        if saved is None:
            raise RuntimeError("backward_rows before forward_rows(save=True)")
        rows = saved.shape[0]
        d_basis = d_basis.to(torch.float32).contiguous()
        if d_row0 is not None:
            d_row0 = d_row0.to(torch.float32).contiguous()
            assert d_row0.numel() == self.num_basis * self.out_dim
        assert d_basis.numel() == (rows - (d_row0 is not None)) * self.num_basis * self.out_dim
        need = int(L.load().rdg_basis_mlp_bwd_workspace_bytes(rows, self.emb_dim, self.width, self.num_basis))
        if self._ws is None or self._ws.numel() * 4 < need:
            self._ws = torch.empty((need + 3) // 4, device=self.device)
        out = self.grad if out is None else out
        a = self._args(rows, None, None, None, saved)
        L.check(L.load().rdg_basis_mlp_bwd(C.byref(a), L.ptr(d_basis), L.ptr(d_row0), L.ptr(out), int(accumulate), L.ptr(self._ws),
                                           self._ws.numel() * 4, L.stream_ptr()))
        return out

    # -- the reference's call pattern --------------------------------------------------------------------------------
    def query_and_table(self, t, train_times: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """(B(t) [K,7], table [T,K,7]) with autograd into `self.params` (one forward launch, two backward)."""
        t = torch.as_tensor(t, dtype=torch.float32, device=self.device).reshape(1)
        times = torch.cat((t, train_times.to(self.device, torch.float32).reshape(-1)))
        out = _BasisMlpFn.apply(self.params, times, self)
        return out[0], out[1:]

    def batch_inference_times(self, times: torch.Tensor) -> torch.Tensor:
        return _BasisMlpFn.apply(self.params, times.to(self.device, torch.float32).reshape(-1), self)


class _BasisMlpFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, params, times, net: BasisMLP):
        basis = net.forward_rows(times=times, save=True)
        ctx.net, ctx.saved = net, net._saved
        return basis

    @staticmethod
    def backward(ctx, d_basis):
        g = torch.empty_like(ctx.net.params)
        ctx.net.backward_rows(d_basis, accumulate=False, saved=ctx.saved, out=g)
        return g, None, None
