"""Stage-1 RGB-sigma NeRFNetwork (mirrors nerf/network.py:10-207): the same field without the instance head.

Same constructor arguments, sub-module names and state-dict keys as the reference (`encoder.embeddings`,
`encoder.offsets`, `sigma_net.{0,1}.weight`, `color_net.{0,1,2}.weight` [, `encoder_bg.*`, `bg_net.*`]), so a stage-1
checkpoint loads unchanged and its tensors can be copied into the instance-stage network (main_nerf_mask.py:166-170).

Execution paths, both on libinerf_b200 (no CPU / PyTorch fallback for the encoders or the ray ops):
* no-grad CUDA calls with the standard architecture reuse the fused tcgen05 field / one-launch renderer of the
  instance stage with the instance head switched off (mask outputs NULL): the interleaved table carries the sigma table
  in both halves and the mask-net operand blob is zero, so no extra kernel variant is needed;
* training (autograd) runs the reference's operator sequence (network.py:96-127) on the op-level kernels:
  GridEncoder fwd/bwd, SHEncoder, nn.Linear under autocast, march_rays_train, composite_rays_train fwd/bwd.
"""
from __future__ import annotations

from types import SimpleNamespace

import torch
import torch.nn as nn
import torch.nn.functional as F

import ctypes

from .._lib import PARAM_EPOCH, call, lib, ptr, stream_ptr
from ..activation import trunc_exp
from ..encoding import get_encoder
from .network_mask import NeRFNetwork as _InstanceNetwork
from .renderer import NeRFRenderer


class _FusedRGBField(torch.autograd.Function):
    """Stage-1 field forward (inerf_field_forward_train_rgb) / backward (inerf_field_backward_rgb), one launch each: sigma_net,
    color_net, SH and the sigma hash table.  The table gradient is accumulated straight into `encoder.embeddings.grad` by the
    kernel's fp32 atomics, so `None` is returned for that input."""

    @staticmethod
    def forward(ctx, model, x, d, table, ws0, ws1, wc0, wc1, wc2):
        B, dev = x.shape[0], x.device
        sigmas = torch.empty(B, dtype=torch.float32, device=dev)
        rgbs = torch.empty(B, 3, dtype=torch.float32, device=dev)
        xs = torch.empty(B, 64, dtype=torch.float16, device=dev)
        desc = model._field_desc()
        desc.n_valid = getattr(model, "_n_valid_ptr", None)
        ctx.n_valid = desc.n_valid
        call("inerf_field_forward_train_rgb", ctypes.byref(desc), ptr(x), ptr(d), B, ptr(sigmas), ptr(rgbs), ptr(xs), stream_ptr(dev))
        ctx.model = model
        ctx.save_for_backward(x, xs, sigmas, rgbs)
        return sigmas, rgbs

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_sigmas, g_rgbs):
        x, xs, sigmas, rgbs = ctx.saved_tensors
        model = ctx.model
        B, dev = x.shape[0], x.device
        table = model.encoder.embeddings
        if table.grad is None:
            table.grad = torch.zeros_like(table)
        gs0 = torch.zeros(64, 32, dtype=torch.float32, device=dev)
        gs1 = torch.zeros(16, 64, dtype=torch.float32, device=dev)
        gc0 = torch.zeros(64, 31, dtype=torch.float32, device=dev)
        gc1 = torch.zeros(64, 64, dtype=torch.float32, device=dev)
        gc2 = torch.zeros(3, 64, dtype=torch.float32, device=dev)
        if B > 0:
            desc = model._field_desc()
            desc.n_valid = ctx.n_valid
            wb = model._packed_weights_rgb_bwd()
            g_sigmas = (torch.zeros_like(sigmas) if g_sigmas is None else g_sigmas.float()).contiguous()
            g_rgbs = (torch.zeros_like(rgbs) if g_rgbs is None else g_rgbs.float()).contiguous()
            call("inerf_field_backward_rgb", ctypes.byref(desc), ptr(wb), ptr(x), ptr(xs), ptr(sigmas), ptr(rgbs), ptr(g_sigmas), ptr(g_rgbs), B,
                 ptr(table.grad), ptr(gs0), ptr(gs1), ptr(gc0), ptr(gc1), ptr(gc2), stream_ptr(dev))
        return None, None, None, None, gs0, gs1, gc0, gc1, gc2


class NeRFNetwork(NeRFRenderer):
    def __init__(self, encoding="hashgrid", encoding_dir="sphere_harmonics", encoding_bg="hashgrid", num_layers=2, hidden_dim=64,
                 geo_feat_dim=15, num_layers_color=3, hidden_dim_color=64, num_layers_bg=2, hidden_dim_bg=64, bound=1,
                 num_instances=None, **kwargs):   # num_instances: accepted and ignored, as in the reference (network.py:22)
        super().__init__(bound, num_instances=1, **kwargs)
        self.num_layers = num_layers
        self.hidden_dim = hidden_dim
        self.geo_feat_dim = geo_feat_dim
        self.encoder, self.in_dim = get_encoder(encoding, desired_resolution=2048 * bound)
        self.sigma_net = nn.ModuleList([
            nn.Linear(self.in_dim if l == 0 else hidden_dim, 1 + geo_feat_dim if l == num_layers - 1 else hidden_dim, bias=False)
            for l in range(num_layers)])
        self.num_layers_color = num_layers_color
        self.hidden_dim_color = hidden_dim_color
        self.encoder_dir, self.in_dim_dir = get_encoder(encoding_dir)
        self.color_net = nn.ModuleList([
            nn.Linear(self.in_dim_dir + geo_feat_dim if l == 0 else hidden_dim_color, 3 if l == num_layers_color - 1 else hidden_dim_color,
                      bias=False) for l in range(num_layers_color)])
        if self.bg_radius > 0:
            self.num_layers_bg = num_layers_bg
            self.hidden_dim_bg = hidden_dim_bg
            self.encoder_bg, self.in_dim_bg = get_encoder(encoding_bg, input_dim=2, num_levels=4, log2_hashmap_size=19,
                                                          desired_resolution=2048)
            self.bg_net = nn.ModuleList([
                nn.Linear(self.in_dim_bg + self.in_dim_dir if l == 0 else hidden_dim_bg, 3 if l == num_layers_bg - 1 else hidden_dim_bg,
                          bias=False) for l in range(num_layers_bg)])
        else:
            self.bg_net = None
        self.use_fused = True
        self._packed = None
        self._tables = None
        self._work_counter = None
        self._zero_head = None
        self._packed_rgb_bwd = None

    # ---- fused inference: the instance-stage kernels with the head switched off ------------------------------------
    @property
    def encoder_mask(self):      # second half of the interleaved table = the sigma table again (never read back)
        return self.encoder

    @property
    def mask_net(self):          # zero operand blob for the (unused) head; plain tensors, not parameters
        dev = self.encoder.embeddings.device
        if self._zero_head is None or self._zero_head[0].weight.device != dev:
            self._zero_head = [SimpleNamespace(weight=torch.zeros(o, i, device=dev)) for o, i in ((64, 47), (64, 64), (1, 64))]
        return self._zero_head

    def _standard_arch(self) -> bool:
        e = self.encoder
        return (self.num_layers == 2 and self.hidden_dim == 64 and self.geo_feat_dim == 15 and self.num_layers_color == 3
                and self.hidden_dim_color == 64 and getattr(e, "num_levels", 0) == 16 and getattr(e, "level_dim", 0) == 2
                and getattr(e, "gridtype", "") == "hash" and not e.align_corners and e.interp_id == 0
                and getattr(self.encoder_dir, "degree", 0) == 4 and hasattr(lib(), "inerf_field_forward"))

    def fused_available(self) -> bool:
        if getattr(self, "fused_requires_autocast", False) and not torch.is_autocast_enabled():
            return False
        return bool(self.use_fused and self._standard_arch() and self.encoder.embeddings.is_cuda)

    def fused_render_available(self, render_mask: bool) -> bool:
        return (not render_mask) and self.fused_available() and hasattr(lib(), "inerf_render_fused")

    _packed_weights = _InstanceNetwork._packed_weights
    _packed_tables = _InstanceNetwork._packed_tables
    _field_desc = _InstanceNetwork._field_desc
    forward_fused = _InstanceNetwork.forward_fused
    _render_fused = _InstanceNetwork._render_fused
    _occupancy_density_fused = _InstanceNetwork._occupancy_density_fused
    _extract_volume_fused = _InstanceNetwork._extract_volume_fused

    def extract_volume(self, resolution, bbox=None, view_dir=None, sigma_thresh=None, skip_empty=True, labels=True, **kwargs):
        """NeRFRenderer.extract_volume for sigma / rgb: this network has no instance head, so `labels` must be False."""
        if labels:
            raise ValueError("the stage-1 network has no instance head: call extract_volume(..., labels=False)")
        return super().extract_volume(resolution, bbox, view_dir, sigma_thresh, skip_empty, labels=False, **kwargs)

    def extract_mesh(self, resolution=256, bbox=None, threshold=10, view_dir=None, labels=True, skip_empty=True):
        """NeRFRenderer.extract_mesh with vertex colours only: this network has no instance head, so `labels` must be False."""
        if labels:
            raise ValueError("the stage-1 network has no instance head: call extract_mesh(..., labels=False)")
        return super().extract_mesh(resolution, bbox, threshold, view_dir, labels=False, skip_empty=skip_empty)

    # ---- fused training (fp16 autocast, standard architecture): one launch forward, one launch backward -----------------
    def fused_train_available(self, x, d) -> bool:
        if not (self.fused_available() and x.is_cuda and torch.is_autocast_enabled() and not x.requires_grad and not d.requires_grad):
            return False
        if not hasattr(lib(), "inerf_field_backward_rgb"):
            return False
        ps = [self.encoder.embeddings, *[l.weight for l in self.sigma_net], *[l.weight for l in self.color_net]]
        return all(p.requires_grad for p in ps)

    def bounded_stream(self) -> bool:
        """The fused training forward / backward stop at the marcher's device-side sample total (inerf_field_desc.n_valid)."""
        ps = [self.encoder.embeddings, *[l.weight for l in self.sigma_net], *[l.weight for l in self.color_net]]
        return bool(self.fused_available() and torch.is_autocast_enabled() and hasattr(lib(), "inerf_field_backward_rgb")
                    and self.bg_radius <= 0 and all(p.requires_grad for p in ps))

    def _packed_weights_rgb_bwd(self):
        ws = [m.weight for m in (*self.sigma_net, *self.color_net)]
        dev = ws[0].device
        key = tuple((w.data_ptr(), w._version) for w in ws) + (str(dev), PARAM_EPOCH[0])
        if self._packed_rgb_bwd is None or self._packed_rgb_bwd[0] != key:
            blob = self._packed_rgb_bwd[1] if self._packed_rgb_bwd is not None and self._packed_rgb_bwd[1].device == dev else \
                torch.empty(lib().inerf_field_rgb_bwd_weights_bytes(), dtype=torch.uint8, device=dev)
            call("inerf_field_pack_weights_rgb_bwd_device", *[ptr(w.detach()) for w in ws], ptr(blob), stream_ptr(dev))
            self._packed_rgb_bwd = (key, blob)
        return self._packed_rgb_bwd[1]

    def forward_fused_train(self, x, d):
        x = x.float().contiguous().view(-1, 3)
        d = d.float().contiguous().view(-1, 3)
        return _FusedRGBField.apply(self, x, d, self.encoder.embeddings, *[l.weight for l in self.sigma_net],
                                    *[l.weight for l in self.color_net])

    # ---- reference operator sequence (network.py:96-127) --------------------------------------------------------------
    @staticmethod
    def _mlp(net, h):
        n = len(net)
        for l in range(n):
            h = net[l](h)
            if l != n - 1:
                h = F.relu(h, inplace=True)
        return h

    def forward(self, x, d):
        """x [N,3] in [-bound,bound], d [N,3] unit -> (sigma [N], rgb [N,3])"""
        if not torch.is_grad_enabled() and x.is_cuda and self.fused_available():
            sigma, rgb, _ = self.forward_fused(x, d, want_masks=False)
            return sigma, rgb
        if torch.is_grad_enabled() and self.fused_train_available(x, d):
            return self.forward_fused_train(x, d)
        h = self._mlp(self.sigma_net, self.encoder(x, bound=self.bound))
        sigma = trunc_exp(h[..., 0])
        geo_feat = h[..., 1:]
        h = self._mlp(self.color_net, torch.cat([self.encoder_dir(d), geo_feat], dim=-1))
        return sigma, torch.sigmoid(h)

    def density(self, x):
        h = self._mlp(self.sigma_net, self.encoder(x, bound=self.bound))
        return {"sigma": trunc_exp(h[..., 0]), "geo_feat": h[..., 1:]}

    def background(self, x, d):
        h = torch.cat([self.encoder_dir(d), self.encoder_bg(x)], dim=-1)
        return torch.sigmoid(self._mlp(self.bg_net, h))

    def color(self, x, d, mask=None, geo_feat=None, **kwargs):
        if mask is not None:
            rgbs = torch.zeros(mask.shape[0], 3, dtype=x.dtype, device=x.device)
            if not mask.any():
                return rgbs
            x, d, geo_feat = x[mask], d[mask], geo_feat[mask]
        h = torch.sigmoid(self._mlp(self.color_net, torch.cat([self.encoder_dir(d), geo_feat], dim=-1)))
        if mask is not None:
            rgbs[mask] = h.to(rgbs.dtype)
            return rgbs
        return h

    def get_params(self, lr):
        params = [
            {"params": self.encoder.parameters(), "lr": lr},
            {"params": self.sigma_net.parameters(), "lr": lr},
            {"params": self.encoder_dir.parameters(), "lr": lr},
            {"params": self.color_net.parameters(), "lr": lr},
        ]
        if self.bg_radius > 0:
            params.append({"params": self.encoder_bg.parameters(), "lr": lr})
            params.append({"params": self.bg_net.parameters(), "lr": lr})
        return params
