"""NeRFNetwork with the instance-logit head (mirrors nerf/network_mask.py:10-272).

Same constructor arguments, sub-module names and therefore the same state-dict
keys as the reference (`encoder.embeddings`, `encoder.offsets`,
`sigma_net.{0,1}.weight`, `color_net.{0,1,2}.weight`, `encoder_mask.*`,
`mask_net.{0,1,2}.weight`), so reference checkpoints load unchanged.

Two execution paths, both on libinerf_b200:
* fused (default for no-grad CUDA calls with the standard architecture): ONE
  kernel for hash encode x2 + SH + the three MLPs on tcgen05 tensor cores;
* modular (autograd / non-standard widths): GridEncoder + SHEncoder kernels and
  nn.Linear, exactly the reference's operator sequence (network_mask.py:119-158).
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from .._lib import PARAM_EPOCH, FieldDesc, call, lib, ptr, stream_ptr
from ..activation import trunc_exp
from ..encoding import get_encoder
from .renderer import NeRFMaskRenderer


class _FusedInstanceField(torch.autograd.Function):
    """Whole field forward (inerf_field_forward_train) / instance-head backward (inerf_field_backward_mask), one launch each.
    The table gradient (13.3 M fp32 entries) is accumulated straight into `encoder_mask.embeddings.grad` by the kernel's
    atomics -- no zero-filled temporary, no extra pass to add it -- so `None` is returned for that input."""

    @staticmethod
    def forward(ctx, model, x, d, table_mask, w0, w1, w2):
        B, K, dev = x.shape[0], model.num_instances, x.device
        sigmas = torch.empty(B, dtype=torch.float32, device=dev)
        rgbs = torch.empty(B, 3, dtype=torch.float32, device=dev)
        masks = torch.empty(B, K, dtype=torch.float32, device=dev)
        x0 = torch.empty(B, 48, dtype=torch.float16, device=dev)
        desc = model._field_desc()
        desc.n_valid = model._n_valid_ptr   # fixed-size (graph-captured) streams: rows past the marcher's device-side total are padding
        ctx.n_valid = model._n_valid_ptr
        call("inerf_field_forward_train", ctypes.byref(desc), ptr(x), ptr(d), B, ptr(sigmas), ptr(rgbs), ptr(masks), ptr(x0), stream_ptr(dev))
        ctx.model = model
        ctx.save_for_backward(x, x0)
        ctx.mark_non_differentiable(sigmas, rgbs)
        return sigmas, rgbs, masks

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_sigmas, g_rgbs, g_masks):
        x, x0 = ctx.saved_tensors
        model = ctx.model
        B, K, dev = x.shape[0], model.num_instances, x.device
        table = model.encoder_mask.embeddings
        if table.grad is None:
            table.grad = torch.zeros_like(table)
        gw0 = torch.zeros(64, 47, dtype=torch.float32, device=dev)
        gw1 = torch.zeros(64, 64, dtype=torch.float32, device=dev)
        gw2 = torch.zeros(K, 64, dtype=torch.float32, device=dev)
        if B > 0:
            desc = model._field_desc()
            desc.n_valid = ctx.n_valid
            _, wb = model._packed_weights(want_bwd=True)
            call("inerf_field_backward_mask", ctypes.byref(desc), ptr(wb), ptr(x), ptr(x0), ptr(g_masks.float().contiguous()), B,
                 ptr(table.grad), ptr(gw0), ptr(gw1), ptr(gw2), stream_ptr(dev))
        return None, None, None, None, gw0, gw1, gw2


class NeRFNetwork(NeRFMaskRenderer):
    def __init__(self, encoding="hashgrid", encoding_dir="sphere_harmonics", encoding_bg="hashgrid", num_layers=2, hidden_dim=64,
                 geo_feat_dim=15, num_layers_color=3, hidden_dim_color=64, num_layers_bg=2, hidden_dim_bg=64, num_layers_mask=3,
                 hidden_dim_mask=64, num_instances=2, bound=1, **kwargs):
        super().__init__(bound, num_instances=num_instances, **kwargs)
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

        self.num_layers_mask = num_layers_mask
        self.hidden_dim_mask = hidden_dim_mask
        self.encoder_mask, self.in_dim_mask = get_encoder(encoding, desired_resolution=2048 * bound)
        self.mask_net = nn.ModuleList([
            nn.Linear(self.in_dim_mask + geo_feat_dim if l == 0 else hidden_dim_mask,
                      num_instances if l == num_layers_mask - 1 else hidden_dim_mask, bias=False) for l in range(num_layers_mask)])

        if self.bg_radius > 0:
            # background model (network_mask.py:95-114): outside the instance-field hot path, kept modular
            self.num_layers_bg = num_layers_bg
            self.hidden_dim_bg = hidden_dim_bg
            self.encoder_bg, self.in_dim_bg = get_encoder(encoding_bg, input_dim=2, num_levels=4, log2_hashmap_size=19,
                                                          desired_resolution=2048)
            self.bg_net = nn.ModuleList([
                nn.Linear(self.in_dim_bg + self.in_dim_dir if l == 0 else hidden_dim_bg, 3 if l == num_layers_bg - 1 else hidden_dim_bg,
                          bias=False) for l in range(num_layers_bg)])
        else:
            self.bg_net = None

        self.use_fused = True     # set False to force the modular operator sequence
        # The fused kernels compute with fp16 tables / weights / activations and fp32 accumulation = the reference under
        # autocast (its `-O` / --fp16 preset, which wraps train, eval and update_extra_state in autocast).  By default every
        # no-grad CUDA call takes them; set True to take them only inside torch.autocast, so that an fp32 run (the
        # reference without --fp16) evaluates with the same fp32 numerics it trains with.
        self.fused_requires_autocast = False
        self._packed = None       # (key, forward fp16 weight blob, backward blob | None) on device
        self._tables = None       # (key, interleaved fp16 hash tables on device)
        self._work_counter = None
        self._n_valid_ptr = None  # device address of the live sample count while a fixed-size training stream is in use

    # ---- fused path ------------------------------------------------------------------
    def _standard_arch(self) -> bool:
        e = self.encoder
        return (self.num_layers == 2 and self.hidden_dim == 64 and self.geo_feat_dim == 15 and self.num_layers_color == 3
                and self.hidden_dim_color == 64 and self.num_layers_mask == 3 and self.hidden_dim_mask == 64
                and getattr(e, "num_levels", 0) == 16 and getattr(e, "level_dim", 0) == 2 and getattr(e, "gridtype", "") == "hash"
                and not e.align_corners and e.interp_id == 0 and getattr(self.encoder_dir, "degree", 0) == 4
                and 1 <= self.num_instances <= 64 and hasattr(lib(), "inerf_field_forward"))

    def fused_available(self) -> bool:
        if getattr(self, "fused_requires_autocast", False) and not torch.is_autocast_enabled():
            return False
        return bool(self.use_fused and self._standard_arch() and self.encoder.embeddings.is_cuda)

    def fused_render_available(self, render_mask: bool) -> bool:
        # the background model (bg_radius > 0) only enters through the `(1 - weights_sum) * bg_color` tail of run_cuda, which is
        # outside the kernel: the one-launch renderer serves it as well
        return self.fused_available() and hasattr(lib(), "inerf_render_fused")

    def _packed_weights(self, want_bwd: bool = False):
        """fp16 operand blobs for the tcgen05 kernels, re-packed ON THE DEVICE (one launch, no host round trip) whenever a
        weight's version counter changes -- every optimizer step while mask_net trains.  -> forward blob (, backward blob)"""
        ws = [m.weight for m in (*self.sigma_net, *self.color_net, *self.mask_net)]
        dev = ws[0].device
        key = tuple((w.data_ptr(), w._version) for w in ws) + (str(dev), PARAM_EPOCH[0])
        if self._packed is None or self._packed[0] != key or (want_bwd and self._packed[2] is None):
            K = self.num_instances
            fwd = self._packed[1] if self._packed is not None and self._packed[1].device == dev else \
                torch.empty(lib().inerf_field_weights_bytes(K), dtype=torch.uint8, device=dev)
            bwd = self._packed[2] if self._packed is not None and self._packed[2] is not None and self._packed[2].device == dev else None
            if want_bwd and bwd is None:
                bwd = torch.empty(lib().inerf_field_bwd_weights_bytes(), dtype=torch.uint8, device=dev)
            call("inerf_field_pack_weights_device", *[ptr(w.detach()) for w in ws], K, ptr(fwd), ptr(bwd), stream_ptr(dev))
            self._packed = (key, fwd, bwd)
        return (self._packed[1], self._packed[2]) if want_bwd else self._packed[1]

    def _packed_tables(self) -> torch.Tensor:
        """Interleaved fp16 copy of both hash tables, (sigma.c0, sigma.c1, mask.c0, mask.c1) per entry, refreshed only when
        a parameter changes (the reference casts both whole tables to fp16 on EVERY encoder call, grid.py:43-44)."""
        e, em = self.encoder.embeddings, self.encoder_mask.embeddings
        key = (e.data_ptr(), e._version, em.data_ptr(), em._version, str(e.device), PARAM_EPOCH[0])
        if self._tables is None or self._tables[0] != key:
            n = e.shape[0]
            out = self._tables[1] if self._tables is not None and self._tables[1].shape[0] == n and self._tables[1].device == e.device \
                else torch.empty(n, 4, dtype=torch.float16, device=e.device)
            call("inerf_field_pack_tables", ptr(e.detach()), ptr(em.detach()), 0, n, ptr(out), stream_ptr(e.device))
            self._tables = (key, out)
        return self._tables[1]

    def _field_desc(self, density_scale: float = 1.0) -> FieldDesc:
        """`density_scale` multiplies sigma inside the kernel.  The per-sample field calls (`forward`) return the UNSCALED
        sigma, as network_mask.py:119-158 does -- `run_cuda` applies `self.density_scale` itself (mask_renderer.py:273) --
        so they keep the default 1; the one-launch renderer and the occupancy sweep, which consume sigma inside the kernel,
        pass `self.density_scale`."""
        e = self.encoder
        d = FieldDesc()
        self._keepalive = (self._packed_tables(), self._packed_weights())
        d.table_packed = self._keepalive[0].data_ptr()
        d.offsets = e.offsets.data_ptr()
        d.weights = self._keepalive[1].data_ptr()
        d.L = e.num_levels
        d.H = e.base_resolution
        d.S = float(np.log2(e.per_level_scale))
        d.bound = float(self.bound)
        d.K = self.num_instances
        d.density_scale = float(density_scale)
        return d

    @torch.no_grad()
    def forward_fused(self, x, d, want_masks=True):
        x = x.float().contiguous().view(-1, 3)
        d = d.float().contiguous().view(-1, 3)
        B = x.shape[0]
        dev = x.device
        sigmas = torch.empty(B, dtype=torch.float32, device=dev)
        rgbs = torch.empty(B, 3, dtype=torch.float32, device=dev)
        masks = torch.empty(B, self.num_instances, dtype=torch.float32, device=dev) if want_masks else None
        desc = self._field_desc()
        call("inerf_field_forward", ctypes.byref(desc), ptr(x), ptr(d), B, ptr(sigmas), ptr(rgbs), ptr(masks), stream_ptr(dev))
        return sigmas, rgbs, masks

    def fused_train_available(self, x, d) -> bool:
        """Instance stage (MaskTrainer, nerf/utils.py:1242-1246): RGB-sigma nets frozen, instance head trainable, fp16 autocast
        (the `-O` preset) -> forward and backward of the whole field are ONE launch each."""
        if not (self.fused_available() and x.is_cuda and torch.is_autocast_enabled() and not x.requires_grad and not d.requires_grad):
            return False
        if not hasattr(lib(), "inerf_field_backward_mask"):
            return False
        frozen = (self.encoder, self.sigma_net, self.encoder_dir, self.color_net)
        if any(p.requires_grad for m in frozen for p in m.parameters()):
            return False
        return self.encoder_mask.embeddings.requires_grad and all(l.weight.requires_grad for l in self.mask_net)

    def bounded_stream(self) -> bool:
        """The fused training forward / backward stop at the marcher's device-side sample total (inerf_field_desc.n_valid)."""
        if not (self.fused_available() and torch.is_autocast_enabled() and hasattr(lib(), "inerf_field_backward_mask")):
            return False
        frozen = (self.encoder, self.sigma_net, self.encoder_dir, self.color_net)
        if any(p.requires_grad for m in frozen for p in m.parameters()):
            return False
        return self.encoder_mask.embeddings.requires_grad and all(l.weight.requires_grad for l in self.mask_net)

    def forward_fused_train(self, x, d):
        x = x.float().contiguous().view(-1, 3)
        d = d.float().contiguous().view(-1, 3)
        return _FusedInstanceField.apply(self, x, d, self.encoder_mask.embeddings, *[l.weight for l in self.mask_net])

    def _render_fused(self, rays_o, rays_d, nears, fars, render_mask, dt_gamma, max_steps, T_thresh, noises=None):
        N = rays_o.shape[0]
        dev = rays_o.device
        K = self.num_instances
        weights_sum = torch.empty(N, dtype=torch.float32, device=dev)
        depth = torch.empty(N, dtype=torch.float32, device=dev)
        image = torch.empty(N, 3, dtype=torch.float32, device=dev)
        mask_out = torch.empty(N, K, dtype=torch.float32, device=dev) if render_mask else None
        if self._work_counter is None or self._work_counter.device != dev:
            self._work_counter = torch.zeros(4, dtype=torch.int32, device=dev)
        desc = self._field_desc(self.density_scale)
        if noises is not None:
            noises = noises.to(device=dev, dtype=torch.float32).contiguous().view(-1)
        call("inerf_render_fused_perturb", ctypes.byref(desc), ptr(rays_o), ptr(rays_d), ptr(nears), ptr(fars), ptr(noises),
             ptr(self.density_bitfield), N, self.cascade, self.grid_size, float(dt_gamma), int(max_steps), float(T_thresh), ptr(weights_sum), ptr(depth),
             ptr(image), ptr(mask_out), ptr(self._work_counter), stream_ptr(dev))
        return weights_sum, depth, image, mask_out

    def _occupancy_density_fused(self, cells, per_cascade, noises, seed, tmp_grid) -> bool:
        """update_extra_state's density sweep as ONE launch (inerf_occupancy_density): cell -> jittered point -> hash encode ->
        sigma-net on tcgen05 -> tmp_grid[c, cell] = sigma * density_scale.  fp16 operands, i.e. what `self.density` computes
        under the reference's autocast (nerf/utils.py wraps update_extra_state in autocast(enabled=fp16))."""
        if not self.fused_available():
            return False
        desc = self._field_desc(self.density_scale)
        call("inerf_occupancy_density", ctypes.byref(desc), self.cascade, self.grid_size, ptr(cells), int(per_cascade), ptr(noises), int(seed),
             ptr(tmp_grid), stream_ptr(tmp_grid.device))
        return True

    def _extract_volume_fused(self, shape, bbox, bitfield, view_dir, sigma_thresh, sigma, rgb, label, n_live) -> bool:
        """extract_volume as ONE launch (inerf_extract_volume; plus its occupancy pre-pass when `bitfield` is given): voxel ->
        point -> hash encode -> sigma / colour / mask nets on tcgen05 -> sigma * density_scale, rgb, 1 + argmax label."""
        if not self.fused_available():
            return False
        X, Y, Z = shape
        dev = sigma.device
        scratch = None if bitfield is None else torch.empty(int(lib().inerf_extract_scratch_ints(X, Y, Z)), dtype=torch.int32, device=dev)
        desc = self._field_desc(self.density_scale)
        call("inerf_extract_volume", ctypes.byref(desc), bbox.ctypes.data, X, Y, Z, ptr(bitfield), self.cascade, self.grid_size,
             None if view_dir is None else view_dir.ctypes.data, float(sigma_thresh), ptr(sigma), ptr(rgb), ptr(label), ptr(scratch),
             ptr(n_live), stream_ptr(dev))
        return True

    # ---- reference operator sequence ----------------------------------------------------
    def _mlp(self, net, h):
        n = len(net)
        for l in range(n):
            h = net[l](h)
            if l != n - 1:
                h = F.relu(h, inplace=True)
        return h

    def forward(self, x, d):
        """x [N,3] in [-bound,bound], d [N,3] unit -> (sigma [N], rgb [N,3], mask_logits [N,K])"""
        if not torch.is_grad_enabled() and x.is_cuda and self.fused_available():
            return self.forward_fused(x, d)
        if torch.is_grad_enabled() and self.fused_train_available(x, d):
            return self.forward_fused_train(x, d)
        h = self._mlp(self.sigma_net, self.encoder(x, bound=self.bound))
        sigma = trunc_exp(h[..., 0])
        geo_feat = h[..., 1:]
        h = self._mlp(self.color_net, torch.cat([self.encoder_dir(d), geo_feat], dim=-1))
        color = torch.sigmoid(h)
        m = torch.cat([self.encoder_mask(x, bound=self.bound), geo_feat], dim=-1)
        mask_logits = self._mlp(self.mask_net, m)
        return sigma, color, mask_logits

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

    def mask(self, x, mask=None, geo_feat=None, **kwargs):
        if mask is not None:
            mask_logits = torch.zeros(mask.shape[0], self.num_instances, dtype=x.dtype, device=x.device)
            if not mask.any():
                return mask_logits
            x, geo_feat = x[mask], geo_feat[mask]
        h = self._mlp(self.mask_net, torch.cat([self.encoder_mask(x, bound=self.bound), geo_feat], dim=-1))
        if mask is not None:
            mask_logits[mask] = h.to(mask_logits.dtype)
            return mask_logits
        return h

    def get_params(self, lr):
        params = [
            {"params": self.encoder.parameters(), "lr": lr},
            {"params": self.sigma_net.parameters(), "lr": lr},
            {"params": self.encoder_dir.parameters(), "lr": lr},
            {"params": self.color_net.parameters(), "lr": lr},
            {"params": self.encoder_mask.parameters(), "lr": lr},
            {"params": self.mask_net.parameters(), "lr": lr},
        ]
        if self.bg_radius > 0:
            params.append({"params": self.encoder_bg.parameters(), "lr": lr})
            params.append({"params": self.bg_net.parameters(), "lr": lr})
        return params
