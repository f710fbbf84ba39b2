"""NeRFRenderer / NeRFMaskRenderer for the B200 path.

Keeps the reference's API (nerf/renderer.py:61-573, nerf/mask_renderer.py:62-589):
`render / run / run_cuda / update_extra_state / mark_untrained_grid /
reset_extra_state`, the same keyword arguments, return-dict keys, buffers
(`aabb_train aabb_infer density_grid density_bitfield step_counter`) and Python
state (`mean_density iter_density mean_count local_step`), so Trainer /
MaskTrainer (nerf/utils.py:1299,1387,1421) run unmodified.

What changed underneath:
* every op goes through libinerf_b200 (hand-written sm_100a kernels);
* inference `run_cuda` is ONE persistent kernel launch (march + hash encode +
  tcgen05 MLP + composite per 128-ray tile) when the network supports the fused
  path (`fused_render_available`), instead of a host loop with two device syncs
  per iteration (mask_renderer.py:342-374).  The reference loop is kept as
  `run_cuda_loop` (used for parity tests and non-standard configurations);
* the occupancy EMA + packbits tail runs as two launches with no `.item()`.
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn as nn

from .. import raymarching
from .._lib import call, lib, ptr, stream_ptr


def _host_seed() -> int:
    """63-bit seed for the counter-based device generators, drawn from torch's default CPU generator (so
    `torch.manual_seed` makes the occupancy sampling reproducible) without touching the GPU."""
    return int(torch.empty((), dtype=torch.int64).random_().item())


def sample_pdf(bins, weights, n_samples, det=False):
    """Inverse-CDF sampling of `n_samples` depths per ray from the piecewise-constant density `weights` over `bins`
    (mask_renderer.py:13-47; `run(upsample_steps > 0)`).  bins [N, B], weights [N, B - 1] -> [N, n_samples]."""
    w = weights + 1e-5                                           # no empty bin
    cdf = torch.cumsum(w / w.sum(-1, keepdim=True), -1)
    cdf = torch.nn.functional.pad(cdf, (1, 0))                   # cdf[..., 0] = 0: one value per bin edge
    N, E = cdf.shape
    if det:
        u = torch.linspace(0.5 / n_samples, 1.0 - 0.5 / n_samples, steps=n_samples, device=w.device).expand(N, n_samples)
    else:
        u = torch.rand(N, n_samples, device=w.device)
    u = u.contiguous()
    hi = torch.searchsorted(cdf, u, right=True)                  # first edge with cdf > u
    lo = (hi - 1).clamp(min=0)
    hi = hi.clamp(max=E - 1)
    c0, c1 = cdf.gather(1, lo), cdf.gather(1, hi)
    b0, b1 = bins.gather(1, lo), bins.gather(1, hi)
    span = c1 - c0
    span = torch.where(span < 1e-5, torch.ones_like(span), span)
    return b0 + (u - c0) / span * (b1 - b0)


def alpha_weights(z_vals, last_delta, sigma, density_scale):
    """Compositing weights of sorted depths (mask_renderer.py:131-137 = :164-170): delta_i = z_{i+1} - z_i (the last interval
    is `last_delta`), alpha = 1 - exp(-delta * density_scale * sigma), w_i = alpha_i * prod_{j<i} (1 - alpha_j + 1e-15)."""
    deltas = torch.cat([z_vals[..., 1:] - z_vals[..., :-1], last_delta * torch.ones_like(z_vals[..., :1])], dim=-1)
    alphas = 1 - torch.exp(-deltas * density_scale * sigma)
    trans = torch.cumprod(torch.cat([torch.ones_like(alphas[..., :1]), 1 - alphas + 1e-15], dim=-1), dim=-1)[..., :-1]
    return alphas * trans, deltas


class NeRFRenderer(nn.Module):
    """Base renderer (nerf/renderer.py:61-123 ctor + state) with the instance-mask
    extensions of NeRFMaskRenderer folded in: `render_mask=False` gives the plain
    RGB-sigma behaviour of the base class."""

    def __init__(self, bound=1, cuda_ray=False, density_scale=1, min_near=0.2, density_thresh=0.01, bg_radius=-1, num_instances=2):
        super().__init__()
        self.bound = bound
        self.cascade = 1 + math.ceil(math.log2(bound))
        self.grid_size = 128
        self.density_scale = density_scale
        self.min_near = min_near
        self.density_thresh = density_thresh
        self.bg_radius = bg_radius
        self.num_instances = num_instances

        aabb_train = torch.FloatTensor([-bound, -bound, -bound, bound, bound, bound])
        self.register_buffer("aabb_train", aabb_train)
        self.register_buffer("aabb_infer", aabb_train.clone())

        self.cuda_ray = cuda_ray
        if cuda_ray:
            self.register_buffer("density_grid", torch.zeros([self.cascade, self.grid_size ** 3]))
            self.register_buffer("density_bitfield", torch.zeros(self.cascade * self.grid_size ** 3 // 8, dtype=torch.uint8))
            self._mean_density = 0
            self.iter_density = 0
            self.register_buffer("step_counter", torch.zeros(16, 2, dtype=torch.int32))
            self._mean_count = 0
            self.local_step = 0

    # mean_density is produced on the device by the fused EMA kernel; it is read back only when somebody asks.
    @property
    def mean_density(self):
        if isinstance(self._mean_density, torch.Tensor):
            self._mean_density = float(self._mean_density.item())
        return self._mean_density

    @mean_density.setter
    def mean_density(self, v):
        self._mean_density = v

    # -- network hooks (implemented by NeRFNetwork) ---------------------------------
    def forward(self, x, d):
        raise NotImplementedError()

    def density(self, x):
        raise NotImplementedError()

    def color(self, x, d, mask=None, **kwargs):
        raise NotImplementedError()

    def mask(self, x, mask=None, **kwargs):
        raise NotImplementedError()

    def fused_render_available(self, render_mask: bool) -> bool:
        return False

    def reset_extra_state(self):
        if not self.cuda_ray:
            return
        self.density_grid.zero_()
        self.mean_density = 0
        self.iter_density = 0
        self.step_counter.zero_()
        self.mean_count = 0
        self.local_step = 0

    # -- non-cuda_ray renderer (mask_renderer.py:89-231) ------------------------------
    def run(self, rays_o, rays_d, render_mask=False, num_steps=128, upsample_steps=128, bg_color=None, perturb=False, **kwargs):
        """Dense renderer without the occupancy grid: `num_steps` uniform depths per ray between the box entry and exit,
        optionally `upsample_steps` more drawn from the coarse weights, density everywhere, colour / instance logits only
        where the weight exceeds 1e-4."""
        prefix = rays_o.shape[:-1]
        rays_o = rays_o.contiguous().view(-1, 3)
        rays_d = rays_d.contiguous().view(-1, 3)
        N, device = rays_o.shape[0], rays_o.device
        aabb = self.aabb_train if self.training else self.aabb_infer
        lo, hi = aabb[:3], aabb[3:]

        def points(z):      # [N, S] depths -> [N, S, 3] positions clipped to the box
            return torch.min(torch.max(rays_o.unsqueeze(-2) + rays_d.unsqueeze(-2) * z.unsqueeze(-1), lo), hi)

        def query(x, S):    # density head on [N, S, 3] -> dict of [N, S, c]
            return {k: v.view(N, S, -1) for k, v in self.density(x.reshape(-1, 3)).items()}

        nears, fars = raymarching.near_far_from_aabb(rays_o, rays_d, aabb, self.min_near)
        nears, fars = nears.unsqueeze(-1), fars.unsqueeze(-1)
        span = fars - nears
        sample_dist = span / num_steps
        z_vals = nears + span * torch.linspace(0.0, 1.0, num_steps, device=device).unsqueeze(0).expand((N, num_steps))
        if perturb:
            z_vals = z_vals + (torch.rand(z_vals.shape, device=device) - 0.5) * sample_dist
        xyzs = points(z_vals)
        fields = query(xyzs, num_steps)

        if upsample_steps > 0:
            with torch.no_grad():
                weights, deltas = alpha_weights(z_vals, sample_dist, fields["sigma"].squeeze(-1), self.density_scale)
                mids = z_vals[..., :-1] + 0.5 * deltas[..., :-1]
                new_z = sample_pdf(mids, weights[:, 1:-1], upsample_steps, det=not self.training).detach()
                new_xyzs = points(new_z)
            new_fields = query(new_xyzs, upsample_steps)
            z_vals, order = torch.sort(torch.cat([z_vals, new_z], dim=1), dim=1)      # merge coarse and fine samples by depth

            def merged(a, b):
                both = torch.cat([a, b], dim=1)
                return torch.gather(both, dim=1, index=order.unsqueeze(-1).expand_as(both))

            xyzs = merged(xyzs, new_xyzs)
            fields = {k: merged(fields[k], new_fields[k]) for k in fields}

        weights, _ = alpha_weights(z_vals, sample_dist, fields["sigma"].squeeze(-1), self.density_scale)
        visible = (weights > 1e-4).reshape(-1)
        flat = {k: v.reshape(-1, v.shape[-1]) for k, v in fields.items()}
        pts = xyzs.reshape(-1, 3)
        rgbs = self.color(pts, rays_d.view(-1, 1, 3).expand_as(xyzs).reshape(-1, 3), mask=visible, **flat).view(N, -1, 3)

        weights_sum = weights.sum(dim=-1)
        depth = torch.sum(weights * ((z_vals - nears) / span).clamp(0, 1), dim=-1)
        image = torch.sum(weights.unsqueeze(-1) * rgbs, dim=-2)
        if self.bg_radius > 0:
            bg_color = self.background(raymarching.sph_from_ray(rays_o, rays_d, self.bg_radius), rays_d.reshape(-1, 3))
        elif bg_color is None:
            bg_color = 1
        image = image + (1 - weights_sum).unsqueeze(-1) * bg_color

        logits = None
        if render_mask:
            per_sample = self.mask(pts, mask=visible, **flat).view(N, -1, self.num_instances)
            logits = torch.sum(weights.unsqueeze(-1) * per_sample, dim=-2).view(*prefix, self.num_instances)
        return {"depth": depth.view(*prefix), "image": image.view(*prefix, 3), "instance_mask_logits": logits, "weights_sum": weights_sum}

    # -- cuda_ray renderer (mask_renderer.py:234-387) --------------------------------
    def run_cuda(self, rays_o, rays_d, render_mask=False, dt_gamma=0, bg_color=None, perturb=False, force_all_rays=False,
                 max_steps=1024, T_thresh=1e-4, **kwargs):
        prefix = rays_o.shape[:-1]
        rays_o = rays_o.contiguous().view(-1, 3)
        rays_d = rays_d.contiguous().view(-1, 3)
        N = rays_o.shape[0]

        nears, fars = raymarching.near_far_from_aabb(rays_o, rays_d, self.aabb_train if self.training else self.aabb_infer,
                                                     self.min_near)
        if self.bg_radius > 0:
            sph = raymarching.sph_from_ray(rays_o, rays_d, self.bg_radius)
            bg_color = self.background(sph, rays_d)
        elif bg_color is None:
            bg_color = 1

        results = {}
        if self.training:
            counter = self.step_counter[self.local_step % 16]
            counter.zero_()
            self.local_step += 1
            budget = int(getattr(self, "sample_budget", 0) or 0)
            # every consumer of the stream stops at the device-side total (fused field forward / backward, n_valid): rows past it
            # are never read, so neither the stream nor the compositing gradients need zero fills
            bounded = budget > 0 and self.bounded_stream()
            if budget > 0:
                # fixed-size sample stream (CUDA-graph-captured training step, nerf/trainer.py): `budget` rows, no host read of
                # the marched total; the field kernels stop at the device-side total (counter[0]), rows beyond it are padding.
                # The caller guarantees budget >= total (and checks counter[0] afterwards), so no ray is dropped.
                xyzs, dirs, deltas, rays = raymarching.march_rays_train(
                    rays_o, rays_d, self.bound, self.density_bitfield, self.cascade, self.grid_size, nears, fars, counter,
                    budget, perturb, -1, False, dt_gamma, max_steps, noises=kwargs.get("noises"), zero_fill=not bounded)
                self._n_valid_ptr = counter.data_ptr()
            else:
                xyzs, dirs, deltas, rays = raymarching.march_rays_train(
                    rays_o, rays_d, self.bound, self.density_bitfield, self.cascade, self.grid_size, nears, fars, counter,
                    -1 if force_all_rays else self.mean_count, perturb, 128, force_all_rays, dt_gamma, max_steps,
                    noises=kwargs.get("noises"))
                self._n_valid_ptr = None
            sigmas, rgbs, masks = self._field(xyzs, dirs, render_mask)
            sigmas = self.density_scale * sigmas
            # fixed-size stream: every row below the device-side total belongs to a ray and the rows above it are never read, so
            # the compositing backward needs no zero-filled gradient buffers (the eager stream has zero-padded alignment rows
            # that ARE fed through the network backward: it keeps the reference's zero fill)
            dense = bounded
            if not render_mask:
                weights_sum, depth, image = raymarching.composite_rays_train(sigmas, rgbs, deltas, rays, T_thresh, dense=dense)
            else:
                weights_sum, depth, image, mask_out = raymarching.composite_rays_with_masks_train(
                    sigmas, rgbs, masks, deltas, rays, T_thresh, dense=dense)
            results["weights_sum"] = weights_sum
        else:
            # perturb (mask_renderer.py:334-337): one uniform draw per ray jitters the first step; `noises` (extra) injects it
            noises = kwargs.get("noises")
            if noises is None and perturb:
                noises = torch.rand(N, dtype=torch.float32, device=rays_o.device)
            if self.fused_render_available(render_mask):
                weights_sum, depth, image, mask_out = self._render_fused(rays_o, rays_d, nears, fars, render_mask, dt_gamma,
                                                                         max_steps, T_thresh, noises=noises)
            else:
                weights_sum, depth, image, mask_out = self.run_cuda_loop(rays_o, rays_d, nears, fars, render_mask, dt_gamma,
                                                                         perturb, max_steps, T_thresh, noises=noises)

        image = image + (1 - weights_sum).unsqueeze(-1) * bg_color
        depth = torch.clamp(depth - nears, min=0) / (fars - nears)
        results["depth"] = depth.view(*prefix)
        results["image"] = image.view(*prefix, 3)
        results["instance_mask_logits"] = mask_out.view(*prefix, self.num_instances) if render_mask else None
        return results

    def bounded_stream(self) -> bool:
        """True when the network's training forward / backward honour `_n_valid_ptr` (see NeRFNetwork in network_mask.py)."""
        return False

    def _field(self, xyzs, dirs, render_mask):
        out = self(xyzs, dirs)
        if len(out) == 3:
            return out
        return out[0], out[1], None  # stage-1 network: (sigma, rgb)

    def run_cuda_loop(self, rays_o, rays_d, nears, fars, render_mask, dt_gamma, perturb, max_steps, T_thresh, noises=None):
        """The reference's alive-ray loop (mask_renderer.py:330-374) on this library's kernels, with the
        same n_step schedule; compaction and the alive count stay on the device except for ONE 4-byte
        read per iteration (the reference pays two syncs: `.shape` of a boolean-indexed tensor, :345,:370)."""
        N = rays_o.shape[0]
        device = rays_o.device
        K = self.num_instances
        weights_sum = torch.zeros(N, dtype=torch.float32, device=device)
        depth = torch.zeros(N, dtype=torch.float32, device=device)
        image = torch.zeros(N, 3, dtype=torch.float32, device=device)
        mask_out = torch.zeros(N, K, dtype=torch.float32, device=device) if render_mask else None

        n_alive = N
        rays_alive = torch.arange(n_alive, dtype=torch.int32, device=device)
        rays_t = nears.clone()
        step = 0
        while step < max_steps and n_alive > 0:
            n_step = max(min(N // n_alive, 8), 1)
            xyzs, dirs, deltas = raymarching.march_rays(n_alive, n_step, rays_alive, rays_t, rays_o, rays_d, self.bound,
                                                        self.density_bitfield, self.cascade, self.grid_size, nears, fars, 128,
                                                        perturb if step == 0 else False, dt_gamma, max_steps,
                                                        noises=noises if step == 0 else None)
            sigmas, rgbs, masks = self._field(xyzs, dirs, render_mask)
            sigmas = self.density_scale * sigmas
            if not render_mask:
                raymarching.composite_rays(n_alive, n_step, rays_alive, rays_t, sigmas, rgbs, deltas, weights_sum, depth, image,
                                           T_thresh)
            else:
                raymarching.composite_rays_with_masks(n_alive, n_step, K, rays_alive, rays_t, sigmas, rgbs, masks, deltas,
                                                      weights_sum, depth, image, mask_out, T_thresh)
            rays_alive, n_out = raymarching.compact_alive(rays_alive, n_alive)
            n_alive = int(n_out.item())
            step += n_step
        return weights_sum, depth, image, mask_out

    def _render_fused(self, rays_o, rays_d, nears, fars, render_mask, dt_gamma, max_steps, T_thresh, noises=None):
        raise NotImplementedError()

    # -- occupancy grid lifecycle ------------------------------------------------------
    @torch.no_grad()
    def mark_untrained_grid(self, poses, intrinsic, S=64):
        """mask_renderer.py:389-452: cells whose centre no training camera sees get density -1 and can never become
        occupied.  One kernel, one thread per (cascade, cell) looping over the cameras (the reference: five nested Python
        loops of meshgrid / batched matmul / index_put).  `S` (the reference's batching knob) is accepted and ignored.
        The number of marked cells stays on the device in `self.n_untrained` (the reference prints it)."""
        if not self.cuda_ray:
            return
        if isinstance(poses, np.ndarray):
            poses = torch.from_numpy(poses)
        fx, fy, cx, cy = (float(v) for v in intrinsic)
        grid = self.density_grid
        dev = grid.device
        poses = poses.to(dev).float().contiguous().view(-1, 4, 4)
        self.n_untrained = torch.zeros(1, dtype=torch.int32, device=dev)
        call("inerf_mark_untrained_grid", ptr(poses), poses.shape[0], fx, fy, cx, cy, self.cascade, self.grid_size, float(self.bound),
             ptr(grid), ptr(self.n_untrained), stream_ptr(dev))

    # mean_count (samples per batch, averaged over the last <= 16 steps) is only consumed as a host int by the budgeted
    # marcher (`force_all_rays=False`, raymarching.py:200-203): it is kept on the device and read back when asked for.
    @property
    def mean_count(self):
        if isinstance(self._mean_count, torch.Tensor):
            self._mean_count = int(self._mean_count.item())
        return self._mean_count

    @mean_count.setter
    def mean_count(self, v):
        self._mean_count = v

    def _occupancy_density_fused(self, cells, per_cascade, noises, seed, tmp_grid) -> bool:
        """Hook: networks with a fused density sweep fill `tmp_grid` and return True (NeRFNetwork)."""
        return False

    @torch.no_grad()
    def sweep_cells(self, uniform_cells=None, occ_picks=None):
        """Cells re-sampled by a partial update (mask_renderer.py:498-513) -> int32 [C, 2N] Morton indices, N = G^3 / 4:
        N uniform cells, then N occupied cells (density_grid > 0) drawn with replacement.  `uniform_cells` / `occ_picks`
        [C, N] inject the two randint draws of the reference (parity tests); otherwise they come from a counter-based
        generator seeded from torch's default generator.  Everything, including the occupied-cell count, stays on the device."""
        dev = self.density_grid.device
        C, G = self.cascade, self.grid_size
        N = G ** 3 // 4
        cells = torch.empty(C, 2 * N, dtype=torch.int32, device=dev)
        n_scr = int(lib().inerf_occupancy_sample_scratch_ints(C, G))
        scr = getattr(self, "_occ_scratch", None)
        if scr is None or scr.numel() < n_scr or scr.device != dev:
            scr = self._occ_scratch = torch.empty(n_scr, dtype=torch.int32, device=dev)
        # both converted tensors must stay alive until the launch is queued (a temporary freed between the two conversions would
        # hand its block to the second one)
        uni = None if uniform_cells is None else uniform_cells.to(device=dev, dtype=torch.int32).contiguous()
        picks = None if occ_picks is None else occ_picks.to(device=dev, dtype=torch.int32).contiguous()
        call("inerf_occupancy_sample_cells", ptr(self.density_grid), C, G, N, ptr(uni), ptr(picks), _host_seed(), ptr(cells), ptr(scr),
             stream_ptr(dev))
        return cells

    @torch.no_grad()
    def update_extra_state(self, decay=0.95, S=128, noises=None, cells=None):
        """mask_renderer.py:454-548 with no Python loop and no host read: the first 16 calls sweep every cell of every
        cascade, later calls re-sample G^3/4 random + G^3/4 occupied cells per cascade (`sweep_cells`); each sample's
        jittered point, its density and the scatter into `tmp_grid` are ONE launch when the network has a fused density
        sweep, else point kernel -> `self.density` -> index_put; then EMA / mean / threshold / packbits (`ema_update_`).

        Extra, optional: `noises` [C * per_cascade, 3] in [0, 1) replaces the jitter draws and `cells` [C, 2N] the
        partial update's cell choice (parity tests); sample s = (cascade s // per_cascade, cell cells[s] or s % G^3).
        `S` (the reference's block size) is accepted and ignored."""
        if not self.cuda_ray:
            return
        grid = self.density_grid
        dev = grid.device
        C, G = self.cascade, self.grid_size
        st = stream_ptr(dev)
        tmp_grid = torch.empty_like(grid)
        if self.iter_density < 16:
            cells, per_cascade = None, G ** 3          # every cell is written: no -1 fill needed
        else:
            if cells is None:
                cells = self.sweep_cells()
            cells = cells.to(device=dev, dtype=torch.int32).contiguous()
            per_cascade = cells.numel() // C
            call("inerf_fill_f32", ptr(tmp_grid), tmp_grid.numel(), -1.0, st)
        if noises is not None:
            noises = noises.to(device=dev, dtype=torch.float32).contiguous().view(-1, 3)
            if noises.shape[0] != C * per_cascade:
                raise ValueError(f"noises must have {C * per_cascade} rows, got {noises.shape[0]}")
        seed = _host_seed()
        if not self._occupancy_density_fused(cells, per_cascade, noises, seed, tmp_grid):
            n = C * per_cascade
            xyzs = torch.empty(n, 3, dtype=torch.float32, device=dev)
            flat = torch.empty(n, dtype=torch.int32, device=dev)
            call("inerf_occupancy_points", C, G, float(self.bound), ptr(cells), per_cascade, ptr(noises), seed, ptr(xyzs), ptr(flat), st)
            sigmas = self.density(xyzs)["sigma"].reshape(-1).detach().float() * self.density_scale
            tmp_grid.view(-1)[flat.long()] = sigmas
        self.ema_update_(tmp_grid, decay)
        self.iter_density += 1

        total_step = min(16, self.local_step)
        if total_step > 0:   # floor of the mean, as int(sum / total_step); read back only if somebody asks (mean_count property)
            self._mean_count = torch.div(self.step_counter[:total_step, 0].sum(), total_step, rounding_mode="floor")
        self.local_step = 0

    @torch.no_grad()
    def ema_update_(self, tmp_grid, decay=0.95):
        """density_grid = max(density_grid*decay, tmp) where both >= 0; mean; threshold; packbits
        (mask_renderer.py:532-540) -- all on the device."""
        grid = self.density_grid
        n_cells = grid.numel()
        dev = grid.device
        total = torch.zeros(1, dtype=torch.float64, device=dev)
        mean = torch.empty(1, dtype=torch.float32, device=dev)
        st = stream_ptr(dev)
        call("inerf_occupancy_ema", ptr(grid), ptr(tmp_grid.contiguous()), n_cells, float(decay), ptr(total), st)
        call("inerf_occupancy_pack", ptr(grid), n_cells, ptr(total), float(self.density_thresh), ptr(self.density_bitfield),
             ptr(mean), st)
        self._mean_density = mean

    # -- volume extraction ------------------------------------------------------------------
    def _extract_volume_fused(self, shape, bbox, bitfield, view_dir, sigma_thresh, sigma, rgb, label, n_live) -> bool:
        """Hook: networks with the fused extraction kernel fill the outputs and return True (NeRFNetwork)."""
        return False

    @torch.no_grad()
    def extract_volume(self, resolution, bbox=None, view_dir=None, sigma_thresh=None, skip_empty=True, labels=True, chunk=1 << 20):
        """The trained fields on an X x Y x Z voxel grid over `bbox` (default `aabb_infer`; 6 floats lo xyz, hi xyz, inside
        [-bound, bound]^3): voxel (i, j, k) sits at lo + (i, j, k) / (X, Y, Z) * (hi - lo), the geometry and label convention of
        `projection.project_rays` / `project_masks`, so the label volume projects into any view unchanged.

        -> {"sigma": float32 [X, Y, Z] (density * density_scale), "label": int32 [X, Y, Z] (1 + argmax of the instance logits
        where sigma >= sigma_thresh, else 0; only with `labels`), "rgb": float32 [X, Y, Z, 3] (the colour seen along the unit
        direction `view_dir`; only when it is given), "bbox": the 6 floats used, "n_live": device int32 [1], voxels evaluated}.

        skip_empty (cuda_ray models): voxels whose occupancy cell is empty are not evaluated and come out 0 everywhere.
        sigma_thresh: default min(mean_density, density_thresh), the threshold the occupancy bitfield was packed with.
        Each of the two defaults costs one host read of a device value (aabb_infer, mean_density); a call that passes `bbox` and
        `sigma_thresh` (host values) does not synchronise with the device.  One fused launch (plus an occupancy pre-pass) when the network has the fused field;
        otherwise inerf_volume_points -> the network's forward under fp16 autocast in chunks of `chunk` voxels -> the same rules
        in torch, on the GPU."""
        X, Y, Z = (int(resolution),) * 3 if isinstance(resolution, int) else (int(r) for r in resolution)
        bb = self.aabb_infer.tolist() if bbox is None else torch.as_tensor(bbox, dtype=torch.float32).reshape(6).tolist()
        bb = tuple(float(v) for v in bb)
        bb_host = np.ascontiguousarray(bb, dtype=np.float32)
        vd = None if view_dir is None else np.ascontiguousarray(torch.as_tensor(view_dir, dtype=torch.float32).cpu().reshape(3).numpy())
        gated = bool(skip_empty and self.cuda_ray)
        if sigma_thresh is None:
            sigma_thresh = min(float(self.mean_density), float(self.density_thresh)) if self.cuda_ray else float(self.density_thresh)
        dev = self.aabb_infer.device
        bitfield = self.density_bitfield if gated else None
        sigma = torch.empty(X, Y, Z, dtype=torch.float32, device=dev)
        rgb = torch.empty(X, Y, Z, 3, dtype=torch.float32, device=dev) if vd is not None else None
        label = torch.empty(X, Y, Z, dtype=torch.int32, device=dev) if labels else None
        n_live = torch.empty(1, dtype=torch.int32, device=dev)
        if not self._extract_volume_fused((X, Y, Z), bb_host, bitfield, vd, float(sigma_thresh), sigma, rgb, label, n_live):
            n = X * Y * Z
            xyzs = torch.empty(n, 3, dtype=torch.float32, device=dev)
            occupied = torch.empty(n, dtype=torch.uint8, device=dev)
            call("inerf_volume_points", bb_host.ctypes.data, X, Y, Z, ptr(bitfield), self.cascade if gated else 0,
                 self.grid_size if gated else 0, float(self.bound), ptr(xyzs), ptr(occupied), stream_ptr(dev))
            live = occupied.bool()
            d = torch.tensor([0.0, 0.0, 1.0] if vd is None else vd.tolist(), dtype=torch.float32, device=dev).expand(min(n, chunk), 3)
            s_flat, c_flat = sigma.view(-1), None if rgb is None else rgb.view(-1, 3)
            l_flat = None if label is None else label.view(-1)
            for i in range(0, n, chunk):
                j = min(n, i + chunk)
                with torch.autocast("cuda", dtype=torch.float16):
                    out = self(xyzs[i:j], d[:j - i])
                s = out[0].float() * self.density_scale
                s_flat[i:j] = torch.where(live[i:j], s, 0.0)
                if c_flat is not None:
                    c_flat[i:j] = torch.where(live[i:j, None], out[1].float(), 0.0)
                if l_flat is not None:
                    arg = torch.argmax(out[2], dim=-1).to(torch.int32) + 1
                    l_flat[i:j] = torch.where(live[i:j] & (s >= sigma_thresh), arg, 0)
            n_live.copy_(live.sum().view(1))
        out = {"sigma": sigma, "bbox": bb, "n_live": n_live}
        if label is not None:
            out["label"] = label
        if rgb is not None:
            out["rgb"] = rgb
        return out

    @torch.no_grad()
    def extract_mesh(self, resolution=256, bbox=None, threshold=10, view_dir=None, labels=True, skip_empty=True):
        """A triangle mesh of the density surface, with the fields at its vertices: extract_volume's sigma on the voxel grid
        -> marching cubes at iso = threshold * density_scale (the reference's save_mesh threshold applies to the density
        before density_scale; extract_volume's sigma includes it) -> the field at every vertex.

        -> {"verts": float32 [V, 3], "faces": int32 [F, 3] (normals toward low density), "bbox", "iso",
        "rgb": float32 [V, 3] (colour seen along `view_dir`; only when it is given),
        "vertex_label": int32 [V] (1 + argmax of the instance logits, lowest index on ties) and "face_label": int32 [F]
        (majority of the face's vertex labels, the smallest when all three differ); both only with `labels`}.

        The vertex fields come from the fused field forward when the network has it, else from the network's forward under
        fp16 autocast.  A call that passes `bbox` reads the device once (the mesh size)."""
        vol = self.extract_volume(resolution, bbox=bbox, sigma_thresh=0.0, skip_empty=skip_empty, labels=False)
        iso = float(threshold) * float(self.density_scale)
        from ..mesh import face_labels, mesh_from_volume
        out = mesh_from_volume(vol["sigma"], vol["bbox"], iso)
        out.update(bbox=vol["bbox"], iso=iso)
        if view_dir is None and not labels:
            return out
        verts = out["verts"]
        d = torch.empty_like(verts)
        for a, c in enumerate((0.0, 0.0, 1.0) if view_dir is None else torch.as_tensor(view_dir, dtype=torch.float32).reshape(3).tolist()):
            d[:, a] = float(c)
        if verts.shape[0] == 0:
            rgb, logits = torch.empty_like(verts), torch.empty(0, 1, device=verts.device)
        elif self.fused_available():
            _, rgb, logits = self.forward_fused(verts, d, want_masks=labels)
        else:
            with torch.autocast("cuda", dtype=torch.float16):
                f = self(verts, d)
            rgb, logits = f[1].float(), f[2] if labels else None
        if view_dir is not None:
            out["rgb"] = rgb
        if labels:
            vl = torch.argmax(logits, dim=-1).to(torch.int32) + 1
            out["vertex_label"] = vl
            out["face_label"] = face_labels(vl, out["faces"])
        return out

    # -- entry point (mask_renderer.py:551-589) ------------------------------------------
    def render(self, rays_o, rays_d, staged=False, max_ray_batch=4096, render_mask=False, **kwargs):
        _run = self.run_cuda if self.cuda_ray else self.run
        B, N = rays_o.shape[:2]
        device = rays_o.device
        if staged and not self.cuda_ray:
            depth = torch.empty((B, N), device=device)
            image = torch.empty((B, N, 3), device=device)
            mask_logits = torch.empty((B, N, self.num_instances), device=device) if render_mask else None
            for b in range(B):
                head = 0
                while head < N:
                    tail = min(head + max_ray_batch, N)
                    r = _run(rays_o[b:b + 1, head:tail], rays_d[b:b + 1, head:tail], render_mask, **kwargs)
                    depth[b:b + 1, head:tail] = r["depth"]
                    image[b:b + 1, head:tail] = r["image"]
                    if render_mask:
                        mask_logits[b:b + 1, head:tail] = r["instance_mask_logits"]
                    head += max_ray_batch
            return {"depth": depth, "image": image, "instance_mask_logits": mask_logits}
        return _run(rays_o, rays_d, render_mask, **kwargs)


class NeRFMaskRenderer(NeRFRenderer):
    """Name kept for drop-in compatibility with nerf/mask_renderer.py:62."""
