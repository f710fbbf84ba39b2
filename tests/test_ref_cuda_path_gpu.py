"""Full-frame parity of the product against the REFERENCE's own CUDA path on the headline configuration (SURVEY.md section 8d,
BASELINE.md B2): frame 0 of c2 -- 640x480, K = 32, bound 8, 4 x 128^3 occupancy grid, 16-level 2^19 hash grids -- rendered
(a) by the reference's kernels built unmodified into oracle/_ref, driven by the reference's run_cuda alive-ray loop with the MLPs
as nn.Linear under fp16 autocast (oracle/ref_cuda_path.py), and (b) by NeRFNetwork.render -> inerf_render_fused (one launch).
(a) is recorded in tests/golden/recorded_test_ref_cuda_path_gpu.npz (helpers.Recorded): a fixed sample of image, depth and
instance probabilities, and the instance argmax of every pixel.
North-star tolerance: image / depth / instance probabilities within 1e-3, instance argmax identical."""
import pytest
import torch

pytestmark = pytest.mark.gpu

# First-step loss of the reference-kernel training step (oracle/ref_cuda_path.RefPath.train_step) on the batch, weights and
# jitter of test_reference_train_step_runs_and_matches_product_loss, measured on a B200.
REFERENCE_FIRST_STEP_LOSS = 3.4657630920410156


def test_c2_frame_matches_reference_cuda_path(recorded, cuda):
    import bench
    from instance_nerf_b200.nerf.utils import get_rays
    model, scene, poses = bench.build_scene_and_model(cuda)
    r = get_rays(poses[0:1].to(cuda), bench.intrinsics(), bench.H_IMG, bench.W_IMG)
    o, d = r["rays_o"].view(-1, 3), r["rays_d"].view(-1, 3)
    kw = dict(dt_gamma=bench.DT_GAMMA, max_steps=bench.MAX_STEPS, T_thresh=bench.T_THRESH)
    with torch.no_grad():
        got = model.render(o[None], d[None], staged=True, render_mask=True, perturb=False, bg_color=1, **kw)
    assert o.shape[0] == 307200
    tol = dict(rtol=0.0, atol=1e-3, sample=1024)
    recorded.close("image", got["image"][0], **tol)
    recorded.close("depth", got["depth"][0], **tol)
    recorded.close("instance_prob", torch.softmax(got["instance_mask_logits"][0], -1), **tol)
    recorded.exact("instance_argmax", got["instance_mask_logits"][0].argmax(-1).to(torch.uint8))


def test_reference_train_step_runs_and_matches_product_loss(cuda):
    """The product's training step (MaskTrainStep) computes the same first-step loss as the reference-kernel training step
    (the baseline bench.py times next to the product's step) on identical weights, rays, labels and jitter."""
    import bench
    from instance_nerf_b200.nerf.trainer import MaskTrainStep
    model, scene, poses = bench.build_scene_and_model(cuda)
    batch = bench.train_batches(cuda, scene, poses, 1024, 0, 1, n=1)[0]
    batch["noises"] = torch.rand(1024, device=cuda, generator=torch.Generator(device=cuda).manual_seed(2))
    kw = dict(dt_gamma=bench.DT_GAMMA, max_steps=bench.MAX_STEPS, T_thresh=bench.T_THRESH)
    l_ref = REFERENCE_FIRST_STEP_LOSS
    tr = MaskTrainStep(model, lr=1e-2, fp16=True, patch_size=8, label_regularization_weight=0.1, **kw)
    l_ours = float(tr.step(batch))
    print(f"[train step] first-step loss: reference kernels {l_ref:.6f}, product {l_ours:.6f}")
    assert abs(l_ours - l_ref) <= 2e-3 * max(1.0, abs(l_ref))
