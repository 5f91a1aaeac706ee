"""CPU: the closed-form MS-SSIM backward (oracle/ms_ssim_bwd.py, the derivation nic_ms_ssim_bwd implements) against float64
autograd over oracle.metrics.ms_ssim, and the host-side validation of the MS-SSIM loss before any launch."""
import pytest
import torch

from oracle import metrics as OM
from oracle import ms_ssim_bwd as MB


def _pair(shape, kind):
    torch.manual_seed(7)
    y = torch.rand(*shape, dtype=torch.float64)
    x = (y + 0.05 * torch.randn_like(y)).float().double()        # x plays x_hat: unclamped
    if kind == "relu":                                            # cs_l < 0 at every level of image 0: its channels are zeroed
        x[0] = 1 - y[0]
    elif kind == "last":                                          # image 0, plane 0: only the last level's ssim is <= 0
        x[0, 0] = y[0, 0] - 1
    return x, y


@pytest.mark.parametrize("hw", [(161, 161), (161, 203), (256, 256)])
@pytest.mark.parametrize("c", [1, 3])
@pytest.mark.parametrize("kind", ["noise", "relu", "last"])
def test_closed_form_backward_matches_float64_autograd(hw, c, kind):
    x, y = _pair((2, c) + hw, kind)
    t = MB.level_stats(x, y)
    if kind == "last":
        assert (t[:4, 0, 0] > 0).all() and t[4, 0, 0] <= 0, t[:, 0, 0]
    if kind == "relu":
        assert (t[:, 0] < 0).any(0).all()
    xr = x.clone().requires_grad_(True)
    OM.ms_ssim(xr, y).backward()
    ref = xr.grad
    got = MB.ms_ssim_grad(x, y)
    assert float((got - ref).norm()) <= 1e-10 * float(ref.norm()), float((got - ref).norm() / ref.norm())
    if kind != "noise":                                           # the relu rule: a channel with a term <= 0 has no gradient
        zero = (t <= 0).any(0)
        assert torch.equal(got[zero], torch.zeros_like(got[zero])) and torch.equal(ref[zero], torch.zeros_like(ref[zero]))
        assert float(ref[~zero].abs().max()) > 0


def test_level_stats_and_term_grads_match_the_device_combination():
    """Evaluator.combine_levels / term_grads (the torch ops the loss runs on the device) against the oracle, on level means
    with a non-positive term."""
    from neural_image_compression_b200.Evaluator import combine_levels, term_grads
    x, y = _pair((2, 3, 161, 203), "last")
    t = MB.level_stats(x, y).float()                              # [5, 2, 3]
    lev = torch.zeros(5, 6, 2)
    lev[:4, :, 1] = t[:4].reshape(4, 6)
    lev[4, :, 0] = t[4].reshape(6)
    terms, val = combine_levels(lev)
    want = torch.prod(torch.relu(t.double()) ** torch.tensor(OM.WEIGHTS, dtype=torch.float64).view(-1, 1, 1), 0).reshape(6)
    torch.testing.assert_close(val.double(), want, rtol=1e-6, atol=0)
    torch.testing.assert_close(term_grads(terms, val).double(), MB.term_grads(t.double()).reshape(5, 6), rtol=1e-5, atol=0)
    assert float(term_grads(terms, val)[:, 0].abs().max()) == 0.0


def test_small_images_are_rejected_before_any_launch():
    from neural_image_compression_b200.RateDistortionLoss import check_ms_ssim_shape, ms_ssim_rd_loss
    from neural_image_compression_b200.training import step_gradients
    for shape in [(1, 3, 160, 256), (2, 3, 256, 160), (1, 3, 64, 64)]:
        with pytest.raises(ValueError, match="160"):
            check_ms_ssim_shape(shape)
        x = torch.zeros(shape)                                    # CPU tensors: any launch would fail with another error
        with pytest.raises(ValueError, match="160"):
            ms_ssim_rd_loss({"x_hat": x, "logp_y": x, "logp_z": x}, x, 1.0)
        with pytest.raises(ValueError, match="160"):
            step_gradients(object(), x, 1.0, distortion="ms-ssim")
    check_ms_ssim_shape((1, 3, 161, 161))
    with pytest.raises(ValueError, match="distortion"):
        step_gradients(object(), torch.zeros(1, 3, 256, 256), 1.0, distortion="ssim")


def test_trainer_rejects_unknown_distortions_and_the_scalable_model():
    from neural_image_compression_b200 import parallel
    from neural_image_compression_b200.Models import JointAutoregressiveHierarchical, ScalableImageCoding
    torch.manual_seed(0)
    model = JointAutoregressiveHierarchical(128, K=3)
    for bad in ("MS-SSIM", "ssim", "l1", None):
        with pytest.raises(ValueError, match="distortion"):
            parallel.ShardedTrainer(model, 1.0, distortion=bad)
    assert parallel.ShardedTrainer(model, 1.0, distortion="ms-ssim").distortion == "ms-ssim"
    scal = ScalableImageCoding(192, 128, K=1)
    with pytest.raises(ValueError, match="ScalableImageCoding"):
        parallel.ShardedTrainer(scal, 1.0, distortion="ms-ssim")
    with pytest.raises(ValueError, match="distortion"):
        parallel.ShardedTrainer(scal, 1.0, distortion="psnr")
    assert parallel.ShardedTrainer(scal, 1.0).distortion == "mse"
