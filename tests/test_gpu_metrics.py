"""GPU: the evaluator's distortion metrics (reference Evaluator.py:26-92) on the device against oracle/metrics.py.
MS-SSIM restates the absent third-party `pytorch_msssim` (parity unpinned by the reference); PSNR / luma follow Evaluator.py."""
import numpy as np
import pytest
import torch

from oracle import metrics as OM
from oracle import metrics_np as ON
from tests import helpers as H

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("shape", [(1, 3, 512, 768), (2, 3, 203, 181), (1, 3, 161, 400)])
def test_compute_metrics_matches_the_oracle(shape, tmp_path):
    from neural_image_compression_b200.Evaluator import CompressionEvaluator, ms_ssim
    torch.manual_seed(sum(shape))
    orig = torch.rand(*shape)
    raw = orig + 0.08 * torch.randn_like(orig)                  # leaves [0, 1]: the evaluator clamps (Evaluator.py:73)
    ref = OM.compute_metrics(orig, raw.clamp(0, 1))
    ev = CompressionEvaluator(None, None, "cuda", 0.005, save_dir=str(tmp_path))
    got = ev.compute_metrics(orig.cuda(), raw.cuda(), clamp=True)
    got2 = ev.compute_metrics(orig.cuda(), raw.clamp(0, 1).cuda())          # the reference's own call pattern
    assert set(got) == set(ref) == {"MSE(255)", "PSNR(RGB)", "MS-SSIM(RGB)", "PSNR(Y)", "MS-SSIM(Y)"}
    for k in ref:
        tol = 2e-5 if "SSIM" in k else 1e-4 * abs(ref[k])
        assert abs(got[k] - ref[k]) <= tol and abs(got2[k] - ref[k]) <= tol, (k, got[k], got2[k], ref[k])
    # per-image values (size_average=False) and the luma helper
    per = ms_ssim(raw.clamp(0, 1).cuda(), orig.cuda(), size_average=False).cpu()
    np.testing.assert_allclose(per.numpy(), OM.ms_ssim(raw.clamp(0, 1), orig, size_average=False).numpy(), atol=2e-5)
    np.testing.assert_allclose(ev.rgb_to_luma(orig.cuda()).cpu().numpy(), OM.rgb_to_luma(orig).numpy(), atol=1e-6)
    assert abs(float(ms_ssim(orig.cuda(), orig.cuda())) - 1.0) < 1e-6
    # ... and against the second, independent (float64 numpy / scipy) statement of the algorithm
    assert abs(got["MS-SSIM(RGB)"] - ON.ms_ssim(raw.clamp(0, 1).numpy(), orig.numpy())) <= 2e-5


def test_ms_ssim_rejects_small_images_like_the_reference_package():
    from neural_image_compression_b200.Evaluator import ms_ssim
    with pytest.raises(AssertionError):
        ms_ssim(torch.rand(1, 3, 160, 300).cuda(), torch.rand(1, 3, 160, 300).cuda())


def test_evaluate_loop_keeps_the_reference_report_and_its_bpp_quirk(tmp_path):
    """Evaluator.py:55-92 on two synthetic 'Kodak' images; 'BPP' is the mean of bpp_y as in the reference (:81) unless fix_bpp."""
    from neural_image_compression_b200.Evaluator import CompressionEvaluator
    from neural_image_compression_b200.RateDistortionLoss import rd_loss
    model = H.seeded_model(128, 3, "calib", precision="bf16x3").cuda()
    loader = [H.seeded_input((1, 3, 256, 192)), H.seeded_input((1, 3, 192, 256)) * 0.5]
    ev = CompressionEvaluator(model, loader, "cuda", 0.005, save_dir=str(tmp_path))
    avg, imgs, recons = ev.evaluate(rd_loss)
    assert set(avg) == {"MSE(255)", "PSNR(RGB)", "MS-SSIM(RGB)", "PSNR(Y)", "MS-SSIM(Y)", "BPP", "BPP(y)", "BPP(z)"}
    assert avg["BPP"] == avg["BPP(y)"] and len(imgs) == len(recons) == 2 and float(recons[0].max()) <= 1.0
    fixed, _, _ = ev.evaluate(rd_loss, fix_bpp=True)
    assert abs(fixed["BPP"] - (fixed["BPP(y)"] + fixed["BPP(z)"])) < 1e-6
    # the metrics of the first image against the oracle on the same tensors
    with torch.no_grad():
        x = loader[0].cuda()
        xh = model(x, training=False)["x_hat"].clamp(0, 1).cpu()
    ref = OM.compute_metrics(loader[0], xh)
    got = ev.compute_metrics(x, xh.cuda())
    for k in ref:
        assert abs(got[k] - ref[k]) <= (2e-5 if "SSIM" in k else 1e-4 * abs(ref[k])), (k, got[k], ref[k])
