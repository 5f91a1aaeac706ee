"""GPU: ScalableImageCoding (BASELINE.json configs[4]'s model, reference Models.py:208-338 with the repairs of SURVEY.md
section 2.4) through the module API -> C ABI, against vectors produced by the reference's own sub-modules."""
import numpy as np
import pytest
import torch

from tests import helpers as H

pytestmark = pytest.mark.gpu


ARMS = ("fp32", "bf16x3")       # CUDA cores / tensor cores with hi/lo-split operands: both parity grade


@pytest.mark.parametrize("precision", ARMS)
@pytest.mark.parametrize("case", H.scalable_cases())
def test_scalable_model_matches_reference_vectors(case, precision):
    from neural_image_compression_b200.RateDistortionLoss import vision_rd_loss
    g = H.load_golden(case)
    M, M1, K, init = int(g["M"]), int(g["M1"]), int(g["K"]), str(g["init"])
    model = H.seeded_scalable_model(M, M1, K, init, precision=precision).cuda()
    x = torch.from_numpy(g["x"]).cuda()
    out = model(x, training=False)
    rd = vision_rd_loss(out, x, 0.005, 0.0)
    ref = {k[4:]: g[k] for k in g.files if k.startswith("out_")}
    want = set(ref) | {"training"}
    assert set(out) == want, set(out) ^ want
    for k, v in out.items():
        if torch.is_tensor(v):
            assert v.dtype == torch.float32 and tuple(v.shape) == tuple(ref[k].shape), k
    o = {k: out[k].cpu().numpy() for k in ("y", "y_in", "z", "z_in", "p_y1", "p_y2", "p_z", "x_hat")}
    rep, flips = {"precision": precision}, 0
    for name, pre in (("y_in", "y"), ("z_in", "z")):
        real, ties = H.symbol_mismatches(o[name], ref[name], ref[pre], H.TIE_TAU)
        rep[name + "_flips_real_ties"] = [real, ties]
        flips += ties
        assert real == 0, (name, real, ties)
        assert ties <= H.tie_flip_bound(o[pre], ref[pre]), (name, ties)
        rel = float(np.abs(o[pre] - ref[pre]).max() / np.abs(ref[pre]).max())
        rep[pre + "_rel_err"] = rel
        assert rel <= H.PRE_RTOL[pre], (pre, rel)
    assert torch.equal(torch.cat([out["y1"], out["y2"]], dim=1), out["y_in"])
    # per-element likelihoods / x_hat: (a) against the reference's vectors off the footprints of flipped symbols (a symbol of
    # either head's channel range only reaches that head's context conv, but the masks are per pixel: conservative), at the
    # main model's bounds (1e-5 outliers, both arms); (b) if anything flipped, everywhere against the oracle on this run's symbols
    ok_y, ok_z, ok_x = H.flip_masks(o["y_in"], ref["y_in"], o["z_in"], ref["z_in"], ref["x_hat"].shape)
    x_tol = 1e-4 if precision == "fp32" else 3e-4
    for name, ok in (("p_y1", ok_y), ("p_y2", ok_y), ("p_z", ok_z)):
        bad, worst, n, frac = H.masked_likelihood_close(o[name], ref[name], ok)
        rep[name] = {"outliers": bad, "max_abs_err": worst, "compared": n, "fraction": frac}
        assert bad <= 1e-5 * n + 1, (name, bad, n, worst)
    okx = np.broadcast_to(ok_x, ref["x_hat"].shape)
    if okx.any():
        xe = float(np.abs(o["x_hat"] - ref["x_hat"])[okx].max() / np.abs(ref["x_hat"]).max())
        rep["x_hat"] = {"rel_err": xe, "fraction": float(okx.mean())}
        assert xe < x_tol, xe
    if flips:
        want_given = H.oracle_scalable_given_symbols(model.state_dict(), o["y_in"], o["z_in"], M, M1, K)
        for name in ("p_y1", "p_y2", "p_z"):
            bad, worst = H.likelihood_close(o[name], want_given[name])
            rep[name + "_given_symbols"] = {"outliers": bad, "max_abs_err": worst}
            assert bad <= 1e-5 * want_given[name].size + 1, (name, bad, worst)
        xe2 = float(np.abs(o["x_hat"] - want_given["x_hat"]).max() / np.abs(want_given["x_hat"]).max())
        rep["x_hat_given_symbols_rel_err"] = xe2
        assert xe2 < x_tol, xe2
    H.record_report(f"scalable/{case}/{precision}", rep)
    for key in ("bpp_y1", "bpp_y2", "bpp_z", "bpp_total"):
        assert abs(rd[key] - float(g["rd_" + key])) <= H.BPP_TOL, (key, rd[key], float(g["rd_" + key]))
    assert abs(rd["psnr"] - float(g["rd_psnr"])) <= H.PSNR_TOL
    assert abs(float(rd["loss"]) - float(g["rd_loss"])) <= 1e-3 * abs(float(g["rd_loss"]))
    print(case, {k: rd[k] for k in ("bpp_y1", "bpp_y2", "bpp_z", "psnr")})


def test_scalable_rejects_bad_arguments_and_ignores_lst_keys():
    from neural_image_compression_b200.Models import ScalableImageCoding
    with pytest.raises(ValueError):
        ScalableImageCoding(192, 192)
    with pytest.raises(ValueError):
        ScalableImageCoding(192, 128, K=0)
    m = ScalableImageCoding(192, 128, K=1)
    sd = dict(m.state_dict())
    sd["LST.net.0.weight"] = torch.zeros(1)          # a reference checkpoint carries the latent-space-transform entries
    m.load_state_dict(sd)


@pytest.mark.parametrize("precision", ARMS)
def test_scalable_full_size_image_properties(precision):
    """BASELINE configs[4] shape (2048 x 1536), one image per GPU: size-independent properties instead of an oracle run."""
    from neural_image_compression_b200.RateDistortionLoss import vision_rd_loss
    model = H.seeded_scalable_model(192, 128, 1, "calib", precision=precision).cuda()
    x = H.seeded_input((1, 3, 1536, 2048)).cuda()
    out = model(x, training=False)
    rd = vision_rd_loss(out, x, 0.005, 0.0)
    assert tuple(out["y"].shape) == (1, 192, 96, 128) and tuple(out["z"].shape) == (1, 192, 24, 32)
    assert tuple(out["p_y1"].shape) == (1, 128, 96, 128) and tuple(out["p_y2"].shape) == (1, 64, 96, 128)
    assert torch.equal(torch.round(out["y"]), out["y_in"]) and torch.equal(torch.cat([out["y1"], out["y2"]], 1), out["y_in"])
    for k in ("p_y1", "p_y2", "p_z"):
        assert float(out[k].min()) >= float(np.float32(1e-9)) and float(out[k].max()) <= 1 + 1e-6
        assert torch.allclose(out["logp" + k[1:]], torch.log(out[k]), atol=1e-6)
    bits = -(out["logp_y1"].double().sum() + out["logp_y2"].double().sum() + out["logp_z"].double().sum()) / np.log(2.0)
    assert abs(float(bits) / (1536 * 2048) - rd["bpp_total"]) < 1e-4
    mse = float(((out["x_hat"].double() - x.double()) ** 2).mean())
    assert abs(mse - rd["mse"]) < 1e-5 * mse
    # a crop-aligned sub-image gives the same interior symbols: the path is convolutional (receptive field << 512 px margin)
    sub = model(x[:, :, :1024, :1024].contiguous(), training=False)
    assert torch.equal(sub["y_in"][:, :, :32, :32], out["y_in"][:, :, :32, :32])
    # timing of the full-size forward (CUDA events, second call): the tensor-core arm against the CUDA-core arm
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); model(x, training=False); e1.record(); torch.cuda.synchronize()
    print(f"ScalableImageCoding(192, 128, K=1) 2048x1536 forward, {precision}: {e0.elapsed_time(e1):.1f} ms")


def test_scalable_training_step_gradients():
    """Forward with noise + vision_rd_loss + hand-written backward of the two-head model (training_scalable.step_gradients) against
    autograd over the oracle's repaired forward.  Weight set: well conditioned at 192 channels (tests/helpers.py: calib192)."""
    from oracle import backward as OB
    from neural_image_compression_b200.training_scalable import step_gradients
    model = H.seeded_scalable_model(192, 128, 1, "calib192", precision="bf16x3")
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    x = H.seeded_input((1, 3, 128, 128))
    torch.manual_seed(17)
    nz, ny = torch.rand(1, 192, 2, 2) - 0.5, torch.rand(1, 192, 8, 8) - 0.5
    ref_rd, ref_g = OB.loss_and_grads_scalable(sd, x, 192, 128, 1, nz, ny, 0.005)
    model = model.cuda()
    loss, terms = step_gradients(model, x.cuda(), 0.005, noise=(nz.cuda(), ny.cuda()))
    torch.cuda.synchronize()
    assert abs(float(loss) - ref_rd["loss"]) <= 1e-4 * abs(ref_rd["loss"]), (float(loss), ref_rd["loss"])
    assert abs(float(terms["bpp_y1"]) - ref_rd["bpp_y1"]) < 1e-4 and abs(float(terms["bpp_y2"]) - ref_rd["bpp_y2"]) < 1e-4
    names = dict(model.named_parameters())
    assert set(ref_g) == set(names)
    worst = {}
    for k, p in names.items():
        assert p.grad is not None, k
        worst[k] = float((p.grad.double().cpu() - ref_g[k].double()).norm() / max(float(ref_g[k].double().norm()), 1e-30))
    print(sorted(worst.items(), key=lambda kv: -kv[1])[:6])
    for k, e in worst.items():
        exposed = k.startswith(("hyper_encoder.", "hyper_decoder.", "context_model", "entropy_parameters_1.net.0", "entropy_parameters_1.net.2",
                                "entropy_parameters_2.net.0", "entropy_parameters_2.net.2"))
        assert e < (3e-2 if exposed else 1e-3), (k, e)           # LeakyReLU kinks: tests/test_gpu_train.py grad_tol


@pytest.mark.parametrize("graph", [False, True])
def test_scalable_trainer_steps(graph):
    """parallel.ShardedTrainer drives the two-head model too (eagerly and as a CUDA-graph replay): the loss goes down, the step
    counter advances on the device and the parameters move by ~lr per step.  graph=True also runs the eager trainer and compares,
    as tests/test_gpu_train.py::test_graphed_trainer_steps_like_the_eager_one does for the single-head model (the captured step
    runs g_s and the weight gradients on parallel branches; the noise is drawn inside the graph, so the check is statistical):
    same first loss within the noise spread, and the loss goes down over 30 steps like the eager trainer's.  The loss of one step
    of this model swings by up to ~10 % with the noise draw, so the two trainers are compared over their last ten steps."""
    from neural_image_compression_b200 import parallel
    x = H.seeded_input((2, 3, 128, 128)).cuda()
    losses = {}
    for mode in sorted({False, graph}):
        model = H.seeded_scalable_model(192, 128, 1, "calib192", precision="bf16x3").cuda()
        w0 = model.decoder.net[6].weight.detach().clone()
        tr = parallel.ShardedTrainer(model, 0.005, lr=1e-4, graph=mode)
        losses[mode] = [float(tr.step(x)["loss"]) for _ in range(30)]
        torch.cuda.synchronize()
        assert tr.optimizer.t == 30 and int(tr.optimizer._t_dev) == 30 and losses[mode][-1] < losses[mode][0], losses[mode]
        moved = float((model.decoder.net[6].weight.detach() - w0).abs().max())
        assert 5e-4 < moved <= 30 * 3.2e-4, moved            # Adam: a few lr per step at most, and the weights did move
    if graph:
        assert abs(losses[True][0] - losses[False][0]) < 0.02 * losses[False][0], (losses[True][0], losses[False][0])
        late = {mode: sum(ls[-10:]) / 10 for mode, ls in losses.items()}
        assert late[True] < losses[True][0] and abs(late[True] - late[False]) < 0.05 * late[False], (late, losses)


def test_scalable_autograd_path_equals_step_gradients():
    """model(x) with autograd on + vision_rd_loss(...)['loss'].backward() (the reference trainer's calls) deposit the same gradients
    as the autograd-free step, and the training dict has the reference's keys."""
    from neural_image_compression_b200.RateDistortionLoss import vision_rd_loss
    from neural_image_compression_b200.training_scalable import step_gradients
    model = H.seeded_scalable_model(192, 128, 3, "calib192", precision="bf16x3").cuda()
    x = H.seeded_input((1, 3, 64, 128)).cuda()
    torch.manual_seed(23)
    noise = (torch.rand(1, 192, 1, 2).cuda() - 0.5, torch.rand(1, 192, 4, 8).cuda() - 0.5)
    out = model(x, noise=noise)
    assert set(out) == {"x_hat", "y", "y_in", "y1", "y2", "z", "z_in", "p_z", "logp_z", "p_y1", "logp_y1", "p_y2", "logp_y2", "training",
                        "weights1", "mus1", "sigmas1", "weights2", "mus2", "sigmas2"}
    assert out["logp_y1"].requires_grad and out["x_hat"].requires_grad and not out["y_in"].requires_grad
    rd = vision_rd_loss(out, x, 0.005)
    rd["loss"].backward()
    ref = {k: p.grad.clone() for k, p in model.named_parameters()}
    model.zero_grad()
    loss, _ = step_gradients(model, x, 0.005, noise=noise)
    torch.cuda.synchronize()
    assert abs(float(loss) - float(rd["loss"].detach())) <= 1e-6 * abs(float(loss))
    for k, p in model.named_parameters():
        assert torch.allclose(p.grad, ref[k], rtol=1e-6, atol=0), k


def test_graphed_forward_matches_the_eager_call_and_follows_weight_changes():
    """parallel.GraphedForward: the scalable model's forward replayed from a CUDA graph (with g_s as a parallel branch) returns
    the eager call's tensors bit for bit, and re-captures after load_state_dict."""
    from neural_image_compression_b200 import parallel
    model = H.seeded_scalable_model(192, 128, 1, "calib", precision="bf16x3").cuda()
    x = H.seeded_input((1, 3, 128, 192)).cuda()
    eager = model(x, training=False)
    gf = parallel.GraphedForward(model)
    for _ in range(2):
        out = gf(x)
    torch.cuda.synchronize()
    for k in ("x_hat", "y_in", "z_in", "p_y1", "p_y2", "p_z"):
        assert torch.equal(out[k], eager[k]), k
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    sd["entropy_parameters_1.net.4.bias"] = sd["entropy_parameters_1.net.4.bias"] + 0.25
    model.load_state_dict(sd)
    out2 = gf(x)
    torch.cuda.synchronize()
    assert torch.equal(out2["p_y1"], model(x, training=False)["p_y1"]) and not torch.equal(out2["p_y1"], eager["p_y1"])
