"""CPU suite: the oracle against the golden fixtures the real reference produced
(oracle/pin_against_reference.py), and the analytic identities of the hot path."""
import numpy as np
import pytest
import torch

import nirgan_oracle as O


def _sd(shapes, g):
    return O.random_state_dict(shapes, seed=int(g["sd_seed"]), bias_std=float(g["bias_std"]))


def test_generator_goldens(golden_dir):
    g = np.load(f"{golden_dir}/g_plain_64.npz")
    sd = _sd(O.generator_param_shapes(), g)
    x = torch.from_numpy(g["x"])
    with torch.no_grad():
        assert float((O.resnet_generator_forward(sd, x) - torch.from_numpy(g["y"])).abs().max()) <= 2e-5
        gp = np.load(f"{golden_dir}/g_plain_64_pad10.npz")
        assert float((O.px2px_forward(sd, x, 10) - torch.from_numpy(gp["y"])).abs().max()) <= 2e-5


@pytest.mark.parametrize("scale", [0.01, 1.0])
def test_inject_goldens(golden_dir, scale):
    g = np.load(f"{golden_dir}/g_inject_64_s{scale}.npz")
    sd = _sd(O.generator_param_shapes(inject=True), g)
    sd["scale_param"] = torch.tensor(float(g["scale"]))
    with torch.no_grad():
        y = O.resnet_generator_forward(sd, torch.from_numpy(g["x"]), embeds=torch.from_numpy(g["embeds"]))
    assert float((y - torch.from_numpy(g["y"])).abs().max()) <= 2e-5


def test_discriminator_and_losses_goldens(golden_dir):
    g = np.load(f"{golden_dir}/d_64.npz")
    sd = _sd(O.discriminator_param_shapes(), g)
    with torch.no_grad():
        y = O.patchgan_forward(sd, torch.from_numpy(g["x"]))
    assert float((y - torch.from_numpy(g["y"])).abs().max()) <= 2e-5
    l = np.load(f"{golden_dir}/losses.npz")
    rgb, nir, pred = (torch.from_numpy(l[k]) for k in ("rgb", "nir", "pred"))
    for name, fn in (("ndvi", O.ndvi_pair), ("ndwi", O.ndwi_pair), ("evi", O.evi_pair)):
        a, b = fn(rgb, nir, pred)
        assert abs(float((a - b).abs().mean()) - float(l[name])) <= 1e-6 * max(1.0, abs(float(l[name])))
    assert abs(float(O.lsgan_loss(torch.from_numpy(l["d_out"]), True)) - float(l["lsgan_real"])) <= 1e-7


def test_training_step_golden(golden_dir):
    g = np.load(f"{golden_dir}/train_step_64.npz")
    sd_g = O.random_state_dict(O.generator_param_shapes(), seed=int(g["sd_g_seed"]))
    sd_d = O.random_state_dict(O.discriminator_param_shapes(), seed=int(g["sd_d_seed"]))
    tr = O.OracleTrainer(sd_g, sd_d)
    out = tr.step(torch.from_numpy(g["rgb"]), torch.from_numpy(g["nir"]))
    assert abs(float(out["loss_D"]) - float(g["loss_D"])) <= 1e-5
    assert abs(float(out["loss_G"]) - float(g["loss_G"])) <= 1e-4 * abs(float(g["loss_G"]))
    assert float((out["pred"] - torch.from_numpy(g["pred"])).abs().max()) <= 2e-5
    k = "model.26.weight"
    ref = torch.from_numpy(g["gG." + k])
    assert float((out["grads_g"][k][:8] - ref).norm() / ref.norm()) <= 1e-3
    k = "model.11.weight"
    ref = torch.from_numpy(g["gD." + k])
    assert float((out["grads_d"][k][:8] - ref).norm() / ref.norm()) <= 1e-4
    assert float((tr.d["model.11.weight"].detach() - torch.from_numpy(g["newD.model.11.weight"])).abs().max()) <= 1e-6


def test_synth_loop_golden_and_ordering(golden_dir):
    g = np.load(f"{golden_dir}/synth_loop_32.npz")
    sd = _sd(O.generator_param_shapes(), g)
    names = [f"tile_{i:06d}.tif" for i in (3, 0, 2, 1, 4)]
    tiles = {n: torch.rand(3, 32, 32, generator=torch.Generator().manual_seed(100 + int(n[5:11]))) for n in names}
    out = O.synth_loop(sd, tiles, 2, 10)
    assert list(out.keys()) == list(g["ids"]) == [f"tile_{i:06d}" for i in range(5)]
    for k in out:
        assert float((out[k] - torch.from_numpy(g["y." + k])).abs().max()) <= 2e-5


def test_flop_model_matches_survey():
    assert abs(O.g_forward_gflop(256, 256) - 98.281) < 0.01
    assert abs(O.g_forward_gflop(276, 276) - 114.237) < 0.01
    assert abs(O.g_forward_gflop(532, 532) - 424.436) < 0.05


def test_pre_norm_bias_is_cancelled_by_instance_norm():
    """The kernels skip the bias add of convs that feed InstanceNorm (DESIGN.md): perturbing those
    biases must not change the oracle's output beyond rounding."""
    sd = O.random_state_dict(O.generator_param_shapes(), seed=5)
    x = torch.rand(1, 3, 32, 32, generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        y0 = O.resnet_generator_forward(sd, x)
        sd2 = dict(sd)
        for k in sd:
            if k.endswith("bias") and not k.startswith("model.26") and not k.startswith("fc"):
                sd2[k] = torch.randn(sd[k].shape, generator=torch.Generator().manual_seed(1))
        y1 = O.resnet_generator_forward(sd2, x)
    assert float((y0 - y1).abs().max()) < 5e-5


def test_oracle_matches_reference_modules_when_present(golden_dir):
    """The oracle port against the outputs of the reference's own define_G_inject / define_D modules (stored in
    tests/golden by oracle/pin_against_reference.py) at 5e-6, four times tighter than the fixture tests above: the
    SatCLIP-injected generator with scale 1.0 and the PatchGAN discriminator with non-zero biases."""
    g = np.load(f"{golden_dir}/g_inject_64_s1.0.npz")
    sd = _sd(O.generator_param_shapes(inject=True), g)
    sd["scale_param"] = torch.tensor(float(g["scale"]))
    with torch.no_grad():
        got = O.resnet_generator_forward(sd, torch.from_numpy(g["x"]), embeds=torch.from_numpy(g["embeds"]))
    assert float((got - torch.from_numpy(g["y"])).abs().max()) <= 5e-6
    gd = np.load(f"{golden_dir}/d_64.npz")
    assert float(gd["bias_std"]) > 0
    sdd = _sd(O.discriminator_param_shapes(), gd)
    with torch.no_grad():
        got = O.patchgan_forward(sdd, torch.from_numpy(gd["x"]))
    assert float((got - torch.from_numpy(gd["y"])).abs().max()) <= 5e-6
