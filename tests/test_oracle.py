"""Pins the CPU oracle (oracle/vd_oracle.py) against the golden fixtures that oracle/make_golden.py produced by
running the UNMODIFIED reference, and against the known-answer constants of SURVEY.md §8c.  fp32 vs fp32: tolerance is
op-reordering round-off."""
import json
import os

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def _close(a, b, rtol=2e-4, what=""):
    a, b = torch.as_tensor(a).float(), torch.as_tensor(b).float()
    err = (a - b).abs().max().item()
    scale = b.abs().max().item() + 1e-12
    assert err <= rtol * scale, f"{what}: {err:.3g} vs scale {scale:.3g}"


@pytest.fixture(scope="module")
def mini():
    from oracle import weights
    from oracle.make_golden import golden_inputs, WEIGHT_SEED
    shapes = {k: tuple(v) for k, v in json.load(open(os.path.join(GOLD, "keys_mini.json"))).items()}
    sd = weights.synth_state_dict(shapes, seed=WEIGHT_SEED)
    return sd, golden_inputs("mini"), dict(np.load(os.path.join(GOLD, "mini.npz")))


def test_schedule_known_answers():
    from oracle import vd_oracle as O
    sched = json.load(open(os.path.join(GOLD, "schedule.json")))
    ddpm = O.ddpm_schedule()
    assert abs(float(ddpm["betas"][0]) - 0.00085) < 1e-9 and abs(float(ddpm["betas"][999]) - 0.012) < 1e-8
    assert abs(float(ddpm["alphas_cumprod"][0]) - 0.99915) < 1e-6
    assert abs(float(ddpm["alphas_cumprod"][999]) - 0.004660098513) < 1e-9
    np.testing.assert_allclose([float(ddpm["betas"][0]), float(ddpm["betas"][999])], sched["betas_0_999"], rtol=0, atol=0)
    # SURVEY §8c KATs (probed from the reference)
    kat = {50: dict(a=[0.998296022, 0.980380774, 0.00728172716, 0.00577550009], p=[0.999149978, 0.998296022, 0.00911730994, 0.00728172716],
                    s=[0.0412792638, 0.14006865, 0.996352494, 0.997108042]),
           10: dict(a=[0.998296022, 0.892980516, 0.0365465246, 0.0140048983], p=[0.999149978, 0.998296022, 0.0819167122, 0.0365465246],
                    s=[0.0412792638, 0.327138335, 0.981556654, 0.992972851])}
    for steps in (50, 10):
        o = O.ddim_schedule(ddpm["alphas_cumprod"], steps)
        g = sched[str(steps)]
        assert list(o["timesteps"]) == g["timesteps"]
        assert g["timesteps"][:3] == ([1, 21, 41] if steps == 50 else [1, 101, 201])
        for k in ("alphas", "alphas_prev", "sigmas", "sqrt_one_minus_alphas"):
            np.testing.assert_array_equal(np.asarray(o[k], dtype=np.float32), np.asarray(g[k], dtype=np.float32))
        idx = [0, 1, -2, -1]
        np.testing.assert_allclose(o["alphas"][idx], kat[steps]["a"], rtol=2e-7)
        np.testing.assert_allclose(o["alphas_prev"][idx], kat[steps]["p"], rtol=2e-7)
        np.testing.assert_allclose(o["sqrt_one_minus_alphas"][idx], kat[steps]["s"], rtol=2e-7)
        assert not np.any(o["sigmas"])


def test_unet_forward_vs_reference_golden(mini):
    from oracle import vd_oracle as O
    sd, gi, gold = mini
    with torch.no_grad():
        _close(O.apply_model(sd, gi["x"], gi["t"], [gi["c_text"]], model_channels=64), gold["eps_text"], what="text ctx")
        _close(O.apply_model(sd, gi["x"], gi["t"], [gi["c_img"]], c_types=("image",), model_channels=64), gold["eps_image"], what="image ctx")
        _close(O.apply_model(sd, gi["x"], gi["t"], [gi["c_text"], gi["c_img"]], ratios=[0.7, 0.3], c_types=("text", "image"),
                             model_channels=64), gold["eps_dual"], what="dual ctx mix")
        _close(O.timestep_embedding(torch.tensor([1, 21, 501, 981]), 320), gold["t_emb"], rtol=1e-6, what="t_emb")


def test_ddim_trajectory_vs_reference_golden(mini):
    from oracle import vd_oracle as O
    sd, gi, gold = mini
    with torch.no_grad():
        x, trace = O.ddim_sample(sd, gi["xT"], [gi["c"]], [gi["u"]], 5, 7.5, collect=True, model_channels=64)
    _close(x, gold["ddim5_final"], rtol=1e-3, what="final latent")
    _close(torch.stack([t["pred_x0"] for t in trace]), gold["ddim5_pred_x0"], rtol=1e-3, what="pred_x0 trace")


def test_vae_vs_reference_golden(mini):
    from oracle import vd_oracle as O
    sd, gi, gold = mini
    with torch.no_grad():
        _close(O.vae_decode(sd, gi["z"]), gold["vae_decode"], what="vae_decode")
        mean = O.vae_encode(sd, gi["img"], noise=None) / 0.18215
    _close(mean, gold["vae_moments"][:, :4], what="vae_encode mean")


def test_c1_full_size_vs_reference_golden():
    """BASELINE config 1 end to end on the oracle at full size (about a minute of CPU)."""
    from oracle import vd_oracle as O, weights
    from oracle.make_golden import golden_inputs, WEIGHT_SEED
    gold = dict(np.load(os.path.join(GOLD, "c1_full.npz")))
    shapes = {k: tuple(v) for k, v in json.load(open(os.path.join(GOLD, "keys_full.json"))).items()}
    sd = weights.synth_state_dict(shapes, seed=WEIGHT_SEED)
    gi = golden_inputs("c1")
    with torch.no_grad():
        eps0 = O.apply_model(sd, torch.cat([gi["xT"]] * 2), torch.tensor([901, 901]), [torch.cat([gi["u"], gi["c"]])])
        _close(eps0, gold["eps0"], what="C1 eps0")
        img = O.vae_decode(sd, torch.as_tensor(gold["final"]))
    assert (img - torch.as_tensor(gold["image"].astype(np.float32))).abs().max().item() <= 2e-3   # fp16-stored fixture


def test_reference_golden_matches_oracle_on_fresh_inputs():
    """The oracle against the unmodified reference's outputs (ref_cases.npz) on other weights and shapes than mini.npz: an odd
    latent shape and context length, vae_decode, the img2img start, the dual-context sampler and the text-latent flows."""
    from oracle import vd_oracle as O, weights
    from oracle.make_golden import golden_inputs, REF_CASES_SEEDS
    gold = {k: torch.as_tensor(v) for k, v in np.load(os.path.join(GOLD, "ref_cases.npz")).items()}
    fi = golden_inputs("fresh")
    shapes = {k: tuple(v) for k, v in json.load(open(os.path.join(GOLD, "keys_mini.json"))).items()}
    sd = weights.synth_state_dict(shapes, seed=REF_CASES_SEEDS["image"])
    with torch.no_grad():
        _close(O.apply_model(sd, fi["x"], fi["t"], [fi["c"]], c_types=("image",), model_channels=64), gold["eps_image"],
               what="apply_model 24x16, 33-token image ctx")
        assert (O.vae_decode(sd, fi["z"]) - gold["vae_decode"]).abs().max().item() <= 1e-4
        # img2img start (ddim.py:97-103) with q_sample's noise given explicitly
        xi = O.ddim_sample(sd, None, [fi["cc"]], [fi["uu"]], 8, 7.5, c_types=("image",), model_channels=64, x0=fi["x0"],
                           x0_forward_timesteps=5, x0_noise=fi["x0_noise"])
        _close(xi, gold["i2i_final"], rtol=5e-4, what="img2img 5-of-8-step latent")
        # dual-context sampler (BASELINE config 4's entry point, ddim.py:173-298): text 0.7 + image 0.3
        xm = O.ddim_sample(sd, fi["xT"], [fi["ct"], fi["ci"]], [fi["ut"], fi["ui"]], 4, 7.5, c_types=("text", "image"),
                           ratios=[0.7, 0.3], model_channels=64)
        _close(xm, gold["dual_final"], rtol=5e-4, what="4-step dual-context latent")
    # text-latent flows (SURVEY 8f rank 4): the 0-D diffuser with its data blocks, apply_model + the 4-step CFG DDIM walk on [n, 768]
    shapes_t = {k: tuple(v) for k, v in json.load(open(os.path.join(GOLD, "keys_mini_text.json"))).items()}
    sd_t = weights.synth_state_dict(shapes_t, seed=REF_CASES_SEEDS["text"])
    with torch.no_grad():
        _close(O.apply_model_text(sd_t, fi["xt"], torch.tensor([5, 900]), [fi["ci2"]], c_types=("image",), model_channels=64),
               gold["text_eps"], what="text-latent apply_model")
        _close(O.ddim_sample_text(sd_t, fi["xt"], [fi["ci2"]], [fi["ui2"]], 4, 7.5, c_types=("image",), model_channels=64),
               gold["text_final"], rtol=5e-4, what="4-step text-latent DDIM")


def test_oracle_text_latent_diffuser_vs_reference_golden():
    """SURVEY §8f rank 4: the 0-D diffuser restatement (Linear_MultiDim / FCBlock_MultiDim walk) against goldens produced by the
    unmodified reference's apply_model on a [B, 768] text latent (tests/golden/mini_text.npz)."""
    import json
    import numpy as np
    from oracle import vd_oracle as O, weights
    from oracle.make_golden import golden_inputs, WEIGHT_SEED
    gold_dir = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    shapes = {k: tuple(v) for k, v in json.load(open(os.path.join(gold_dir, "keys_mini_text.json"))).items()}
    sd = weights.synth_state_dict(shapes, seed=WEIGHT_SEED)
    gold = dict(np.load(os.path.join(gold_dir, "mini_text.npz")))
    gt = golden_inputs("text")
    with torch.no_grad():
        t2t = O.apply_model_text(sd, gt["x"], gt["t"], [gt["c_text"]], c_types=("text",), model_channels=64)
        i2t = O.apply_model_text(sd, gt["x"], gt["t"], [gt["c_img"]], c_types=("image",), model_channels=64)
    for out, key in ((t2t, "eps_t2t"), (i2t, "eps_i2t")):
        ref = torch.as_tensor(gold[key])
        assert (out - ref).abs().max().item() <= 2e-4 * ref.abs().max().item(), key
