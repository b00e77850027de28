"""The CPU oracle against the committed golden vectors (outputs of the live reference, produced by
oracle/gen_golden.py).  Runs without a GPU."""
import numpy as np
import pytest
import torch

from conftest import golden, rs_normal
from oracle import diffnet_oracle as O

pytestmark = pytest.mark.usefixtures("fixture_threads")


def test_schedules_match_reference_buffers():
    g = golden("schedules.npz")
    for name, betas in (("linear006_T100", O.linear_beta_schedule(100, 0.06)),
                        ("linear002_T1000", O.linear_beta_schedule(1000, 0.02)),
                        ("cosine_T100", O.cosine_beta_schedule(100))):
        S = O.make_schedule(betas)
        for b in O.SCHEDULE_BUFFERS:
            assert np.array_equal(S[b].numpy(), g[f"{name}.{b}"]), (name, b)
    # appendix B anchors (SURVEY.md): coef1[0] = 1, coef2[0] = 0, clipped log-variance at 0 = ln(1e-20)
    S = O.make_schedule(O.linear_beta_schedule(100, 0.06))
    assert S["posterior_mean_coef1"][0] == 1 and S["posterior_mean_coef2"][0] == 0
    assert abs(float(S["posterior_log_variance_clipped"][0]) - np.log(1e-20)) < 1e-4
    assert abs(float(S["alphas_cumprod"][-1]) - 4.654703e-02) < 1e-7


@pytest.mark.parametrize("cycle", [1, 4])
def test_diffnet_forward_and_taps(cycle):
    g = golden(f"diffnet_fwd_cycle{cycle}.npz")
    sd = O.build_state_dict(0, dilation_cycle_length=cycle)
    taps = {}
    with torch.no_grad():
        eps = O.diffnet_forward(sd, torch.from_numpy(g["spec"]), torch.from_numpy(g["t"]), torch.from_numpy(g["cond"]),
                                cycle, taps=taps)
        emb = O.step_embedding(sd, torch.from_numpy(g["t"]))
    assert np.array_equal(eps.numpy(), g["eps"])
    assert np.array_equal(taps["x1"][0].numpy(), g["x1_b0"])
    assert np.array_equal(taps["x20"][1].numpy(), g["x20_b1"])
    assert np.array_equal(taps["skip_sum"][0].numpy(), g["skip_sum_b0"])
    assert np.array_equal(emb.numpy(), g["step_emb"])


def test_ddpm_single_steps_and_loop():
    g = golden("ddpm_lj_K100.npz")
    sd = O.build_state_dict(0)
    S = O.make_schedule(O.linear_beta_schedule(100, 0.06))
    cond, xT = torch.from_numpy(g["cond"]), torch.from_numpy(g["xT"])
    noise = rs_normal(int(g["noise_seed"]), (100,) + tuple(xT.shape))
    assert abs(float(noise.double().sum()) - float(g["noise_checksum"])) < 1e-6
    assert np.array_equal(noise[3, 1, 0, 5, :8].numpy(), g["noise_probe"])
    with torch.no_grad():
        for t in (99, 50, 1, 0):
            out = O.p_sample(sd, S, xT, t, cond, noise[7])
            assert np.array_equal(out.numpy(), g[f"single_t{t}"]), t
        # t == 0: output is exactly clamp(x0_hat) (coef1 = 1, coef2 = 0, no noise)
        assert float(out.abs().max()) <= 1.0
        x0 = O.sample_ddpm(sd, S, xT, cond, 100, noise)
    assert np.abs(x0.numpy() - g["x0"]).max() <= 2e-5


def test_plms_loop_and_warmup_step():
    g = golden("plms_T1000_cycle4.npz")
    sd = O.build_state_dict(0, dilation_cycle_length=4)
    S = O.make_schedule(O.linear_beta_schedule(1000, 0.02))
    cond, xT = torch.from_numpy(g["cond"]), torch.from_numpy(g["xT"])
    with torch.no_grad():
        hist = []
        first = O.p_sample_plms(sd, S, xT[:1], 960, 40, cond[:1], hist, 4)
        assert np.array_equal(first.numpy(), g["first_step_b0"]) and len(hist) == 1
        x0 = torch.cat([O.sample_plms(sd, S, xT[b:b + 1], cond[b:b + 1], 1000, 40, 4) for b in range(2)], 0)
    assert np.array_equal(x0.numpy(), g["x0_interval40"])


def test_infer_forward_shallow_start_with_mask():
    g = golden("infer_forward_K51.npz")
    sd = O.build_state_dict(0)
    S = O.make_schedule(O.linear_beta_schedule(100, 0.06))
    K = 51
    B, T = g["mel2ph"].shape
    noise = rs_normal(int(g["noise_seed"]), (K, B, 1, 80, T))
    with torch.no_grad():
        mel = O.infer_loop(sd, S, torch.from_numpy(g["decoder_inp"]).transpose(1, 2), K, torch.from_numpy(g["spec_min"]),
                           torch.from_numpy(g["spec_max"]), fs2_mel=torch.from_numpy(g["fs2_mel"]),
                           start_noise=torch.from_numpy(g["start_noise"]), step_noise=noise,
                           mel2ph=torch.from_numpy(g["mel2ph"]))
    assert np.abs(mel.numpy() - g["mel_out"]).max() <= 1e-4
    assert np.all(mel.numpy()[1, 60:] == 0)           # masked frames (mel2ph == 0)


def test_ddpm_full_T1000_loop():
    """BASELINE config 3 class: T = K = 1000, beta <= 0.02, dilation cycle 4."""
    g = golden("ddpm_T1000_cycle4.npz")
    sd = O.build_state_dict(0, dilation_cycle_length=4)
    S = O.make_schedule(O.linear_beta_schedule(1000, 0.02))
    cond, xT = torch.from_numpy(g["cond"]), torch.from_numpy(g["xT"])
    noise = rs_normal(int(g["noise_seed"]), (1000,) + tuple(xT.shape))
    assert abs(float(noise.double().sum()) - float(g["noise_checksum"])) < 1e-6
    x = xT
    with torch.no_grad():
        for j, t in enumerate(reversed(range(1000))):
            x = O.p_sample(sd, S, x, t, cond, noise[j], 4)
            if t in (900, 500):
                assert np.abs(x.numpy() - g[f"x_after_t{t}"]).max() <= 5e-5, t
    assert np.abs(x.numpy() - g["x0"]).max() <= 5e-5


def test_plms_bounded_state_fixture():
    g = golden("plms_K300_cycle4.npz")
    sd = O.build_state_dict(0, dilation_cycle_length=4)
    S = O.make_schedule(O.linear_beta_schedule(1000, 0.02))
    cond, xT = torch.from_numpy(g["cond"]), torch.from_numpy(g["xT"])
    for interval in (40, 10):
        with torch.no_grad():
            x0 = torch.cat([O.sample_plms(sd, S, xT[b:b + 1], cond[b:b + 1], 300, interval, 4) for b in range(2)], 0)
        assert np.array_equal(x0.numpy(), g[f"x0_interval{interval}"])
        assert np.abs(g[f"x0_interval{interval}"]).max() < 10       # bounded: an absolute tolerance is meaningful


def test_old_sampler_cosine_schedule():
    """usr/diff/diffusion.py:313-320: gaussian start, full-T DDPM on the cosine schedule, denorm, no mask."""
    g = golden("old_sampler_cosine_K100.npz")
    sd = O.build_state_dict(0)
    S = O.make_schedule(O.cosine_beta_schedule(100))
    B, T, _ = g["decoder_inp"].shape
    noise = rs_normal(int(g["noise_seed"]), (100, B, 1, 80, T))
    with torch.no_grad():
        mel = O.infer_loop(sd, S, torch.from_numpy(g["decoder_inp"]).transpose(1, 2), 100, torch.from_numpy(g["spec_min"]),
                           torch.from_numpy(g["spec_max"]), x_start=torch.from_numpy(g["x_start"]), step_noise=noise)
    assert np.abs(mel.numpy() - g["mel_out"]).max() <= 1e-4


def test_offline_forward():
    """OfflineGaussianDiffusion.forward(infer=True), usr/diff/shallow_diffusion_tts.py:291-323."""
    g = golden("offline_forward_K51.npz")
    sd = O.build_state_dict(0)
    S = O.make_schedule(O.linear_beta_schedule(100, 0.06))
    B, T, _ = g["decoder_inp"].shape
    noise = rs_normal(int(g["noise_seed"]), (51, B, 1, 80, T))
    with torch.no_grad():
        mel = O.infer_loop(sd, S, torch.from_numpy(g["decoder_inp"]).transpose(1, 2), 51, torch.from_numpy(g["spec_min"]),
                           torch.from_numpy(g["spec_max"]), fs2_mel=torch.from_numpy(g["fs2_mel"]),
                           start_noise=torch.from_numpy(g["start_noise"]), step_noise=noise)
    assert np.abs(mel.numpy() - g["mel_out"]).max() <= 1e-4
