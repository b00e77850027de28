"""CPU: the HiFi-GAN (NSF) oracle -- groundwork for the next scope row (SURVEY.md section 8f rank 2); no kernel yet -- against
the fixtures produced by the unmodified reference (oracle/gen_golden_hifigan.py)."""
import numpy as np
import pytest
import torch

from conftest import golden
from oracle import hifigan_oracle as H

pytestmark = pytest.mark.usefixtures("fixture_threads")


def _case():
    g = golden("hifigan_nsf.npz")
    sd = {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd.")}
    h = dict(H.HPARAMS_TTS, upsample_initial_channel=int(g["upsample_initial_channel"]))
    return g, sd, h, torch.from_numpy(g["mel"]), torch.from_numpy(g["f0"])


def test_generator_matches_reference_fixture():
    g, sd, h, mel, f0 = _case()
    with torch.no_grad():
        torch.manual_seed(int(g["rng_seed"]))
        wav = H.generator(sd, h, mel, f0)
        plain = H.generator(sd, h, mel)
    assert wav.shape == (mel.shape[0], 1, mel.shape[2] * int(np.prod(h["upsample_rates"])))
    assert np.array_equal(wav.numpy(), g["wav_nsf"])          # bit-exact: same ATen kernels, same RNG stream
    assert np.array_equal(plain.numpy(), g["wav_plain"])
    assert np.abs(g["wav_nsf"] - g["wav_plain"]).max() > 1e-4   # the harmonic source does reach the output


def test_weight_norm_and_plain_weights_agree():
    """after remove_weight_norm() a checkpoint carries plain `.weight` tensors: both forms give the same output"""
    g, sd, h, mel, f0 = _case()
    plain_sd = dict(sd)
    for k in list(sd):
        if k.endswith(".weight_g"):
            name = k[:-len(".weight_g")]
            plain_sd[name + ".weight"] = H.conv_weight(sd, name)
            del plain_sd[name + ".weight_g"], plain_sd[name + ".weight_v"]
    with torch.no_grad():
        a, b = H.generator(sd, h, mel), H.generator(plain_sd, h, mel)
    assert torch.equal(a, b)


def test_flops_per_frame_of_the_shipped_config():
    assert H.flops_per_frame(H.HPARAMS_TTS) == 38510592.0


def test_oracle_is_bit_exact_against_the_live_reference():
    """an odd-length utterance (T = 9) under another NSF random stream, recorded from the reference with the same weights"""
    _, sd, h, _, _ = _case()
    s = golden("hifigan_nsf_B1T9.npz")
    with torch.no_grad():
        torch.manual_seed(int(s["rng_seed"]))
        b = H.generator(sd, h, torch.from_numpy(s["mel"]), torch.from_numpy(s["f0"]))
    assert np.array_equal(b.numpy(), s["wav_nsf"])
