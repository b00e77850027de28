"""TEST INFRASTRUCTURE ONLY -- pins oracle/hifigan_oracle.py to the LIVE reference (container only: needs /root/reference)
and writes tests/golden/hifigan_nsf.npz and hifigan_nsf_B1T9.npz.  Run:  python oracle/gen_golden_hifigan.py

The reference module is imported unmodified (stubs only for librosa / pycwt and scipy.signal.kaiser, which newer SciPy moved
to scipy.signal.windows); weights are the constructor's random initialisation under a fixed seed, inputs are seeded; the NSF
source's random draws come from torch's global generator, seeded identically for both sides."""
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import FIXTURE_THREADS, hifigan_oracle as H  # noqa: E402

REF_ROOT = os.environ.get("DSX_REFERENCE_ROOT", "/root/reference")


def load_reference():
    sys.dont_write_bytecode = True
    for n in ("librosa", "librosa.filters", "pycwt"):
        sys.modules.setdefault(n, types.ModuleType(n))
    import scipy.signal
    import scipy.signal.windows
    if not hasattr(scipy.signal, "kaiser"):
        scipy.signal.kaiser = scipy.signal.windows.kaiser
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    from modules.hifigan.hifigan import HifiGanGenerator
    return HifiGanGenerator


def make_case(seed=0, B=2, T=16):
    HifiGanGenerator = load_reference()
    torch.set_num_threads(FIXTURE_THREADS)
    h = dict(H.HPARAMS_TTS, upsample_initial_channel=32)     # the shipped topology at 1/4 of the width: a 250 KB fixture
    torch.manual_seed(seed)
    g = HifiGanGenerator(h).eval()
    sd = {k: v.detach().clone() for k, v in g.state_dict().items()}
    gen = torch.Generator().manual_seed(seed + 1)
    mel = torch.randn(B, 80, T, generator=gen)
    f0 = torch.rand(B, T, generator=gen) * 300 + 100
    f0[0, 4:7] = 0                                   # an unvoiced stretch
    return g, h, sd, mel, f0


def write_odd_length_case():
    """One utterance of odd length (T = 9) through the weights of the main fixture (weight seed 0), the NSF source's random
    draws under seed 11: tests/golden/hifigan_nsf_B1T9.npz (inputs and output only; the weights are in hifigan_nsf.npz)."""
    g, h, sd, _, _ = make_case(seed=0)
    _, _, _, mel, f0 = make_case(seed=3, B=1, T=9)
    with torch.no_grad():
        torch.manual_seed(11)
        ref = g(mel, f0)
        torch.manual_seed(11)
        ora = H.generator(sd, h, mel, f0)
    assert torch.equal(ref, ora), "the oracle must be bit-exact against the reference"
    out = os.path.join(ROOT, "tests", "golden", "hifigan_nsf_B1T9.npz")
    np.savez_compressed(out, mel=mel.numpy(), f0=f0.numpy(), wav_nsf=ref.numpy(), rng_seed=np.int64(11))
    print("wrote", out)


def main():
    write_odd_length_case()
    g, h, sd, mel, f0 = make_case()
    with torch.no_grad():
        torch.manual_seed(7)
        ref_nsf = g(mel, f0)
        torch.manual_seed(7)
        ora_nsf = H.generator(sd, h, mel, f0)
        ref_plain = g(mel)
        ora_plain = H.generator(sd, h, mel)
    d1, d2 = (ref_nsf - ora_nsf).abs().max().item(), (ref_plain - ora_plain).abs().max().item()
    print(f"oracle vs live reference: NSF path max |d| = {d1:.3e}, mel-only path max |d| = {d2:.3e}")
    assert d1 == 0.0 and d2 == 0.0, "the oracle must be bit-exact against the reference"
    out = os.path.join(ROOT, "tests", "golden", "hifigan_nsf.npz")
    np.savez_compressed(out, mel=mel.numpy(), f0=f0.numpy(), wav_nsf=ref_nsf.numpy(), wav_plain=ref_plain.numpy(),
                        rng_seed=np.int64(7), weight_seed=np.int64(0), upsample_initial_channel=np.int64(h["upsample_initial_channel"]),
                        **{"sd." + k: v.numpy() for k, v in sd.items()})
    print("wrote", out, os.path.getsize(out) // 1024, "KB; FLOPs per mel frame:", H.flops_per_frame(h))


if __name__ == "__main__":
    main()
