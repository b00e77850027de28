"""TEST INFRASTRUCTURE ONLY -- records what tests/test_reference_live.py compares the drop-in against, from the LIVE
reference (container only: needs the reference tree, see oracle/ref_bridge.py), into tests/golden/reference_dropin.npz.
Run:  python -m oracle.gen_golden_dropin

Recorded, for the reference's GaussianDiffusion built the way usr/diffspeech_task.py builds it (config lj_ds_beta6, torch seed
0): every state-dict key with its shape and the SHA-256 of its float32 bytes (the values themselves are tens of MB: the
conditioner), the hparams the model reads, one DiffNet evaluation and one p_losses value on seeded inputs.  The digests of
the conditioner's `_float_tensor` buffers are of uninitialised memory and change from run to run; the test does not use them."""
import hashlib
import os

import numpy as np
import torch

from . import FIXTURE_THREADS, ref_bridge
from .diffnet_oracle import diffnet_forward

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "reference_dropin.npz")
HP_KEYS = ("timesteps", "K_step", "diff_loss_type", "spec_min", "spec_max", "keep_bins", "schedule_type", "max_beta",
           "hidden_size", "residual_layers", "residual_channels", "dilation_cycle_length", "audio_num_mel_bins")


def tensor_sha256(v):
    return hashlib.sha256(np.ascontiguousarray(v.detach().cpu().numpy()).tobytes()).hexdigest()


def inputs():
    """Seeded inputs and the output-projection weights (the constructor zero-initialises them)."""
    g = torch.Generator().manual_seed(2024)
    x = torch.randn(2, 1, 80, 24, generator=g)
    cond = torch.randn(2, 256, 24, generator=g)
    noise = torch.randn(2, 1, 80, 24, generator=g)
    out_w = torch.randn(80, 256, 1, generator=g) * 0.02
    return x, torch.tensor([3, 50]), cond, noise, out_w


def main():
    assert ref_bridge.available(), "needs the reference tree"
    torch.set_num_threads(FIXTURE_THREADS)
    ns = ref_bridge.load("usr/configs/lj_ds_beta6.yaml")
    hp = ns.hparams
    enc = ns.TokenTextEncoder(None, vocab_list=["a", "b", "c"], replace_oov=",")
    torch.manual_seed(0)
    model = ns.GaussianDiffusion(enc, 80, ns.DiffNet(80), timesteps=hp["timesteps"], K_step=hp["K_step"],
                                 loss_type=hp["diff_loss_type"], spec_min=hp["spec_min"], spec_max=hp["spec_max"])
    sd = model.state_dict()
    shapes = [",".join(map(str, v.shape)) for v in sd.values()]
    hashes = [tensor_sha256(v) for v in sd.values()]          # before the output projection is overwritten below
    x, t, cond, noise, out_w = inputs()
    net = model.denoise_fn
    with torch.no_grad():
        net.output_projection.weight.copy_(out_w)
        eps = net.eval()(x, t, cond)
        assert torch.equal(eps, diffnet_forward({k: v for k, v in net.state_dict().items()}, x, t, cond,
                                                hp["dilation_cycle_length"]))
        loss = model.train().p_losses(x, t, cond, noise=noise)
    np.savez_compressed(
        OUT, sd_keys=np.array(list(sd)), sd_shapes=np.array(shapes), sd_sha256=np.array(hashes),
        x=x.numpy(), t=t.numpy(), cond=cond.numpy(), noise=noise.numpy(), out_w=out_w.numpy(), eps=eps.numpy(),
        p_loss=loss.detach().numpy(),
        **{"hp." + k: np.array(hp[k]) for k in HP_KEYS})
    print("wrote", OUT, os.path.getsize(OUT) // 1024, "KB;", len(sd), "state-dict entries, loss", float(loss))


if __name__ == "__main__":
    main()
