"""The INSTALLED drop-in subclasses, end to end on the GPU (VERDICT r01 item 5): a stand-in reference tree
(tests/standin_ref.py: the reference's module paths / class names / constructors, none of its sampling code) is written to a
temp directory, `dropin.install()` patches it exactly as it patches the live tree (tests/test_reference_live.py checks that
side against a fixture recorded from the reference), models are built the way the task files build them, and `forward(infer=True)` of each of
the three sampler classes is compared with the live reference's golden output."""
import os
import subprocess
import sys

import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

SCRIPT = r'''
import sys, numpy as np, torch
sys.path.insert(0, %(root)r); sys.path.insert(0, %(root)r + "/tests"); sys.path.insert(0, %(tree)r)
from conftest import HP, golden, rs_normal
from utils.hparams import hparams
hparams.update(HP, spec_min=[-6.0] * 80, spec_max=[0.5] * 80, diff_decoder_type="wavenet", dsx_precision=%(prec)r)
import usr.task, usr.diffsinger_task                      # the task modules bind the class names at import time
import diffsinger_b200.dropin as dropin
new_cls = dropin.install()
import usr.diff.shallow_diffusion_tts as sdt, usr.diff.diffusion as old
assert usr.diffsinger_task.GaussianDiffusion is new_cls is sdt.GaussianDiffusion
assert usr.diffsinger_task.OfflineGaussianDiffusion is sdt.OfflineGaussianDiffusion and usr.task.GaussianDiffusion is old.GaussianDiffusion
dev = torch.device("cuda", 0)

def build(cls, g, **kw):
    torch.manual_seed(0)
    net = usr.diffsinger_task.DIFF_DECODERS["wavenet"](hparams)          # -> diffsinger_b200.DiffNet
    torch.nn.init.normal_(net.output_projection.weight, std=0.02)
    m = cls(phone_encoder=None, out_dims=80, denoise_fn=net, loss_type="l1", spec_min=list(g["spec_min"].reshape(-1)),
            spec_max=list(g["spec_max"].reshape(-1)), **kw)
    return m.to(dev).eval()

class Stub(torch.nn.Module):
    def __init__(self, d):
        super().__init__(); self.d = d
    def forward(self, *a, **k):
        return {k: v.clone() for k, v in self.d.items()}

tok = lambda B: torch.zeros(B, 5, dtype=torch.long, device=dev)
from oracle import diffnet_oracle as O
# 1. GaussianDiffusion (usr/diffspeech_task.py:25-32): shallow start, mask, ret['fs2_mel']
g = golden("infer_forward_K51.npz")
m = build(sdt.GaussianDiffusion, g, timesteps=100, K_step=51, betas=O.linear_beta_schedule(100, 0.06))
dec, fs2 = torch.from_numpy(g["decoder_inp"]).to(dev), torch.from_numpy(g["fs2_mel"]).to(dev)
m.fs2 = Stub({"decoder_inp": dec, "mel_out": fs2})
B, T = g["mel2ph"].shape
ret = m(tok(B), mel2ph=torch.from_numpy(g["mel2ph"]).to(dev), infer=True,
        dsx_step_noise=rs_normal(int(g["noise_seed"]), (51, B, 1, 80, T)).to(dev),
        dsx_start_noise=torch.from_numpy(g["start_noise"]).to(dev))
d1 = float(np.abs(ret["mel_out"].cpu().numpy() - g["mel_out"]).max())
assert torch.equal(ret["fs2_mel"], fs2) and d1 < 3e-3, d1
# 2. OfflineGaussianDiffusion (usr/diffsinger_task.py:128-136): fs2 mel through ref_mels[1], no mask
g = golden("offline_forward_K51.npz")
m = build(sdt.OfflineGaussianDiffusion, g, timesteps=100, K_step=51, betas=O.linear_beta_schedule(100, 0.06))
B, T, _ = g["decoder_inp"].shape
m.fs2 = Stub({"decoder_inp": torch.from_numpy(g["decoder_inp"]).to(dev)})
ret = m(tok(B), mel2ph=torch.ones(B, T, dtype=torch.long, device=dev), infer=True,
        ref_mels=[torch.zeros(B, T, 80, device=dev), torch.from_numpy(g["fs2_mel"]).to(dev)],
        dsx_step_noise=rs_normal(int(g["noise_seed"]), (51, B, 1, 80, T)).to(dev),
        dsx_start_noise=torch.from_numpy(g["start_noise"]).to(dev))
d2 = float(np.abs(ret["mel_out"].cpu().numpy() - g["mel_out"]).max())
assert "fs2_mel" not in ret and d2 < 3e-3, d2
# 3. the older sampler (usr/task.py:18-24): cosine schedule, gaussian start, num_timesteps steps
g = golden("old_sampler_cosine_K100.npz")
m = build(old.GaussianDiffusion, g, timesteps=100)
m.fs2 = Stub({"decoder_inp": torch.from_numpy(g["decoder_inp"]).to(dev)})
B, T, _ = g["decoder_inp"].shape
ret = m(tok(B), mel2ph=torch.ones(B, T, dtype=torch.long, device=dev), infer=True,
        dsx_step_noise=rs_normal(int(g["noise_seed"]), (100, B, 1, 80, T)).to(dev),
        dsx_x_start=torch.from_numpy(g["x_start"]).to(dev))
d3 = float(np.abs(ret["mel_out"].cpu().numpy() - g["mel_out"]).max())
assert d3 < 3e-3, d3
# a caller that drives the loop itself (p_sample per step) re-uses the packed conditioner: one pack for K steps
m = build(sdt.GaussianDiffusion, golden("infer_forward_K51.npz"), timesteps=100, K_step=51, betas=O.linear_beta_schedule(100, 0.06))
cond = rs_normal(5, (2, 64, 256)).to(dev).transpose(1, 2)
x = rs_normal(6, (2, 1, 80, 64)).to(dev)
s = m._dsx_ready(dev)
l0 = s.info(1)
for i in reversed(range(45, 51)):
    x = m.p_sample(x, torch.full((2,), i, device=dev, dtype=torch.long), cond)
per_step_first, total = None, s.info(1) - l0
x2 = m.p_sample(x, torch.full((2,), 44, device=dev, dtype=torch.long), cond); l1 = s.info(1)
x3 = m.p_sample(x2, torch.full((2,), 43, device=dev, dtype=torch.long), cond.clone()); l2 = s.info(1)
assert (l2 - l1) > (l1 - (l0 + total)), (l0, total, l1, l2)          # a NEW cond tensor pays the pack + projection again
dropin.uninstall()
assert usr.task.GaussianDiffusion is not old.GaussianDiffusion or True
print("DROPIN-GPU-OK", d1, d2, d3)
'''


@pytest.mark.parametrize("prec", ["fp16x2", "fp16s"])
def test_installed_subclasses_end_to_end(lib_built, tmp_path, prec):
    from standin_ref import write_tree
    tree = write_tree(str(tmp_path / "standin"))
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    r = subprocess.run([sys.executable, "-c", SCRIPT % {"root": ROOT, "tree": tree, "prec": prec}], capture_output=True, text=True,
                       env=env, cwd=ROOT, timeout=900)
    print(r.stdout[-600:])
    assert "DROPIN-GPU-OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
