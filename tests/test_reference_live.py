"""The drop-in against what the reference computed (tests/golden/reference_dropin.npz, recorded from the unmodified
reference by oracle/gen_golden_dropin.py): `dropin.install()` patches a stand-in of the reference's modules
(tests/standin_ref.py) without editing them, the model the task files build has the reference's state-dict keys, shapes and
values (so reference checkpoints load with strict=True), the training branch is the reference's, inference has no CPU
fallback, and the oracle agrees with the reference for one network evaluation."""
import os
import subprocess
import sys

from conftest import ROOT

SCRIPT = r'''
import hashlib, sys, numpy as np, torch
sys.path.insert(0, %(root)r); sys.path.insert(0, %(root)r + "/tests"); sys.path.insert(0, %(tree)r)
from conftest import golden
from oracle import FIXTURE_THREADS, diffnet_oracle as O
torch.set_num_threads(FIXTURE_THREADS)
g = golden("reference_dropin.npz")
hp = {k[3:]: g[k].item() if g[k].ndim == 0 else list(g[k]) for k in g.files if k.startswith("hp.")}
from utils.hparams import hparams
hparams.update(hp)
import usr.diff.shallow_diffusion_tts as sdt, usr.diff.net as net_mod
ref_cls = sdt.GaussianDiffusion
import diffsinger_b200.dropin as dropin
new_cls = dropin.install()
assert sdt.GaussianDiffusion is new_cls and issubclass(new_cls, ref_cls)
assert net_mod.DiffNet.__module__.startswith("diffsinger_b200")
# the task files build the model exactly like this (usr/diffspeech_task.py:25-32)
torch.manual_seed(0)
model = sdt.GaussianDiffusion(phone_encoder=None, out_dims=80, denoise_fn=net_mod.DiffNet(hp["audio_num_mel_bins"]),
                              timesteps=hp["timesteps"], K_step=hp["K_step"], loss_type=hp["diff_loss_type"],
                              spec_min=hp["spec_min"], spec_max=hp["spec_max"])
# every tensor the drop-in contributes (denoise_fn, schedule buffers) has the reference's key, shape and value under the same
# seed; the keys left over are the conditioner's (fs2), which the reference class builds itself
ref = {k: (s, h) for k, s, h in zip(g["sd_keys"], g["sd_shapes"], g["sd_sha256"])}
sd = model.state_dict()
assert set(sd) <= set(ref) and all(k.startswith("fs2.") for k in set(ref) - set(sd)), set(sd) ^ set(ref)
for k, v in sd.items():
    assert ",".join(map(str, v.shape)) == ref[k][0], k
    assert hashlib.sha256(np.ascontiguousarray(v.numpy()).tobytes()).hexdigest() == ref[k][1], k
model.load_state_dict(sd, strict=True)
# training branch unchanged: p_losses is the reference class's own, running through the module graph
assert "p_losses" not in vars(new_cls) and "forward" in vars(new_cls)
# the inference branch has no CPU fallback
class Stub(torch.nn.Module):
    def forward(self, *a, **k):
        return {"decoder_inp": torch.randn(2, 24, 256), "mel_out": torch.randn(2, 24, 80)}
model.fs2 = Stub()
try:
    with torch.no_grad():
        model(torch.zeros(2, 5, dtype=torch.long), infer=True)
    raise SystemExit("expected DsxError on CPU")
except Exception as e:
    assert type(e).__name__ == "DsxError", repr(e)
dropin.uninstall()
assert sdt.GaussianDiffusion is ref_cls and net_mod.DiffNet is not model.denoise_fn.__class__
# oracle == reference for one network evaluation; the package's training branch gives the reference's p_losses value
x, t, cond, noise = (torch.from_numpy(g[k]) for k in ("x", "t", "cond", "noise"))
net = model.denoise_fn
with torch.no_grad():
    net.output_projection.weight.copy_(torch.from_numpy(g["out_w"]))
    b = O.diffnet_forward({k: v for k, v in net.state_dict().items()}, x, t, cond, hp["dilation_cycle_length"])
assert torch.equal(b, torch.from_numpy(g["eps"]))
import diffsinger_b200 as dsx
gd = dsx.GaussianDiffusion(None, 80, net.train(), timesteps=hp["timesteps"], K_step=hp["K_step"], loss_type=hp["diff_loss_type"],
                           spec_min=hp["spec_min"], spec_max=hp["spec_max"], fs2=torch.nn.Identity(), hparams=hp)
loss = gd.p_losses(x, t, cond, noise=noise)
assert loss.requires_grad and abs(loss.item() - float(g["p_loss"])) < 1e-6, (loss.item(), float(g["p_loss"]))
print("LIVE-OK")
'''


def test_dropin_against_live_reference(lib_built, tmp_path):
    from standin_ref import write_tree
    tree = write_tree(str(tmp_path / "standin"))
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    r = subprocess.run([sys.executable, "-c", SCRIPT % {"root": ROOT, "tree": tree}], capture_output=True, text=True, env=env,
                       cwd=ROOT, timeout=600)
    assert "LIVE-OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
