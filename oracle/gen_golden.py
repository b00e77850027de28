"""TEST INFRASTRUCTURE ONLY -- pins the oracle against the LIVE reference and writes tests/golden.

Run in the build container (needs /root/reference):

    cd /root/repo && python -m oracle.gen_golden

Every vector written here is an output of the unmodified reference modules
(usr/diff/net.py DiffNet, usr/diff/shallow_diffusion_tts.py GaussianDiffusion) on seeded
inputs; alongside, the oracle restatement is asserted to agree with the reference
(bit-exact for one network evaluation / one sampler step, <=2e-5 after a full K-step loop).
Inputs that are too large to commit (per-step noise, weights) are regenerated from
numpy RandomState / torch seeds and fingerprinted in the fixture.
"""
import os
import sys
from collections import deque

import numpy as np
import torch

from . import FIXTURE_THREADS
from . import diffnet_oracle as O
from . import ref_bridge

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def rs_normal(seed, shape):
    """Stable-forever noise stream (legacy numpy RandomState), fp32."""
    return torch.from_numpy(np.random.RandomState(seed).standard_normal(size=shape).astype(np.float32))


def fingerprint(sd):
    """Order-dependent fp64 checksum of a state dict (guards seed-regenerated weights)."""
    acc = 0.0
    for i, (k, v) in enumerate(sd.items()):
        acc += float(v.double().sum()) * (1 + (i % 7)) + float(v.double().abs().sum())
    return acc


def make_ref_net(ns, seed, cycle, out_std=0.02):
    ns.hparams["dilation_cycle_length"] = cycle
    torch.manual_seed(seed)
    net = ns.DiffNet(80).eval()
    if out_std is not None:
        torch.nn.init.normal_(net.output_projection.weight, std=out_std)
    return net


def make_ref_gd(ns, net, betas, K_step):
    enc = ns.TokenTextEncoder(None, vocab_list=["a", "b", "c"], replace_oov=",")
    hp = ns.hparams
    gd = ns.GaussianDiffusion(enc, 80, net, timesteps=len(betas), K_step=K_step, loss_type="l1",
                              betas=torch.tensor(betas), spec_min=hp["spec_min"], spec_max=hp["spec_max"]).eval()
    return gd


def main():
    assert ref_bridge.available(), "needs /root/reference"
    torch.set_num_threads(FIXTURE_THREADS)
    ns = ref_bridge.load("usr/configs/lj_ds_beta6.yaml")
    sdt = ns.sdt
    os.makedirs(OUT, exist_ok=True)
    report = {}

    # ---- 1. schedules --------------------------------------------------------------
    sched = {}
    for name, betas in (("linear006_T100", O.linear_beta_schedule(100, 0.06)),
                        ("linear002_T1000", O.linear_beta_schedule(1000, 0.02)),
                        ("cosine_T100", O.cosine_beta_schedule(100))):
        net = make_ref_net(ns, 0, 1)
        gd = make_ref_gd(ns, net, betas, len(betas))
        S = O.make_schedule(betas)
        for b in O.SCHEDULE_BUFFERS:
            assert torch.equal(getattr(gd, b), S[b]), (name, b)
            sched[f"{name}.{b}"] = getattr(gd, b).numpy()
    # the reference's own schedule functions
    assert np.array_equal(sdt.cosine_beta_schedule(100), O.cosine_beta_schedule(100))
    assert np.array_equal(sdt.linear_beta_schedule(100, 0.06), O.linear_beta_schedule(100, 0.06))
    np.savez(os.path.join(OUT, "schedules.npz"), **sched)

    # ---- 2. one DiffNet evaluation, both dilation cycles, with layer taps -----------
    for cycle in (1, 4):
        net = make_ref_net(ns, 0, cycle)
        sd = O.build_state_dict(0, dilation_cycle_length=cycle)
        rsd = net.state_dict()
        assert all(torch.equal(sd[k], rsd[k]) for k in rsd)
        B, T = 2, 150
        spec = rs_normal(11, (B, 1, 80, T))
        cond = rs_normal(12, (B, 256, T))
        t = torch.tensor([37, 5], dtype=torch.long)
        # reference taps via forward hooks on the residual layers
        ref_taps = {}
        hooks = []
        for i, layer in enumerate(net.residual_layers):
            hooks.append(layer.register_forward_hook(
                lambda m, inp, out, i=i: ref_taps.__setitem__(i, (inp[0].clone(), out[0].clone(), out[1].clone()))))
        with torch.no_grad():
            eps = net(spec, t, cond)
        for h in hooks:
            h.remove()
        taps = {}
        with torch.no_grad():
            eps_o = O.diffnet_forward(sd, spec, t, cond, cycle, taps=taps)
        assert torch.equal(eps, eps_o)
        for i in (0, 1, 7, 19):
            assert torch.equal(ref_taps[i][0], taps[f"x{i}"])
        assert torch.equal(ref_taps[19][0 + 1], taps["x20"])
        e_ref = net.mlp(net.diffusion_embedding(t))
        assert torch.equal(e_ref, O.step_embedding(sd, t))
        np.savez(os.path.join(OUT, f"diffnet_fwd_cycle{cycle}.npz"),
                 spec=spec.numpy(), cond=cond.numpy(), t=t.numpy(), eps=eps.numpy(),
                 x1_b0=ref_taps[0][1][0].numpy(), x20_b1=ref_taps[19][1][1].numpy(),
                 skip_sum_b0=taps["skip_sum"][0].numpy(), step_emb=e_ref.detach().numpy(),
                 weights_fingerprint=np.float64(fingerprint(rsd)))
        report[f"fwd_cycle{cycle}"] = float(eps.abs().max())

    # ---- 3. DDPM: single steps and the full K=100 loop (LJ schedule) ----------------
    betas = O.linear_beta_schedule(100, 0.06)
    S = O.make_schedule(betas)
    net = make_ref_net(ns, 0, 1)
    sd = O.build_state_dict(0)
    gd = make_ref_gd(ns, net, betas, 100)
    B, T, K = 2, 96, 100
    cond = rs_normal(21, (B, 256, T))
    xT = rs_normal(22, (B, 1, 80, T))
    noise = rs_normal(23, (K, B, 1, 80, T))
    feed = {"i": 0}
    orig_noise_like = sdt.noise_like

    def fake_noise_like(shape, device, repeat=False):
        n = noise[feed["i"]]
        feed["i"] += 1
        assert tuple(shape) == tuple(n.shape)
        return n

    sdt.noise_like = fake_noise_like
    try:
        singles = {}
        for t in (99, 50, 1, 0):
            feed["i"] = 7
            with torch.no_grad():
                r = gd.p_sample(xT, torch.full((B,), t, dtype=torch.long), cond)
                o = O.p_sample(sd, S, xT, t, cond, noise[7])
            assert torch.equal(r, o), t
            singles[f"t{t}"] = r.numpy()
        feed["i"] = 0
        x = xT
        with torch.no_grad():
            for i in reversed(range(K)):
                x = gd.p_sample(x, torch.full((B,), i, dtype=torch.long), cond)
            xo = O.sample_ddpm(sd, S, xT, cond, K, noise)
        d = (x - xo).abs().max().item()
        assert d <= 2e-5, d
        report["ddpm_loop_oracle_vs_ref"] = d
        np.savez(os.path.join(OUT, "ddpm_lj_K100.npz"), cond=cond.numpy(), xT=xT.numpy(), x0=x.numpy(),
                 noise_seed=23, noise_checksum=np.float64(noise.double().sum().item()),
                 noise_probe=noise[3, 1, 0, 5, :8].numpy(),
                 **{f"single_{k}": v for k, v in singles.items()},
                 weights_fingerprint=np.float64(fingerprint(net.state_dict())))
    finally:
        sdt.noise_like = orig_noise_like

    # ---- 4. PLMS (PNDM), T=K=1000, interval 40, dilation cycle 4 (OpenCpop ds1000) ---
    betas = O.linear_beta_schedule(1000, 0.02)
    S = O.make_schedule(betas)
    net = make_ref_net(ns, 0, 4)
    sd = O.build_state_dict(0, dilation_cycle_length=4)
    gd = make_ref_gd(ns, net, betas, 1000)
    B, T, K = 2, 96, 1000
    cond = rs_normal(31, (B, 256, T))
    xT = rs_normal(32, (B, 1, 80, T))
    outs = {}
    for interval in (40, 100):
        ref_rows = []
        for b in range(B):       # the reference's PLMS only runs at B=1 (max() on a tensor, :192)
            gd.noise_list = deque(maxlen=4)
            x = xT[b:b + 1]
            with torch.no_grad():
                for i in reversed(range(0, K, interval)):
                    x = gd.p_sample_plms(x, torch.full((1,), i, dtype=torch.long), interval, cond[b:b + 1])
            ref_rows.append(x)
        ref = torch.cat(ref_rows, 0)
        with torch.no_grad():
            xo1 = torch.cat([O.sample_plms(sd, S, xT[b:b + 1], cond[b:b + 1], K, interval, 4) for b in range(B)], 0)
            xo = O.sample_plms(sd, S, xT, cond, K, interval, 4)
        assert torch.equal(ref, xo1)                      # per-utterance: bit-exact
        # batched (B=2) evaluation only changes the CPU conv summation order; with random weights the
        # un-clamped PLMS state grows to |x| ~ 4e2, so the check is relative
        d = ((ref - xo).abs().max() / ref.abs().max()).item()
        assert d <= 2e-6, d
        report[f"plms{interval}_oracle_vs_ref_rel"] = d
        report[f"plms{interval}_absmax"] = ref.abs().max().item()
        outs[f"x0_interval{interval}"] = ref.numpy()
    # one warm-up step (two net evals) on its own
    gd.noise_list = deque(maxlen=4)
    with torch.no_grad():
        r = gd.p_sample_plms(xT[:1], torch.full((1,), 960, dtype=torch.long), 40, cond[:1])
        hist = []
        o = O.p_sample_plms(sd, S, xT[:1], 960, 40, cond[:1], hist, 4)
    assert torch.equal(r, o)
    outs["first_step_b0"] = r.numpy()
    np.savez(os.path.join(OUT, "plms_T1000_cycle4.npz"), cond=cond.numpy(), xT=xT.numpy(), **outs,
             weights_fingerprint=np.float64(fingerprint(net.state_dict())))

    # ---- 5. GaussianDiffusion.forward(infer=True) around a stubbed fs2 ---------------
    #      (prologue norm_spec + q_sample, loop, epilogue denorm + mel2ph mask)
    betas = O.linear_beta_schedule(100, 0.06)
    S = O.make_schedule(betas)
    net = make_ref_net(ns, 0, 1)
    sd = O.build_state_dict(0)
    K_step = 51
    gd = make_ref_gd(ns, net, betas, K_step)
    B, T = 2, 80
    dec_inp = rs_normal(41, (B, T, 256))
    fs2_mel = rs_normal(42, (B, T, 80)) * 1.5 - 2.5
    mel2ph = torch.ones(B, T, dtype=torch.long)
    mel2ph[1, 60:] = 0
    dec_inp[1, 60:] = 0
    start_noise = rs_normal(43, (B, 1, 80, T))
    noise = rs_normal(44, (K_step, B, 1, 80, T))

    class StubFS2(torch.nn.Module):
        def forward(self, *a, **kw):
            return {"decoder_inp": dec_inp.clone(), "mel_out": fs2_mel.clone()}

    gd.fs2 = StubFS2()
    feed["i"] = 0
    noise_ref = noise

    def fake_noise_like2(shape, device, repeat=False):
        n = noise_ref[feed["i"]]
        feed["i"] += 1
        return n

    orig_randn_like = torch.randn_like
    sdt.noise_like = fake_noise_like2
    sdt.torch.randn_like = lambda x: start_noise          # q_sample's default noise (:207)
    try:
        with torch.no_grad():
            ret = gd(torch.zeros(B, 5, dtype=torch.long), mel2ph=mel2ph, infer=True)
    finally:
        sdt.noise_like = orig_noise_like
        sdt.torch.randn_like = orig_randn_like
    smin, smax = gd.spec_min, gd.spec_max
    with torch.no_grad():
        mo = O.infer_loop(sd, S, dec_inp.transpose(1, 2), K_step, smin, smax, fs2_mel=fs2_mel,
                          start_noise=start_noise, step_noise=noise, mel2ph=mel2ph)
    d = (ret["mel_out"] - mo).abs().max().item()
    assert d <= 1e-4, d
    report["infer_forward_oracle_vs_ref"] = d
    np.savez(os.path.join(OUT, "infer_forward_K51.npz"), decoder_inp=dec_inp.numpy(), fs2_mel=fs2_mel.numpy(),
             mel2ph=mel2ph.numpy(), start_noise=start_noise.numpy(), mel_out=ret["mel_out"].numpy(),
             spec_min=smin.numpy(), spec_max=smax.numpy(), noise_seed=44,
             noise_checksum=np.float64(noise.double().sum().item()))

    # ---- 6. BASELINE config 3 class: full T = K = 1000 DDPM (beta <= 0.02), dilation cycle 4, injected noise ---
    betas = O.linear_beta_schedule(1000, 0.02)
    S = O.make_schedule(betas)
    net = make_ref_net(ns, 0, 4)
    sd = O.build_state_dict(0, dilation_cycle_length=4)
    gd = make_ref_gd(ns, net, betas, 1000)
    B, T, K = 1, 96, 1000
    cond = rs_normal(51, (B, 256, T))
    xT = rs_normal(52, (B, 1, 80, T))
    noise = rs_normal(53, (K, B, 1, 80, T))
    feed["i"] = 0

    def fake_noise_like3(shape, device, repeat=False):
        n = noise[feed["i"]]
        feed["i"] += 1
        return n

    sdt.noise_like = fake_noise_like3
    try:
        x = xT
        mids = {}
        with torch.no_grad():
            for i in reversed(range(K)):
                x = gd.p_sample(x, torch.full((B,), i, dtype=torch.long), cond)
                if i in (900, 500):
                    mids[f"x_after_t{i}"] = x.numpy().copy()
            xo = O.sample_ddpm(sd, S, xT, cond, K, noise, 4)
        d = (x - xo).abs().max().item()
        assert d <= 5e-5, d
        report["ddpm1000_oracle_vs_ref"] = d
        np.savez(os.path.join(OUT, "ddpm_T1000_cycle4.npz"), cond=cond.numpy(), xT=xT.numpy(), x0=x.numpy(), noise_seed=53,
                 noise_checksum=np.float64(noise.double().sum().item()), **mids,
                 weights_fingerprint=np.float64(fingerprint(net.state_dict())))
    finally:
        sdt.noise_like = orig_noise_like

    # ---- 7. PLMS with a bounded state: shallow start K_step = 300 of the T = 1000 schedule (alpha_cumprod[299] ~ 0.4, so the
    #         un-clamped state stays O(1) and an ABSOLUTE per-bin bound applies), intervals 40 and 10, B = 2 ---------------
    gd = make_ref_gd(ns, net, betas, 300)
    B, T, K = 2, 96, 300
    cond = rs_normal(61, (B, 256, T))
    xT = rs_normal(62, (B, 1, 80, T))
    outs = {}
    for interval in (40, 10):
        ref_rows = []
        for b in range(B):
            gd.noise_list = deque(maxlen=4)
            x = xT[b:b + 1]
            with torch.no_grad():
                for i in reversed(range(0, K, interval)):
                    x = gd.p_sample_plms(x, torch.full((1,), i, dtype=torch.long), interval, cond[b:b + 1])
            ref_rows.append(x)
        ref = torch.cat(ref_rows, 0)
        with torch.no_grad():
            xo1 = torch.cat([O.sample_plms(sd, S, xT[b:b + 1], cond[b:b + 1], K, interval, 4) for b in range(B)], 0)
        assert torch.equal(ref, xo1)
        report[f"plms_bounded{interval}_absmax"] = ref.abs().max().item()
        outs[f"x0_interval{interval}"] = ref.numpy()
    np.savez(os.path.join(OUT, "plms_K300_cycle4.npz"), cond=cond.numpy(), xT=xT.numpy(), **outs,
             weights_fingerprint=np.float64(fingerprint(net.state_dict())))

    # ---- 8. the older sampler usr/diff/diffusion.py (usr/task.py:18): cosine schedule, gaussian start, full-T DDPM, no mask ---
    import importlib
    cwd = os.getcwd()
    os.chdir(ref_bridge.REF_ROOT)
    try:
        dmod = importlib.import_module("usr.diff.diffusion")
    finally:
        os.chdir(cwd)
    net = make_ref_net(ns, 0, 1)
    sd = O.build_state_dict(0)
    enc = ns.TokenTextEncoder(None, vocab_list=["a", "b", "c"], replace_oov=",")
    gd_old = dmod.GaussianDiffusion(enc, 80, net, timesteps=100, loss_type="l1", spec_min=ns.hparams["spec_min"],
                                    spec_max=ns.hparams["spec_max"]).eval()
    Sc = O.make_schedule(O.cosine_beta_schedule(100))
    for bname in O.SCHEDULE_BUFFERS:
        assert torch.equal(getattr(gd_old, bname), Sc[bname]), bname
    B, T, K = 2, 80, 100
    dec_inp = rs_normal(71, (B, T, 256))
    x_start = rs_normal(72, (B, 1, 80, T))
    noise = rs_normal(73, (K, B, 1, 80, T))

    class StubFS2Old(torch.nn.Module):
        def forward(self, *a, **kw):
            return {"decoder_inp": dec_inp.clone()}

    class TorchProxy:           # torch, except randn(shape, device=...) -> the fixture's start noise
        def __getattr__(self, name):
            return getattr(torch, name)

        def randn(self, *a, **kw):
            return x_start.clone()

    gd_old.fs2 = StubFS2Old()
    feed["i"] = 0

    def fake_noise_like4(shape, device, repeat=False):
        n = noise[feed["i"]]
        feed["i"] += 1
        return n

    orig_nl, orig_torch = dmod.noise_like, dmod.torch
    dmod.noise_like, dmod.torch = fake_noise_like4, TorchProxy()
    try:
        with torch.no_grad():
            ret = gd_old(torch.zeros(B, 5, dtype=torch.long), mel2ph=torch.ones(B, T, dtype=torch.long), infer=True)
    finally:
        dmod.noise_like, dmod.torch = orig_nl, orig_torch
    with torch.no_grad():
        mo = O.infer_loop(sd, Sc, dec_inp.transpose(1, 2), K, gd_old.spec_min, gd_old.spec_max, x_start=x_start,
                          step_noise=noise)
    d = (ret["mel_out"] - mo).abs().max().item()
    assert d <= 1e-4, d
    report["old_sampler_cosine_oracle_vs_ref"] = d
    np.savez(os.path.join(OUT, "old_sampler_cosine_K100.npz"), decoder_inp=dec_inp.numpy(), x_start=x_start.numpy(),
             mel_out=ret["mel_out"].numpy(), spec_min=gd_old.spec_min.numpy(), spec_max=gd_old.spec_max.numpy(), noise_seed=73,
             noise_checksum=np.float64(noise.double().sum().item()))

    # ---- 9. OfflineGaussianDiffusion.forward(infer=True) (usr/diffsinger_task.py:128): fs2 mel handed in through ref_mels[1],
    #         shallow start, DDPM, no mel2ph mask ------------------------------------------------------------------------------
    betas = O.linear_beta_schedule(100, 0.06)
    S = O.make_schedule(betas)
    K_step = 51
    gd_off = sdt.OfflineGaussianDiffusion(enc, 80, net, timesteps=100, K_step=K_step, loss_type="l1", betas=torch.tensor(betas),
                                          spec_min=ns.hparams["spec_min"], spec_max=ns.hparams["spec_max"]).eval()
    dec_inp = rs_normal(81, (B, T, 256))
    fs2_mel = rs_normal(82, (B, T, 80)) * 1.5 - 2.5
    start_noise = rs_normal(83, (B, 1, 80, T))
    noise = rs_normal(84, (K_step, B, 1, 80, T))

    class StubFS2Off(torch.nn.Module):
        def forward(self, *a, **kw):
            return {"decoder_inp": dec_inp.clone()}

    gd_off.fs2 = StubFS2Off()
    feed["i"] = 0

    def fake_noise_like5(shape, device, repeat=False):
        n = noise[feed["i"]]
        feed["i"] += 1
        return n

    sdt.noise_like = fake_noise_like5
    sdt.torch.randn_like = lambda x: start_noise
    try:
        with torch.no_grad():
            ret = gd_off(torch.zeros(B, 5, dtype=torch.long), mel2ph=torch.ones(B, T, dtype=torch.long),
                         ref_mels=[torch.zeros(B, T, 80), fs2_mel], infer=True)
    finally:
        sdt.noise_like = orig_noise_like
        sdt.torch.randn_like = orig_randn_like
    with torch.no_grad():
        mo = O.infer_loop(sd, S, dec_inp.transpose(1, 2), K_step, gd_off.spec_min, gd_off.spec_max, fs2_mel=fs2_mel,
                          start_noise=start_noise, step_noise=noise)
    d = (ret["mel_out"] - mo).abs().max().item()
    assert d <= 1e-4, d
    report["offline_forward_oracle_vs_ref"] = d
    np.savez(os.path.join(OUT, "offline_forward_K51.npz"), decoder_inp=dec_inp.numpy(), fs2_mel=fs2_mel.numpy(),
             start_noise=start_noise.numpy(), mel_out=ret["mel_out"].numpy(), spec_min=gd_off.spec_min.numpy(),
             spec_max=gd_off.spec_max.numpy(), noise_seed=84, noise_checksum=np.float64(noise.double().sum().item()))

    for k, v in report.items():
        print(f"{k}: {v:.3e}")
    print("golden vectors written to", OUT)


if __name__ == "__main__":
    main()
