"""Launch structure of the diffusion step on every precision path: the kernel launches (DSX_INFO_KERNEL_LAUNCHES) of a DDPM
loop, a PNDM loop (warm-up and every Adams-Bashforth order), dsx_infer with either sampler and one DiffNet evaluation, and
one DSX_OPT_PROFILE bracket per evaluation."""
import pytest
import torch

from conftest import rs_normal
from oracle import diffnet_oracle as O
from test_gpu_parity import dsx, make_sampler  # noqa: F401  (dsx: fixture)

pytestmark = pytest.mark.gpu

L = 20                       # residual layers (conftest.HP)
B, T = 2, 150                # 4 tiles: one launch group of either residual-stack kernel
K = 5                        # DDPM steps
K_PLMS, INTERVAL = 300, 40   # PNDM steps t = 280, 240, ..., 0: warm-up (2 evaluations), then orders 2, 3, 4, 4, 4, 4, 4
N_PLMS = 8


def costs(prec, fused):
    """Launches (that start a call's first evaluation, per evaluation of a sampling loop, per DiffNet evaluation)."""
    if prec == "fp32":
        # input projection, 4 per residual layer (conv GEMM, gate, GEMM, residual), head (4), sampler update
        return 0, 4 * L + 4 + 1 + 1, 1 + 4 * L + 4
    per = 1 if fused and prec != "fp16x3" else 2       # k_tc_stack with the head inside, or residual stack + k_tc_head
    return 1, per, 1 + per                             # k_tc_head with the input projection only starts a call


@pytest.mark.parametrize("prec,fused", [("fp32", 1), ("fp16x3", 1), ("fp16x2", 0), ("fp16x2", 1), ("fp16s", 1)])
def test_step_launches(dsx, prec, fused):
    from diffsinger_b200 import _capi
    s, dev = make_sampler(dsx, 1, prec, O.make_schedule(O.linear_beta_schedule(1000, 0.02)))
    s.set_option(_capi.OPT_FUSED_HEAD, fused)
    start, per, fwd = costs(prec, fused)
    setup = 2 + (1 if prec == "fp32" else 2)            # step-embedding table (2), conditioner pack (+ its projection)
    cond, x = rs_normal(1, (B, 256, T)).to(dev), rs_normal(2, (B, 1, 80, T)).to(dev)
    fs2 = rs_normal(3, (B, T, 80)).to(dev) - 2.0
    smin, smax = torch.full((80,), -5.0, device=dev), torch.full((80,), 0.5, device=dev)
    t = torch.tensor([5, 60], device=dev)
    # (call, evaluations, launches besides setup and the evaluations); cond.clone(): the conditioner is packed every call
    calls = {
        "sample_ddpm": (lambda: s.sample_ddpm(x, cond.clone(), 1000, K, seed=1), K, 0),
        "sample_plms": (lambda: s.sample_plms(x, cond.clone(), K_PLMS, INTERVAL), N_PLMS + 1, 0),
        "infer_ddpm": (lambda: s.infer(cond, K, smin, smax, fs2_mel=fs2, seed=1), K, 2),            # + prologue, epilogue
        "infer_plms": (lambda: s.infer(cond, K_PLMS, smin, smax, fs2_mel=fs2, seed=1, pndm_interval=INTERVAL), N_PLMS + 1, 2),
        "diffnet_forward": (lambda: s.diffnet_forward(x, t, cond.clone()), 1, None),
    }
    for name, (call, evals, extra) in calls.items():
        l0 = s.info(_capi.INFO_KERNEL_LAUNCHES)
        call()
        n = s.info(_capi.INFO_KERNEL_LAUNCHES) - l0
        assert n == setup + (fwd if extra is None else start + evals * per + extra), (name, n)
        s.set_option(_capi.OPT_PROFILE, 1)              # one (start, stop) bracket per evaluation
        call()
        assert s.info(_capi.INFO_LAYER_KERNEL_LAUNCHES) == evals, name
        assert s.info(_capi.INFO_LAYER_KERNEL_NS) > 0, name
        s.set_option(_capi.OPT_PROFILE, 0)
    s.close()
