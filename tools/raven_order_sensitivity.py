"""How far two fp32 evaluation orders of the SAME Raven update (raven.py:126-143) drift apart on a 29.5 M-element tensor, CPU only.

Order A = CPU ATen as the oracle runs it (``oracle/host_ref.raven_update_``); order B = CUDA ATen's (FMA contraction, multiply by
1/sqrt_bc2) as ``raven_step_bulk_kernel`` implements it, emulated here through float64 FMAs.  Output: how many elements exceed
1e-6 x (|p| + |update|) -- the cancelled result -- and 1e-6 x (|p| + update TERMS), the scale tests/test_gpu_fullsize.py uses.
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import host_ref  # noqa: E402

HP = dict(lr=1e-3, betas=(0.9, 0.999), weight_decay=0.01, eps=1e-8, debias_strength=0.3)


def fma(a, b, c):
    return (a.double() * b.double() + c.double()).float()


def main():
    n = 1280 * 2560 * 9
    g = torch.Generator().manual_seed(90)
    p = torch.randn(n, generator=g) * 0.02
    rp, rm, rv = p.clone(), torch.zeros(n), torch.zeros(n)
    ep, em, ev = p.clone(), torch.zeros(n), torch.zeros(n)
    f = lambda x: torch.tensor(x, dtype=torch.float32)
    for step in (1, 2):
        grad = torch.randn(n, generator=g) * 1e-2
        before, m_prev = rp.clone(), rm.clone()
        host_ref.raven_update_(rp, grad, rm, rv, step=step, **HP)
        s = host_ref.raven_scalars(HP["lr"], HP["betas"], HP["eps"], HP["weight_decay"], HP["debias_strength"], step)
        em = fma(f(s["one_m_b1"]), grad, em * f(s["beta1"]))
        ev = fma(f(s["one_m_b2"]) * grad, grad, ev * f(s["beta2"]))
        ep = ep * f(s["wd_factor"])
        denom = ev.sqrt() * f(1.0 / s["sqrt_bc2"]) + f(HP["eps"])
        ep = fma(-f(s["step_size"]), em / denom, ep)
    err = (ep - rp).abs()
    naive = 1e-6 * (rp.abs() + (rp - before).abs()) + 1e-12
    d = rv.sqrt() / s["sqrt_bc2"] + HP["eps"]
    terms = before.abs() + s["step_size"] * (s["beta1"] * m_prev.abs() + s["one_m_b1"] * grad.abs()) / d
    scaled = 1e-6 * (rp.abs() + terms) + 1e-12
    print(f"elements {n}; beyond 1e-6 x (|p| + |update|): {int((err > naive).sum())} (worst {float((err / naive).max()):.1f} x); "
          f"beyond 1e-6 x (|p| + update terms): {int((err > scaled).sum())} (worst {float((err / scaled).max()):.3f} x); "
          f"plain isclose(rtol 1e-6, atol 1e-9) misses: {int((~torch.isclose(ep, rp, rtol=1e-6, atol=1e-9)).sum())}")


if __name__ == "__main__":
    main()
