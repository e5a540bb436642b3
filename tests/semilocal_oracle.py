"""Torch restatement of the semilocal kinetic functionals LuoKarasievTrickey and PauliGaussian in the style of
oracle/ofdft_oracle.py (fp64, the oracle's Grid, potentials and stresses by autograd)  --  TEST HELPER ONLY.

The reduced gradient / Laplacian follow functional_tools.py:230-287; the constants are those of the papers (LKT: a = 1.3,
PRB 98, 041111 (2018); PGSL0.25: mu = 40/27, beta = 0.25, JPCL 9, 4385 (2018)).  No golden vectors of the reference pin
these two functionals.  Nothing in the product imports this file."""
import math

import torch

from oracle.ofdft_oracle import C_TF, Grid

PI = math.pi


def _reduced_p_q(g, den):
    gx, gy, gz = g.grad(den)
    c = 0.25 * (3.0 * PI * PI) ** (-2.0 / 3.0)
    p = c * (gx * gx + gy * gy + gz * gz) / den.pow(8.0 / 3.0)
    q = c * g.laplacian(den) / den.pow(5.0 / 3.0)
    return p, q


def LuoKarasievTrickey(box, den, a=1.3):
    """functionals.py:309 : T = int C_TF n^(5/3) (1 / cosh(a s) + (5/3) s^2)"""
    g = Grid(box, den.shape)
    p, _ = _reduced_p_q(g, den)
    s = torch.sqrt(p + 1e-300)        # keeps autograd finite where grad n = 0 (a uniform start); the value is unchanged
    return g.integral(C_TF * den.pow(5.0 / 3.0) * (1.0 / torch.cosh(a * s) + (5.0 / 3.0) * p))


def PauliGaussian(box, den, mu=40.0 / 27.0, beta=0.25):
    """functionals.py:336 : T = int C_TF n^(5/3) ((5/3) p + exp(-mu p) + beta q^2)"""
    g = Grid(box, den.shape)
    p, q = _reduced_p_q(g, den)
    return g.integral(C_TF * den.pow(5.0 / 3.0) * ((5.0 / 3.0) * p + torch.exp(-mu * p) + beta * q * q))
