"""``MH`` -- isotropic random-walk Metropolis for a batch of chains (reference ``mh.py:7-37``).

Same constructor as the reference (``MH(model, stepsize, seed=None, theta=None)``) plus ``chains``,
``dtype``, ``device``, ``chain_offset``.  Each ``draw()`` proposes ``theta + stepsize * N(0, I)`` and
accepts with the Metropolis ratio; everything runs in ``klhr_mh_run`` (csrc/klhr_mh.cuh).
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from .bsmodel import _dtype_code
from .engine import _ptr
from .mcmc import MCMCBase


class MH(MCMCBase):
    def __init__(self, model, stepsize, seed=None, theta=None, *, chains=1, dtype=torch.float64, device=None,
                 chain_offset=0):
        super().__init__(model, stepsize, theta=theta, seed=seed, chains=chains, dtype=dtype, device=device)
        if not stepsize > 0:
            raise ValueError("stepsize must be positive")
        self._draw = 0
        self._chain_offset = int(chain_offset)
        self._accept_count = torch.zeros(self.chains, dtype=torch.int64, device=self.device)

    def _advance(self, n, draws=None, thin=1, chain_s1=None, chain_s2=None, trace=None, shift=None, thin_offset=0):
        lib = _lib.load()
        md = self.model.descriptor(self.dtype, self.device)
        ad = _lib.AccumDesc(accept_count=_ptr(self._accept_count), draws=_ptr(draws), thin=int(thin),
                            chain_s1=_ptr(chain_s1), chain_s2=_ptr(chain_s2), shift=_ptr(shift),
                            thin_offset=int(thin_offset))
        trd = trace.descriptor() if trace is not None else None
        with torch.cuda.device(self.device):
            st = torch.cuda.current_stream(self.device).cuda_stream
            _lib.check(lib.klhr_mh_run(C.byref(md), _dtype_code(self.dtype), self._theta.data_ptr(),
                                       float(self.stepsize), self.chains, self._chain_offset, self._draw, int(n),
                                       C.c_uint64(self.seed & (2 ** 64 - 1)), C.byref(ad),
                                       C.byref(trd) if trd else None, st), "klhr_mh_run")
        self._draw += int(n)

    def draw(self):
        self._advance(1)
        return self.theta

    def sample(self, M, thin=1):
        out = torch.empty(M, self.chains, self.D, dtype=self.dtype, device=self.device)
        out[0] = self._theta
        if M > 1:
            self._advance((M - 1) * thin, draws=out[1:], thin=thin)
        return out[:, 0].double().cpu().numpy() if self.chains == 1 else out

    def run(self, n, chain_stats=False):
        if not chain_stats:
            self._advance(n)
            return None
        s1 = torch.zeros(self.chains, self.D, dtype=torch.float64, device=self.device)
        s2 = torch.zeros_like(s1)
        self._advance(n, chain_s1=s1, chain_s2=s2)
        return s1, s2

    @property
    def acceptance_probability(self):
        return float(self._accept_count.double().mean()) / self._draw if self._draw else 0.0
