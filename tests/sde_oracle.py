"""The numpy executor with the SDE step -- TEST INFRASTRUCTURE.

`SdeOracleBackend` is `oracle_backend.OracleBackend` plus `sde_step`, the numpy restatement of dpm_sde_step
(include/dpm_solver_b200.h): the LIN1 / DIFF2 step exactly as `OracleBackend.step` computes it, followed by one more
separately rounded term, out = ((a*x + c0*NEW) + c1*D) + noise_scale*z, each product and sum rounded in IEEE fp32.
"""
import numpy as np
import torch

from dpm_solver_b200._lib import FORM_DIFF2, FORM_LIN1
from oracle_backend import OracleBackend, _np, _round

f32 = np.float32


class SdeOracleBackend(OracleBackend):
    name = "numpy-oracle-sde"

    def sde_step(self, a, noise_scale, generator=None, noise=None):
        """z is `noise`, or torch.randn_like(x, dtype=torch.float32) drawn from `generator` (None: torch's default
        generator of x's device); returns (m_out, out) like CudaBackend.sde_step."""
        if a.form not in (FORM_LIN1, FORM_DIFF2):
            raise ValueError("the SDE step serves the LIN1 and DIFF2 forms only")
        self.launches += 1
        self.log.append((a.form, a.n_model))
        ref = a.reference_tensor()
        if noise is None:
            noise = torch.randn_like(ref, dtype=torch.float32, generator=generator)
        sdt = a.state_dtype
        if sdt is None:
            st = a.state_tensors()
            sdt = st[0].dtype if st else a.e_cond.dtype
        if a.n_model > 0:
            T0 = _round(self._model_value(a, _np(a.thr) if a.thr is not None else None), sdt)
        else:
            T0 = _np(a.m0)
        m_out = None
        if a.n_model > 0 and a.want_m_out:
            m_out = torch.from_numpy(np.ascontiguousarray(T0)).to(sdt).reshape(ref.shape)
        x = _np(a.x)
        A, c0, c1, w0 = f32(a.a), f32(a.c0), f32(a.c1), f32(a.w0)
        if a.form == FORM_LIN1:
            o = A * x + c0 * T0
        else:
            m1 = _np(a.m1)
            D = w0 * (T0 - m1)
            o = (A * x + c0 * (m1 if a.c0_on_old else T0)) + c1 * D
        z = _np(noise).reshape(o.shape)
        o = o.astype(f32) + f32(noise_scale) * z
        out = torch.from_numpy(np.ascontiguousarray(o.astype(f32))).to(sdt).reshape(ref.shape)
        if a.out is not None:
            a.out.copy_(out.reshape(a.out.shape))
            out = a.out
        if a.out2 is not None:
            a.out2.copy_(out.reshape(a.out2.shape))
        return m_out, out
