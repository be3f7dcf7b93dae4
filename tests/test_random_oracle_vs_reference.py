"""The oracle itself against the UNMODIFIED reference (its results stored in tests/golden/reference/) on random
sampling configurations: torch-CPU namespace bit-identical, numpy namespace within its transcendental-ulp
tolerance. Complements the fixed golden vectors that pin the oracle (tests/test_oracle_golden.py)."""
import random

import numpy as np
import pytest
import torch

import helpers
import refstore as S
from oracle import dpm_oracle as O
from test_random_configs_vs_reference import draw, run_reference

REF = S.Store(__file__)


@pytest.mark.parametrize("chunk", range(3))
def test_oracle_matches_reference_on_random_configurations(chunk):
    rng = random.Random(70000 + chunk)
    done = i = 0
    while done < 20:
        c = draw(rng)
        i += 1
        case = dict(schedule=c["schedule"], algo=c["algo"], method=c["method"], order=c["order"], steps=c["steps"],
                    skip_type=c["skip_type"], solver_type=c["solver_type"], model_type=c["model_type"], cfg=c["cfg"],
                    lower_order_final=c["lower_order_final"], denoise_to_zero=c["denoise_to_zero"], t_end=c["t_end"],
                    seed=c["seed"], thresholding=c["thresholding"], shape=(2, 3, 8, 8), net="exact")
        try:
            yr = REF(f"oracle/{chunk}/{i}", lambda: run_reference(c)[0])
        except Exception:
            continue
        if not S.all_finite(yr):
            continue
        yt, _, _ = helpers.run_oracle_case(case, None, O.torch_namespace("cpu"))
        yt = yt if torch.is_tensor(yt) else torch.from_numpy(np.asarray(yt))
        S.assert_same(yt, yr, case)
        # yt is bit-identical to the reference: it stands for the reference's values below
        yn, _, _ = helpers.run_oracle_case(case, None, O.NP)
        yn = yn.numpy() if torch.is_tensor(yn) else np.asarray(yn)
        assert helpers.rel_err(yn, yt.numpy()) <= 1e-3, case
        done += 1
