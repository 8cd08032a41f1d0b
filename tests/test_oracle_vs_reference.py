"""Oracle <-> unmodified reference at shapes the other goldens do not cover (odd lengths, one source,
four sources, depth 1).  The reference's forward on these seeded inputs is stored in
``golden/oracle_vs_reference.npz`` (``golden/make_golden_reference.py``), so the comparison runs
without the reference checkout."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import sudormrf_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "oracle_vs_reference.npz")

CASES = [
    ("improved", dict(out_channels=64, in_channels=128, num_blocks=4, upsampling_depth=5,
                      enc_kernel_size=21, enc_num_basis=128, num_sources=2), 3333),
    ("improved", dict(out_channels=32, in_channels=32, num_blocks=1, upsampling_depth=1,
                      enc_kernel_size=21, enc_num_basis=16, num_sources=1), 7),
    ("groupcomm", dict(out_channels=64, in_channels=128, num_blocks=2, upsampling_depth=4,
                       enc_kernel_size=21, enc_num_basis=64, num_sources=2,
                       group_size=16), 2000),
    ("causal", dict(in_audio_channels=1, out_channels=32, in_channels=64, num_blocks=3, upsampling_depth=4,
                    enc_kernel_size=21, enc_num_basis=64, num_sources=2), 2000),
    ("original", dict(out_channels=64, in_channels=128, num_blocks=3, upsampling_depth=4,
                      enc_kernel_size=21, enc_num_basis=128, num_sources=2), 3333),
    ("original", dict(out_channels=32, in_channels=64, num_blocks=2, upsampling_depth=5,
                      enc_kernel_size=21, enc_num_basis=32, num_sources=4), 1600),      # no reshape layer, T a multiple of the lcm
]


def case_inputs(variant, kw, T):
    """-> (config, seeded state_dict, seeded input) of one case."""
    cfg = O.Config(variant=variant, **kw)
    sd = O.make_state_dict(cfg, seed=11)
    x = torch.randn(2, 1, T, generator=torch.Generator().manual_seed(5))
    return cfg, sd, x


def fingerprint(sd, x):
    """fp64 sums of the input and of |weights|: tells a change of the seeded inputs from a change of the oracle."""
    return np.array([float(x.double().sum()), float(sum(v.double().abs().sum() for v in sd.values()))])


@pytest.mark.parametrize("variant,kw,T", CASES)
def test_live(variant, kw, T):
    ci = CASES.index((variant, kw, T))
    z = np.load(GOLDEN)
    assert json.loads(bytes(z[f"c{ci}/meta"]).decode()) == dict(variant=variant, kwargs=kw, T=T)
    cfg, sd, x = case_inputs(variant, kw, T)
    assert list(sd.keys()) == json.loads(bytes(z[f"c{ci}/keys"]).decode())     # the reference's state_dict order
    np.testing.assert_allclose(fingerprint(sd, x), z[f"c{ci}/fingerprint"], rtol=1e-12)
    ref = torch.from_numpy(z[f"c{ci}/out"])
    assert max(O.parity_errors(O.forward(cfg, sd, x), ref)) < 2e-5
