"""-m gpu: gmm2d_lean_kernel reads Philox's launch-uniform round-2 words from a table in its kernel parameters, so one launch
runs at most as many rounds as the table holds and the host splits longer runs into several lean launches.  A run that needs
two of them must still equal the replay of the library's own draws bit for bit."""
import numpy as np
import pytest
import torch

import psgla_b200 as P

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name,alg", [("symetric_gaussians", "psgla"), ("cross", "pnp_ula")])
def test_lean_kernel_split_at_table_capacity(name, alg):
    """333 chains from global id 3 * 2^32 + 5, 9000 steps from global step 5 * 2^32 + 1 (no 2^32 boundary crossed): one lead
    step, 1124 lean rounds of 8 steps and 7 tail steps.  The table holds 677 rounds, so the rounds take two lean launches
    (677 + 447): 1 + 2 + 1 = 4 launches."""
    lib = P._lib.lib()
    C, n, id0, off = 333, 9000, (3 << 32) + 5, (5 << 32) + 1
    z = torch.empty(n, C, 2, device="cuda")
    P._lib.check(lib.psgla_gmm2d_noise(z.data_ptr(), C, id0, n, off, 77, None), "noise")
    D = P.Theorical_MMSE(*P.gaussian_mixt_example(name))
    prm = dict(delta=0.3, alpha=2 / 3, epsilon=1.0) if alg == "psgla" else dict(delta=0.1, alpha=1.5, epsilon=0.5)
    kw = dict(y=np.array([0.0, -2.0]), A=np.eye(2), sigma=1, denoiser=D, n_chains=C, **prm)
    want, _ = P.run_chains(alg, n, noise=z, **kw)
    got, _ = P.run_chains(alg, n, seed=77, chain_id0=id0, philox_offset=off, **kw)
    assert torch.equal(got, want) and lib.psgla_gmm2d_last_launches() == 4
