"""-m gpu: the 2D throughput kernel (gmm2d_lean_kernel) takes the high words of the chain id and of the Philox counter pair as
launch constants and computes Philox's first two rounds from them once per thread or per launch; the host splits its launches
where either high word changes.  A run whose chain ids and counter pairs both cross a multiple of 2^32 must still equal the
replay of the library's own draws bit for bit."""
import numpy as np
import pytest
import torch

import psgla_b200 as P

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name,alg", [("symetric_gaussians", "psgla"), ("cross", "pnp_ula")])
def test_lean_kernel_across_high_word_boundaries(name, alg):
    """Chains 2^32 - 700 .. 2^32 + 799 and global steps 2^33 - 13 .. 2^33 + 31 (counter pairs 2^32 - 7 .. 2^32 + 15): one lead
    step, 5 lean rounds of 8 steps and 4 tail steps; per chain-id half, one lean round before pair 2^32, the round that
    straddles it on the general kernel and 3 lean rounds after: 1 + 2 x 3 + 1 = 8 launches."""
    lib = P._lib.lib()
    C, n, id0, off = 1500, 45, (1 << 32) - 700, (1 << 33) - 13
    z = torch.empty(n, C, 2, device="cuda")
    P._lib.check(lib.psgla_gmm2d_noise(z.data_ptr(), C, id0, n, off, 77, None), "noise")
    D = P.Theorical_MMSE(*P.gaussian_mixt_example(name))
    prm = dict(delta=0.3, alpha=2 / 3, epsilon=1.0) if alg == "psgla" else dict(delta=0.1, alpha=1.5, epsilon=0.5)
    kw = dict(y=np.array([0.0, -2.0]), A=np.eye(2), sigma=1, denoiser=D, n_chains=C, **prm)
    want, _ = P.run_chains(alg, n, noise=z, **kw)
    got, _ = P.run_chains(alg, n, seed=77, chain_id0=id0, philox_offset=off, **kw)
    assert torch.equal(got, want) and lib.psgla_gmm2d_last_launches() == 8
