"""CPU: the travelling oracle (oracle/egnn_oracle.py) against the golden vectors that the UNMODIFIED
reference produced (tests/golden/make_golden.py)."""
import os

import numpy as np
import pytest
import torch

from helpers import GOLDEN, golden_cases, load_golden, assert_close
from oracle import egnn_oracle

# The oracle runs the reference's ATen ops in the reference's order, so on the CPU that wrote a fixture the fp32 outputs
# agree to the last bit.  Another CPU or thread count splits the sums inside matmuls and reductions differently, which
# moves outputs by a few fp32 ulps of the O(1) intermediates (up to 5e-7 measured).  In fp64 that effect is ~1e-15.
ATOL32, RTOL32 = 1e-6, 1e-6
ATOL64 = 1e-12
FP64_CASES = sorted(os.path.splitext(f)[0] for f in os.listdir(os.path.join(GOLDEN, 'fp64')))


@pytest.mark.parametrize('case', golden_cases())
def test_oracle_matches_golden(case):
    cfg, sd, inp, want, edges = load_golden(case)
    got_a, got_r, got_edges = egnn_oracle.denoiser_forward(cfg, sd, *inp, return_edges=True)
    assert torch.equal(got_edges, edges), 'edge list differs from the reference get_edges'
    assert_close(got_a, want[0], 'ligand output', atol=ATOL32, rtol=RTOL32)
    assert_close(got_r, want[1], 'pocket output', atol=ATOL32, rtol=RTOL32)


@pytest.mark.parametrize('case', FP64_CASES)
def test_oracle_matches_golden_fp64(case):
    """The oracle in fp64 against the reference module in fp64 on the same inputs (tests/golden/fp64/): a bound that
    holds on any CPU and is five orders of magnitude tighter than the fp32 one."""
    cfg, sd, inp, _, _ = load_golden(case)
    z = np.load(os.path.join(GOLDEN, 'fp64', case + '.npz'))
    got_a, got_r = egnn_oracle.denoiser_forward(cfg, sd, *inp, dtype=torch.float64)
    assert_close(got_a, torch.from_numpy(z['out_atoms']), 'ligand output (fp64)', atol=ATOL64, rtol=0)
    assert_close(got_r, torch.from_numpy(z['out_residues']), 'pocket output (fp64)', atol=ATOL64, rtol=0)


@pytest.mark.parametrize('case', ['config1_n64_l4', 'joint_b2_h128_l5'])
def test_oracle_fp64_noise_floor(case):
    """fp32 oracle vs fp64 oracle: documents the reference's own rounding noise (SURVEY.md §4)."""
    cfg, sd, inp, want, _ = load_golden(case)
    o64 = egnn_oracle.denoiser_forward(cfg, sd, *inp, dtype=torch.float64)
    assert_close(want[0], o64[0], 'ligand fp32 vs fp64', atol=2e-6, rtol=1e-5)
    assert_close(want[1], o64[1], 'pocket fp32 vs fp64', atol=2e-6, rtol=1e-5)


@pytest.mark.parametrize('case', ['ragged_b3_l4', 'moad_emb8_h192_l3', 'reflect_sub2_nocut_l2'])
def test_oracle_matches_live_reference(case):
    """The same configurations on a second input draw, against what the reference module computed for it
    (tests/golden/second_draw/, written by tests/golden/make_golden.py)."""
    cfg, sd, inp, want, edges = load_golden(os.path.join('second_draw', case))
    oa, orr, oe = egnn_oracle.denoiser_forward(cfg, sd, *inp, return_edges=True)
    assert torch.equal(oe, edges), 'edge list differs from the reference get_edges'
    assert_close(oa, want[0], 'ligand', atol=ATOL32, rtol=RTOL32)
    assert_close(orr, want[1], 'pocket', atol=ATOL32, rtol=RTOL32)


def test_oracle_nan_convention():
    cfg, sd, inp, _, _ = load_golden('config1_n64_l4')
    bad = inp[0].clone()
    bad[0, 0] = float('nan')
    with pytest.raises(ValueError, match='NaN detected in EGNN output'):
        egnn_oracle.denoiser_forward(cfg, sd, bad, *inp[1:])
