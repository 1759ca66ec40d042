"""GPU parity tests proper: the sm_100a kernels, called through the C ABI (libdiffsbdd_b200.so via
diffsbdd_b200.EGNNDynamics), against (i) the committed golden vectors produced by the unmodified
reference and (ii) the travelling CPU oracle on fresh seeded inputs.  Tolerance: atol 1e-5 / rtol 1e-4
(fp32; helpers.ATOL/RTOL)."""
import pytest
import torch

from helpers import golden_cases, load_golden, assert_close, ATOL, RTOL
from diffsbdd_b200 import synthetic as syn
from diffsbdd_b200.config import FULLATOM_COND, CONFIG1, DynamicsConfig
from diffsbdd_b200.dynamics import EGNNDynamics
from oracle import egnn_oracle

pytestmark = pytest.mark.gpu


def make_net(cfg, sd):
    net = EGNNDynamics.from_config(cfg, device='cuda')
    net.load_state_dict(sd, strict=True)
    net.eval()
    return net


def run(net, inp):
    with torch.no_grad():
        out = net(*[x.cuda() for x in inp])
    torch.cuda.synchronize()
    return out[0].cpu(), out[1].cpu()


@pytest.mark.parametrize('case', golden_cases())
def test_golden_edges_bit_exact(case):
    cfg, sd, inp, want, edges = load_golden(case)
    net = make_net(cfg, sd)
    got = net.get_edges(inp[3].cuda(), inp[4].cuda(), inp[0][:, :3].cuda(), inp[1][:, :3].cuda()).cpu()
    assert got.shape == edges.shape and torch.equal(got, edges)


@pytest.mark.parametrize('mode', ['fp32', '3xtf32', 1, 2, 4, 9, 10, 12])
@pytest.mark.parametrize('case', ['config1_n64_l4', 'ragged_b3_l4', 'fullatom_b2_n200_l6', 'ca_b3_l6'])
def test_golden_forward_every_math_mode(case, mode):
    """hidden_nf=256 cases through each arithmetic path: fp32 FFMA kernels; tcgen05 3xTF32 everywhere; and the node
    GEMMs (1), edge kernel (2), coordinate kernel (4) individually in 3xTF32 and in 3xFP16 (+8).  The default 'auto'
    (= '3xfp16', all kernels) is covered by test_golden_forward."""
    cfg, sd, inp, want, edges = load_golden(case)
    net = make_net(cfg, sd)
    net.math_mode = mode
    got_a, got_r = run(net, inp)
    assert_close(got_a, want[0], f'{case} mode {mode} ligand out')
    assert_close(got_r, want[1], f'{case} mode {mode} pocket out')


H256_VARIANTS = ['joint_ca_h256_l6', 'reflect_h256_l3', 'sub2_h256_l2', 'noatt_notanh_h256_l2', 'emb8_h256_l3',
                 'joint_emb8_sub2_reflect_h256_l2', 'mean_h256_l3']


@pytest.mark.parametrize('mode', ['fp32', '3xtf32', '3xfp16'])
@pytest.mark.parametrize('case', H256_VARIANTS)
def test_golden_h256_variants_every_arithmetic(case, mode):
    """The branches the production config does not take, at hidden_nf=256 so that they run on the tcgen05 kernels too:
    joint mode (all coordinate rows live, velocity mean removal; crossdock_ca_joint.yml dims), reflection-equivariant
    (one coordinate MLP per tile), two sub-layers, no attention / no tanh, the edge-type table of the producers, a
    combination of them, and aggregation_method='mean'.  Goldens come from the unmodified reference (tests/golden/make_golden.py)."""
    cfg, sd, inp, want, edges = load_golden(case)
    net = make_net(cfg, sd)
    net.math_mode = mode
    got_a, got_r = run(net, inp)
    assert net.last_num_edges == edges.shape[1]
    assert_close(got_a, want[0], f'{case} mode {mode} ligand out')
    assert_close(got_r, want[1], f'{case} mode {mode} pocket out')


OTHER_WIDTHS = ['joint_b2_h128_l5', 'moad_emb8_h192_l3', 'reflect_sub2_nocut_l2', 'noatt_notanh_l2', 'mean_joint_h128_l2']


@pytest.mark.parametrize('mode', ['fp32', '3xtf32', '3xfp16'])
@pytest.mark.parametrize('case', OTHER_WIDTHS)
def test_golden_other_widths_every_arithmetic(case, mode):
    """hidden_nf 128 and 192 (crossdock_fullatom_joint / moad_* dims, configs/moad_fullatom_cond.yml:32-38): the tcgen05
    kernels are templated on the width (accumulator N = H, H/64 pipeline chunks); the fp32 FFMA kernels stay available."""
    cfg, sd, inp, want, edges = load_golden(case)
    net = make_net(cfg, sd)
    assert net.math_mode == 15          # 'auto' picks the tensor-core path for these widths too
    net.math_mode = mode
    got_a, got_r = run(net, inp)
    assert_close(got_a, want[0], f'{case} mode {mode} ligand out')
    assert_close(got_r, want[1], f'{case} mode {mode} pocket out')


def test_tensor_core_mode_rejected_for_unsupported_width():
    cfg = DynamicsConfig(joint_nf=16, hidden_nf=64, n_layers=2)
    sd = syn.synthetic_state_dict(cfg, 1)
    inp = syn.synthetic_denoiser_inputs(cfg, [5, 7], [20, 17], seed=2)
    net = make_net(cfg, sd)
    assert net.math_mode == 0
    want = egnn_oracle.denoiser_forward(cfg, sd, *inp)
    got = run(net, inp)
    assert_close(got[0], want[0], 'H=64 ligand out')
    with pytest.raises(RuntimeError, match='128, 192 and 256'):
        net.math_mode = '3xfp16'


def test_fp16_split_range_overflow_is_reported():
    """3xFP16 operands overflow beyond |x| ~ 6.5e4: the result turns NaN and the reference's NaN convention fires
    (ValueError); the range-robust 3xTF32 path handles the same input."""
    cfg, sd, inp, want, _ = load_golden('config1_n64_l4')
    big = {k: v.clone() for k, v in sd.items()}
    big['egnn.embedding.bias'] = big['egnn.embedding.bias'] + 3.0e5      # hidden features far outside the fp16 range
    net = make_net(cfg, big)
    with pytest.raises(ValueError, match='NaN detected'):
        run(net, inp)
    net.math_mode = '3xtf32'
    a = run(net, inp)
    net.math_mode = 'fp32'
    b = run(net, inp)
    assert torch.isfinite(a[0]).all() and torch.allclose(a[0], b[0], atol=1e-3, rtol=1e-3)


@pytest.mark.parametrize('case', golden_cases())
def test_golden_forward(case):
    cfg, sd, inp, want, edges = load_golden(case)
    net = make_net(cfg, sd)
    got_a, got_r = run(net, inp)
    assert net.last_num_edges == edges.shape[1]
    ea = assert_close(got_a, want[0], f'{case} ligand out')
    er = assert_close(got_r, want[1], f'{case} pocket out')
    print(f'{case}: max abs err ligand {ea:.2e} pocket {er:.2e}')


def test_forward_does_not_mutate_inputs_and_is_repeatable():
    cfg, sd, inp, want, _ = load_golden('ragged_b3_l4')
    net = make_net(cfg, sd)
    dev = [x.cuda() for x in inp]
    keep = [x.clone() for x in dev]
    with torch.no_grad():
        a1, r1 = net(*dev)
        a2, r2 = net(*dev)
    for x, k in zip(dev, keep):
        assert torch.equal(x, k)
    # tensor-core path: a receiver's messages are reduced per 32-row warp group and combined with RED.ADD, so the
    # summation order of >2 partials can vary run to run (fp32 rounding level, like the reference's own scatter_add_ on GPU)
    assert torch.allclose(a1, a2, atol=2e-6, rtol=1e-5) and torch.allclose(r1, r2, atol=2e-6, rtol=1e-5)
    net.math_mode = 'fp32'
    with torch.no_grad():
        b1, q1 = net(*dev)
        b2, q2 = net(*dev)
    # fp32 FFMA path: every receiver spans at most two partial sums at these degrees -> bitwise repeatable
    assert torch.equal(b1, b2) and torch.equal(q1, q2)
    assert torch.allclose(a1, b1, atol=ATOL, rtol=RTOL)


def test_oracle_parity_fresh_batch():
    """8 graphs with the per-graph shape of BASELINE configs[2] (N_L=25, N_P=175), full 6-layer net."""
    cfg = FULLATOM_COND
    sd = syn.synthetic_state_dict(cfg, 11)
    inp = syn.synthetic_denoiser_inputs(cfg, [25] * 8, [175] * 8, seed=12)
    assert syn.min_cutoff_margin(cfg, inp[0], inp[1], inp[3], inp[4]) > 2e-5
    want = egnn_oracle.denoiser_forward(cfg, sd, *inp)
    got = run(make_net(cfg, sd), inp)
    assert_close(got[0], want[0], 'ligand out')
    assert_close(got[1], want[1], 'pocket out')


def _rot(seed):
    g = torch.Generator().manual_seed(seed)
    q, r = torch.linalg.qr(torch.randn(3, 3, generator=g, dtype=torch.float64))
    q = q * torch.sign(torch.diagonal(r))
    if torch.det(q) < 0:
        q[:, 0] = -q[:, 0]
    return q


def test_se3_equivariance_and_reflection_sensitivity():
    """vel rotates with the input, h is invariant (SURVEY.md §4); with reflection_equivariant=False a
    mirror image must NOT be equivariant (the cross-product term changes sign)."""
    cfg = CONFIG1
    sd = syn.synthetic_state_dict(cfg, 0)
    inp = syn.synthetic_denoiser_inputs(cfg, [12, 9], [40, 31], seed=21)
    net = make_net(cfg, sd)
    base = run(net, inp)
    Rm, shift = _rot(3), torch.tensor([0.7, -1.1, 0.4], dtype=torch.float64)

    def transform(M):
        xa, xr = inp[0].clone().double(), inp[1].clone().double()
        xa[:, :3] = xa[:, :3] @ M.T + shift
        xr[:, :3] = xr[:, :3] @ M.T + shift
        return (xa.float(), xr.float()) + tuple(inp[2:])

    rot = run(net, transform(Rm))
    assert_close(rot[0][:, :3], (base[0][:, :3].double() @ Rm.T).float(), 'rotated vel', atol=2e-5)
    assert_close(rot[0][:, 3:], base[0][:, 3:], 'invariant h (ligand)', atol=2e-5)
    assert_close(rot[1][:, 3:], base[1][:, 3:], 'invariant h (pocket)', atol=2e-5)
    mirror = torch.diag(torch.tensor([-1.0, 1.0, 1.0], dtype=torch.float64))
    ref = run(net, transform(mirror))
    dev = (ref[0][:, :3].double() - base[0][:, :3].double() @ mirror.T).abs().max()
    assert dev > 1e-3, 'cross-product branch inactive?'


def test_permutation_equivariance_within_graph():
    cfg = CONFIG1
    sd = syn.synthetic_state_dict(cfg, 0)
    inp = syn.synthetic_denoiser_inputs(cfg, [14], [50], seed=22, t_value=0.3)
    net = make_net(cfg, sd)
    base = run(net, inp)
    g = torch.Generator().manual_seed(5)
    pa, pr = torch.randperm(14, generator=g), torch.randperm(50, generator=g)
    perm = run(net, (inp[0][pa], inp[1][pr], inp[2], inp[3], inp[4]))
    assert_close(perm[0], base[0][pa], 'permuted ligand', atol=2e-5)
    assert_close(perm[1], base[1][pr], 'permuted pocket', atol=2e-5)


def test_nan_raises_value_error_and_recovers():
    cfg, sd, inp, want, _ = load_golden('config1_n64_l4')
    net = make_net(cfg, sd)
    bad = inp[0].clone()
    bad[3, 1] = float('nan')
    with pytest.raises(ValueError, match='NaN detected in EGNN output'):
        run(net, (bad,) + tuple(inp[1:]))
    got = run(net, inp)     # the sticky flag was cleared by the raise
    assert_close(got[0], want[0], 'ligand after NaN')


def test_argument_errors():
    cfg, sd, inp, _, _ = load_golden('config1_n64_l4')
    net = make_net(cfg, sd)
    with pytest.raises(RuntimeError, match='CUDA'):
        with torch.no_grad():
            net(*inp)      # CPU tensors: no fallback
    dev = [x.cuda() for x in inp]
    with pytest.raises(ValueError, match='non-decreasing'):
        with torch.no_grad():
            net(dev[0], dev[1], dev[2], dev[3], torch.flip(torch.arange(48, device='cuda') // 24, [0]))
    net.train()
    with pytest.raises(NotImplementedError):
        net(*dev)


def test_weight_update_repacks():
    cfg, sd, inp, want, _ = load_golden('config1_n64_l4')
    net = make_net(cfg, sd)
    a = run(net, inp)[0]
    with torch.no_grad():
        net.egnn.embedding.bias.add_(0.05)
    b = run(net, inp)[0]
    assert (a - b).abs().max() > 1e-4
    net.load_state_dict(sd)
    c = run(net, inp)[0]
    assert torch.allclose(a, c, atol=2e-6, rtol=1e-5)     # same weights again (RED.ADD order may differ in the last bit)


def test_full_size_properties_config3():
    """BASELINE configs[2] size (B=64, N=200): too slow for the oracle at full batch; check size-independent
    properties: per-graph results are independent of batching (graph 5 alone == graph 5 in the batch),
    conditional mode leaves pocket velocities exactly zero, every edge joins same-graph nodes."""
    cfg = FULLATOM_COND
    sd = syn.synthetic_state_dict(cfg, 0)
    B = 64
    inp = syn.synthetic_denoiser_inputs(cfg, [25] * B, [175] * B, seed=3)
    net = make_net(cfg, sd)
    out = run(net, inp)
    E = net.last_num_edges
    assert 64 * 3000 < E < 64 * 8000
    assert torch.count_nonzero(out[1][:, :3]) == 0
    edges = net.get_edges(inp[3].cuda(), inp[4].cuda(), inp[0][:, :3].cuda(), inp[1][:, :3].cuda()).cpu()
    mask = torch.cat([inp[3], inp[4]])
    assert edges.shape[1] == E and torch.all(mask[edges[0]] == mask[edges[1]])
    key = edges[0] * mask.numel() + edges[1]
    assert torch.all(key[1:] > key[:-1]), 'edges not sorted by (row, col)'
    g = 5
    sa, sr = inp[3] == g, inp[4] == g
    single = (inp[0][sa], inp[1][sr], inp[2][g:g + 1], torch.zeros(int(sa.sum()), dtype=torch.int64),
              torch.zeros(int(sr.sum()), dtype=torch.int64))
    one = run(net, single)
    assert_close(one[0], out[0][sa], 'graph 5 alone vs batched (ligand)', atol=2e-6, rtol=1e-5)
    assert_close(one[1], out[1][sr], 'graph 5 alone vs batched (pocket)', atol=2e-6, rtol=1e-5)
    want = egnn_oracle.denoiser_forward(cfg, sd, *single)
    assert_close(one[0], want[0], 'graph 5 vs oracle')


def test_full_batch_oracle_config3():
    """BASELINE configs[2] at FULL size (B=64, N_L=25, N_P=175, 6 layers): every output row of the native kernels against
    the CPU oracle (one oracle call, a few seconds on the box's host cores)."""
    cfg = FULLATOM_COND
    sd = syn.synthetic_state_dict(cfg, 0)
    inp = syn.synthetic_denoiser_inputs(cfg, [25] * 64, [175] * 64, seed=43)      # seed with no pair within 2e-5 A of a cut-off
    assert syn.min_cutoff_margin(cfg, inp[0], inp[1], inp[3], inp[4]) > 2e-5
    torch.set_num_threads(min(32, torch.get_num_threads() or 1) or 1)
    want = egnn_oracle.denoiser_forward(cfg, sd, *inp)
    net = make_net(cfg, sd)
    for mode in ('3xfp16', '3xtf32'):
        net.math_mode = mode
        got = run(net, inp)
        ea = assert_close(got[0], want[0], f'full batch ligand out ({mode})')
        er = assert_close(got[1], want[1], f'full batch pocket out ({mode})')
        print(f'configs[2] full batch, {mode}: E={net.last_num_edges} max abs err ligand {ea:.2e} pocket {er:.2e}')


def test_single_cta_kernel_forms_still_match():
    """dsb_set_kernel_variants(0): the single-CTA edge kernels that stream the weight images and the separate node MLP +
    merged GEMM launches (the forms 3xTF32 always uses) in 3xFP16, against the golden vectors; then back to the default
    CTA-pair forms, which must agree with them to rounding."""
    from diffsbdd_b200 import _native
    lib = _native.load()
    cfg, sd, inp, want, edges = load_golden('fullatom_b2_n200_l6')
    net = make_net(cfg, sd)
    net.math_mode = '3xfp16'
    old = lib.dsb_set_kernel_variants(0)
    try:
        a = run(net, inp)
        assert_close(a[0], want[0], 'single-CTA forms, ligand out')
        assert_close(a[1], want[1], 'single-CTA forms, pocket out')
        for v in (1, 2):
            lib.dsb_set_kernel_variants(v)
            b = run(net, inp)
            assert_close(b[0], want[0], f'kernel variants {v}, ligand out')
    finally:
        lib.dsb_set_kernel_variants(old)
    assert old == 3
    c = run(net, inp)
    assert_close(c[0], a[0], 'pair vs single-CTA forms', atol=3e-6, rtol=1e-5)


def test_more_row_tiles_than_cta_pairs():
    """100 graphs x (25 + 175) nodes = 157 row tiles = 79 tile pairs on 74 CTA pairs: five pairs of the fused node block
    kernel work on a SECOND item (slot hand-over between items, accumulator phase carried across items).  The graphs whose
    pocket rows fall into those items must come out as when run alone; one of them is checked against the oracle."""
    cfg = FULLATOM_COND
    sd = syn.synthetic_state_dict(cfg, 0)
    B = 100
    inp = syn.synthetic_denoiser_inputs(cfg, [25] * B, [175] * B, seed=11)
    net = make_net(cfg, sd)
    out = run(net, inp)
    assert torch.count_nonzero(out[1][:, :3]) == 0
    for g in (0, 93, 97, 99):
        sa, sr = inp[3] == g, inp[4] == g
        single = (inp[0][sa], inp[1][sr], inp[2][g:g + 1], torch.zeros(int(sa.sum()), dtype=torch.int64),
                  torch.zeros(int(sr.sum()), dtype=torch.int64))
        one = run(net, single)
        assert_close(one[0], out[0][sa], f'graph {g} alone vs batched (ligand)', atol=3e-6, rtol=1e-5)
        assert_close(one[1], out[1][sr], f'graph {g} alone vs batched (pocket)', atol=3e-6, rtol=1e-5)
    want = egnn_oracle.denoiser_forward(cfg, sd, *single)
    assert_close(one[0], want[0], 'graph 99 vs oracle')


@pytest.mark.parametrize('case', ['sin_h256_l2', 'sin_emb8_joint_h128_l2'])
def test_golden_sin_embedding(case):
    """sin_embedding=True (egnn_new.py:282-293; unused by the shipped configs): 2 x 12 sinusoidal distance features in the fp32
    FFMA kernels; the tensor-core modes are rejected for such a module."""
    from diffsbdd_b200 import _native
    cfg, sd, inp, want, edges = load_golden(case)
    net = make_net(cfg, sd)
    assert net.math_mode == 0
    got_a, got_r = run(net, inp)
    assert net.last_num_edges == edges.shape[1]
    assert_close(got_a, want[0], f'{case} ligand out')
    assert_close(got_r, want[1], f'{case} pocket out')
    with pytest.raises(_native.NativeError):
        net.math_mode = '3xfp16'
    net.math_mode = 'fp32'
