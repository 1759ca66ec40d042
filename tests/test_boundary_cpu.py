"""CPU: drop-in boundary — state-dict / constructor / façade contracts (SURVEY.md §8(b))."""
import json
import os
from argparse import Namespace

import pytest
import torch

from diffsbdd_b200 import synthetic as syn
from diffsbdd_b200.config import CONFIG1, FULLATOM_COND, DynamicsConfig
from diffsbdd_b200.conditional_model import ConditionalDDPM
from diffsbdd_b200.dynamics import EGNNDynamics
from diffsbdd_b200.en_diffusion import EnVariationalDiffusion, DistributionNodes
from diffsbdd_b200.lightning_modules import LigandPocketDDPM


def tied_groups(state_dict):
    """Groups of state-dict keys that hold one tensor (as tests/golden/make_golden.py records them)."""
    by_ptr = {}
    for k, v in state_dict.items():
        by_ptr.setdefault(v.data_ptr(), []).append(k)
    return [g for g in by_ptr.values() if len(g) > 1]


def reference_layout(cfg):
    """State-dict layout of the reference module for ``cfg`` (tests/golden/state_dict_layout.json, written by
    tests/golden/make_golden.py): keys in order with shapes, and the groups of keys that hold one shared tensor."""
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'state_dict_layout.json')) as f:
        for entry in json.load(f):
            if entry['cfg'] == cfg.kwargs():
                return entry
    raise KeyError(f'no reference layout recorded for {cfg}')


@pytest.mark.parametrize('cfg', [CONFIG1, DynamicsConfig(update_pocket_coords=True, reflection_equivariant=True, hidden_nf=128),
                                 DynamicsConfig(edge_embedding_dim=8, hidden_nf=192, n_layers=2, attention=False)])
def test_state_dict_is_interchangeable_with_reference_module(cfg):
    ref = reference_layout(cfg)
    mine = EGNNDynamics.from_config(cfg)
    assert [[k, list(v.shape)] for k, v in mine.state_dict().items()] == ref['params']
    # a reference checkpoint (shared parameters stored under each of their keys) -> this module
    g = torch.Generator().manual_seed(0)
    r = {k: torch.randn(shape, generator=g) for k, shape in ref['params']}
    for group in ref['tied']:
        for k in group[1:]:
            r[k] = r[group[0]]
    mine.load_state_dict(r, strict=True)
    m = mine.state_dict()                               # and back
    assert list(m) == list(r) and all(torch.equal(m[k], r[k]) for k in r)
    assert tied_groups(m) == ref['tied']
    if not cfg.reflection_equivariant:                  # shared last layer stays shared (egnn_new.py:78)
        q = mine.egnn.e_block_0.gcl_equiv
        assert q.coord_mlp._modules['4'].weight is q.cross_product_mlp._modules['4'].weight


def test_constructor_defaults_and_attributes_match_reference_signature():
    net = EGNNDynamics(atom_nf=10, residue_nf=20, n_dims=3)
    assert (net.cfg.joint_nf, net.cfg.hidden_nf, net.cfg.n_layers, net.cfg.inv_sublayers) == (16, 64, 4, 2)
    assert net.update_pocket_coords is True and net.n_dims == 3 and net.mode == 'egnn_dynamics'
    assert net.edge_cutoff_l is None and net.edge_cutoff_p is None and net.edge_cutoff_i is None
    assert net.cfg.norm_constant == 0 and net.cfg.attention is False and net.cfg.tanh is False
    assert hasattr(net, 'egnn') and net.device == 'cpu' and net.node_nf == 17


def test_conditional_ddpm_requires_frozen_pocket():
    joint = EGNNDynamics.from_config(FULLATOM_COND.with_(update_pocket_coords=True, n_layers=1, hidden_nf=64))
    with pytest.raises(AssertionError):
        ConditionalDDPM(dynamics=joint, atom_nf=10, residue_nf=10, n_dims=3, size_histogram=[[1.0]],
                        timesteps=10, noise_schedule='polynomial_2', noise_precision=5e-4, loss_type='l2',
                        norm_values=(1, 4))


def test_norm_value_sanity_check_fires():
    dyn = EGNNDynamics.from_config(FULLATOM_COND.with_(n_layers=1, hidden_nf=64))
    with pytest.raises(ValueError, match='normalization value'):
        EnVariationalDiffusion(dynamics=dyn, atom_nf=10, residue_nf=10, n_dims=3, size_histogram=[[1.0]],
                               timesteps=500, noise_schedule='polynomial_2', noise_precision=5e-4, loss_type='l2',
                               norm_values=(1, 100.0))


def test_distribution_nodes_conditional_sampling():
    d = DistributionNodes([[0, 0, 5], [0, 0, 0], [7, 0, 0]])
    torch.manual_seed(0)
    n1 = d.sample_conditional(n1=None, n2=torch.tensor([2, 0, 2, 0]))
    assert n1.tolist() == [0, 2, 0, 2]


def _hparams(mode='pocket_conditioning', rep='full-atom'):
    egnn = Namespace(device='cuda', joint_nf=16, hidden_nf=64, n_layers=2, attention=True, tanh=True, norm_constant=1,
                     inv_sublayers=1, sin_embedding=False, normalization_factor=100, aggregation_method='sum',
                     edge_cutoff_ligand=None, edge_cutoff_pocket=5.0, edge_cutoff_interaction=5.0,
                     reflection_equivariant=False)
    diff = Namespace(diffusion_steps=20, diffusion_noise_schedule='polynomial_2', diffusion_noise_precision=5e-4,
                     diffusion_loss_type='l2', normalize_factors=[1, 4])
    return dict(outdir=None, dataset='crossdock', datadir=None, batch_size=4, lr=1e-3, egnn_params=egnn,
                diffusion_params=diff, num_workers=0, augment_noise=0, augment_rotation=False, clip_grad=True,
                eval_epochs=1, eval_params=Namespace(), visualize_sample_epoch=1, visualize_chain_epoch=1,
                auxiliary_loss=False, loss_params=Namespace(), mode=mode, node_histogram=[[1.0, 2.0], [3.0, 1.0]],
                pocket_representation=rep)


def test_lightning_facade_builds_and_roundtrips_checkpoint(tmp_path):
    model = LigandPocketDDPM(**_hparams())
    assert type(model.ddpm) is ConditionalDDPM and isinstance(model.ddpm.dynamics, EGNNDynamics)
    assert (model.atom_nf, model.aa_nf, model.x_dims) == (10, 10, 3)
    keys = set(model.state_dict())
    assert 'ddpm.gamma.gamma' in keys and 'ddpm.buffer' in keys
    assert 'ddpm.dynamics.egnn.e_block_1.gcl_equiv.cross_product_mlp.4.weight' in keys
    assert model.ddpm.dynamics.cfg.edge_embedding_dim is None     # optional keys read with .get (lightning_modules.py:153-158)
    ckpt = tmp_path / 'last.ckpt'
    torch.save({'state_dict': model.state_dict(), 'hyper_parameters': _hparams()}, ckpt)
    again = LigandPocketDDPM.load_from_checkpoint(str(ckpt), map_location='cpu')
    for k, v in model.state_dict().items():
        assert torch.equal(v.cpu(), again.state_dict()[k])      # the denoiser of `model` lives on cuda when there is one
    ca = LigandPocketDDPM(**_hparams(rep='CA'))
    assert ca.aa_nf == 20 and ca.pocket_type_encoder['A'] == 0
    joint = LigandPocketDDPM(**_hparams(mode='joint'))
    assert type(joint.ddpm) is EnVariationalDiffusion and joint.ddpm.dynamics.update_pocket_coords


def test_prepare_pocket_from_arrays_layout():
    model = LigandPocketDDPM(**_hparams())
    pocket = model.prepare_pocket_from_arrays([[0.0, 0, 0], [1, 0, 0], [0, 2, 0]], [0, 1, 2], repeats=2)
    assert pocket['x'].shape == (6, 3) and pocket['one_hot'].shape == (6, 10)
    assert pocket['size'].tolist() == [3, 3] and pocket['mask'].tolist() == [0, 0, 0, 1, 1, 1]
