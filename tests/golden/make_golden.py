"""Generates tests/golden/*.npz, tests/golden/second_draw/*.npz, tests/golden/fp64/*.npz and
tests/golden/state_dict_layout.json by running the UNMODIFIED reference (imported through oracle/ref_shim.py, which
finds its sources through DIFFSBDD_REFERENCE) on seeded synthetic inputs and weights.

    python tests/golden/make_golden.py [name ...]

Each fixture stores the forward arguments, the reference outputs of ``EGNNDynamics.forward``
(dynamics.py:87-167), the edge list the reference built (dynamics.py:169-187), the config, the weight
seed and a fingerprint of the regenerated weights (weights themselves are a pure function of the
seed — diffsbdd_b200/synthetic.py — and are not stored).
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from diffsbdd_b200.config import DynamicsConfig, CONFIG1, FULLATOM_COND, CA_COND  # noqa: E402
from diffsbdd_b200 import synthetic as syn  # noqa: E402
from oracle import ref_shim  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))

# name -> (cfg, n_lig list, n_pocket list, input seed, weight seed, density, t_value, norm_values)
CASES = {
    # BASELINE.json configs[0]: one graph, N=64, h_dim=256, 4 layers
    'config1_n64_l4': (CONFIG1, [16], [48], 1, 0, 0.045, 0.5, (1.0, 4.0)),
    # ragged multi-graph batch incl. a 1-atom ligand, per-graph t
    'ragged_b3_l4': (CONFIG1, [5, 9, 1], [30, 17, 40], 2, 0, 0.045, None, (1.0, 4.0)),
    # full-atom conditional dims, 6 layers, two N=200 graphs (per-graph shape of configs[2])
    'fullatom_b2_n200_l6': (FULLATOM_COND, [25, 25], [175, 175], 3, 0, 0.045, None, (1.0, 4.0)),
    # C-alpha conditional dims (residue_nf=20, sparse pocket), configs[1] per-graph shape
    'ca_b3_l6': (CA_COND, [25, 18, 30], [40, 33, 52], 4, 0, 0.007, None, (1.0, 1.0)),
    # joint model: all coordinates updated + velocity mean removal (dynamics.py:161-164), H=128
    'joint_b2_h128_l5': (DynamicsConfig(update_pocket_coords=True, joint_nf=32, hidden_nf=128, n_layers=5),
                         [12, 20], [60, 45], 5, 1, 0.045, None, (1.0, 4.0)),
    # moad full-atom conditional: edge-type embedding (dynamics.py:118-125), H=192, cutoffs 4/7
    'moad_emb8_h192_l3': (DynamicsConfig(hidden_nf=192, n_layers=3, edge_embedding_dim=8,
                                         edge_cutoff_pocket=4.0, edge_cutoff_interaction=7.0),
                          [14, 22], [70, 90], 6, 2, 0.045, None, (1.0, 4.0)),
    # reflection-equivariant (no cross-product MLP), two sub-layers, no cut-offs, scalar t (dynamics.py:105-107)
    'reflect_sub2_nocut_l2': (DynamicsConfig(n_layers=2, inv_sublayers=2, reflection_equivariant=True,
                                             edge_cutoff_pocket=None, edge_cutoff_interaction=None,
                                             hidden_nf=128, joint_nf=64),
                              [7, 11], [25, 19], 7, 3, 0.045, 'scalar', (1.0, 4.0)),
    # no attention / no tanh branches (egnn_new.py:41-42, :103) with a ligand cut-off
    'noatt_notanh_l2': (DynamicsConfig(n_layers=2, attention=False, tanh=False, edge_cutoff_ligand=3.0,
                                       hidden_nf=128, joint_nf=32),
                        [20, 15], [40, 50], 9, 4, 0.045, None, (1.0, 4.0)),
    # ---- hidden_nf=256 variants: the same branches on the tcgen05 kernels (VERDICT r1 "what's weak" #1) ----
    # crossdock_ca_joint.yml dims: joint model (all coordinates move, velocity mean removed), residue_nf=20, H=256
    'joint_ca_h256_l6': (DynamicsConfig(update_pocket_coords=True, residue_nf=20), [20, 14, 1], [45, 38, 27], 21, 5,
                         0.007, None, (1.0, 1.0)),
    # reflection-equivariant at H=256 (one coordinate MLP per tile, no cross product)
    'reflect_h256_l3': (DynamicsConfig(n_layers=3, reflection_equivariant=True), [9, 13], [41, 30], 22, 6, 0.045,
                        None, (1.0, 4.0)),
    # two invariant sub-layers per block at H=256 (second GCL's first layer is not merged into the previous GEMM)
    'sub2_h256_l2': (DynamicsConfig(n_layers=2, inv_sublayers=2), [10, 6], [33, 52], 23, 7, 0.045, None, (1.0, 4.0)),
    # no attention gate, no tanh at H=256, with a ligand cut-off
    'noatt_notanh_h256_l2': (DynamicsConfig(n_layers=2, attention=False, tanh=False, edge_cutoff_ligand=3.0),
                             [18, 12], [44, 36], 24, 8, 0.045, None, (1.0, 4.0)),
    # edge-type embedding table at H=256 (the has_tb branch of the tensor-core producers), moad cut-offs 4/7
    'emb8_h256_l3': (DynamicsConfig(n_layers=3, edge_embedding_dim=8, edge_cutoff_pocket=4.0,
                                    edge_cutoff_interaction=7.0), [11, 17], [60, 48], 25, 9, 0.045, None, (1.0, 4.0)),
    # joint + edge embedding + two sub-layers + reflection-equivariant in one net (moad_fullatom_joint-like, H=256)
    'joint_emb8_sub2_reflect_h256_l2': (DynamicsConfig(n_layers=2, update_pocket_coords=True, edge_embedding_dim=8,
                                                       inv_sublayers=2, reflection_equivariant=True,
                                                       edge_cutoff_pocket=4.0, edge_cutoff_interaction=7.0),
                                        [8, 15], [39, 51], 26, 10, 0.045, 'scalar', (1.0, 4.0)),
    # aggregation_method='mean' (egnn_new.py:330-334): messages and coordinate updates divided by the receiver's edge count;
    # conditional H=256 (tensor-core kernels) and joint H=128 with an isolated ligand atom behind a ligand cut-off
    'mean_h256_l3': (DynamicsConfig(n_layers=3, aggregation_method='mean'), [13, 21], [52, 47], 27, 11, 0.045, None, (1.0, 4.0)),
    'mean_joint_h128_l2': (DynamicsConfig(n_layers=2, aggregation_method='mean', update_pocket_coords=True, hidden_nf=128,
                                          joint_nf=32, edge_cutoff_ligand=2.0), [9, 16], [35, 28], 28, 12, 0.045, None, (1.0, 4.0)),
    # sin_embedding=True (egnn_new.py:282-293): 2 x 12 sinusoidal distance features instead of the two squared distances;
    # with the edge-type embedding behind them, H=256 and H=128
    'sin_h256_l2': (DynamicsConfig(n_layers=2, sin_embedding=True), [12, 9], [40, 33], 29, 13, 0.045, None, (1.0, 4.0)),
    'sin_emb8_joint_h128_l2': (DynamicsConfig(n_layers=2, sin_embedding=True, edge_embedding_dim=8, update_pocket_coords=True,
                                              hidden_nf=128, joint_nf=32), [10, 7], [30, 36], 30, 14, 0.045, None, (1.0, 4.0)),
}


# a second input draw (input seed 100) of three of the cases, written to second_draw/<case>.npz in the same format
SECOND_DRAW = ('ragged_b3_l4', 'moad_emb8_h192_l3', 'reflect_sub2_nocut_l2')
SECOND_DRAW_SEED = 100

# cases whose reference outputs are also computed in fp64 (the module and the stored inputs in double), written to
# fp64/<case>.npz: unlike fp32 outputs, these do not depend on the CPU and thread count beyond ~1e-15
FP64_CASES = ('config1_n64_l4', 'ca_b3_l6', 'joint_b2_h128_l5', 'mean_joint_h128_l2', 'reflect_sub2_nocut_l2',
              'noatt_notanh_l2', 'sin_emb8_joint_h128_l2')

# modules whose state-dict layout (keys in order, shapes, keys that name one shared tensor) goes to state_dict_layout.json
LAYOUT_CONFIGS = [CONFIG1, DynamicsConfig(update_pocket_coords=True, reflection_equivariant=True, hidden_nf=128),
                  DynamicsConfig(edge_embedding_dim=8, hidden_nf=192, n_layers=2, attention=False)]


def make_inputs(case, seed=None):
    cfg, n_lig, n_poc, case_seed, wseed, density, t_value, norm_values = CASES[case]
    seed = case_seed if seed is None else seed
    tv = 0.37 if t_value == 'scalar' else t_value
    inp = list(syn.synthetic_denoiser_inputs(cfg, n_lig, n_poc, seed=seed, density=density,
                                             t_value=tv, norm_values=norm_values))
    if t_value == 'scalar':
        inp[2] = inp[2][:1].reshape(1)
    return cfg, wseed, tuple(inp)


def tied_groups(state_dict):
    """Groups of state-dict keys that hold one tensor (a parameter shared between modules)."""
    by_ptr = {}
    for k, v in state_dict.items():
        by_ptr.setdefault(v.data_ptr(), []).append(k)
    return [g for g in by_ptr.values() if len(g) > 1]


def state_dict_layout(cfg):
    net = ref_shim.load_reference().EGNNDynamics(device='cpu', act_fn=torch.nn.SiLU(), **cfg.kwargs())
    sd = net.state_dict()
    return {'cfg': cfg.kwargs(), 'params': [[k, list(v.shape)] for k, v in sd.items()], 'tied': tied_groups(sd)}


def main():
    """Arguments, if any, name what to regenerate: a case, second_draw/<case>, fp64/<case> or state_dict_layout."""
    only = sys.argv[1:]
    todo = [(case, case, None) for case in CASES] + [('second_draw/' + c, c, SECOND_DRAW_SEED) for c in SECOND_DRAW]
    for name, case, seed in todo:
        if only and name not in only:
            continue
        cfg, wseed, inp = make_inputs(case, seed)
        sd = syn.synthetic_state_dict(cfg, wseed)
        margin = syn.min_cutoff_margin(cfg, inp[0], inp[1], inp[3], inp[4])
        assert margin > 1e-4, (case, margin)
        net = ref_shim.build_reference_dynamics(cfg, sd)
        with torch.no_grad():
            out_a, out_r = net(*inp)
            edges = net.get_edges(inp[3], inp[4], inp[0][:, :3], inp[1][:, :3])
        os.makedirs(os.path.dirname(os.path.join(OUT, name)), exist_ok=True)
        np.savez_compressed(
            os.path.join(OUT, name + '.npz'),
            xh_atoms=inp[0].numpy(), xh_residues=inp[1].numpy(), t=inp[2].numpy(),
            mask_atoms=inp[3].numpy(), mask_residues=inp[4].numpy(),
            out_atoms=out_a.numpy(), out_residues=out_r.numpy(),
            edges=edges.numpy().astype(np.int32),
            cfg=json.dumps(cfg.kwargs()), weight_seed=wseed,
            weight_checksum=syn.state_dict_checksum(sd), cutoff_margin=margin,
        )
        print(f'{name}: N_L={len(inp[3])} N_P={len(inp[4])} E={edges.shape[1]} margin={margin:.2e} '
              f'|vel|max={out_a[:, :3].abs().max():.3f} |h|max={out_a[:, 3:].abs().max():.3f}')
    for case in FP64_CASES:
        if only and 'fp64/' + case not in only:
            continue
        z = np.load(os.path.join(OUT, case + '.npz'))
        cfg = DynamicsConfig(**json.loads(str(z['cfg'])))
        net = ref_shim.build_reference_dynamics(cfg, syn.synthetic_state_dict(cfg, int(z['weight_seed']))).double()
        inp = [torch.from_numpy(z[k]) for k in ('xh_atoms', 'xh_residues', 't', 'mask_atoms', 'mask_residues')]
        with torch.no_grad():
            out_a, out_r = net(*[x.double() if x.is_floating_point() else x for x in inp])
        os.makedirs(os.path.join(OUT, 'fp64'), exist_ok=True)
        np.savez_compressed(os.path.join(OUT, 'fp64', case + '.npz'), out_atoms=out_a.numpy(), out_residues=out_r.numpy())
        print(f'fp64/{case}: |out|max={max(out_a.abs().max(), out_r.abs().max()):.3f}')
    if not only or 'state_dict_layout' in only:
        with open(os.path.join(OUT, 'state_dict_layout.json'), 'w') as f:
            json.dump([state_dict_layout(cfg) for cfg in LAYOUT_CONFIGS], f, indent=1)
            f.write('\n')
        print('state_dict_layout:', len(LAYOUT_CONFIGS), 'modules')


if __name__ == '__main__':
    main()
