"""Pins the oracle (oracle/restate.py) against what the UNMODIFIED reference modules returned on the same seeded
inputs: tests/golden/oracle_vs_reference.npz and the unet_*.npz / state_shapes.json fixtures, all written by
oracle/gen_golden.py.  Exact results are compared by digest, float results on a fixed row sample."""
import json
import os
import numpy as np
import pytest
import torch

from oracle import restate as R
from oracle.gen_golden import PIN_GRAPHS, operator_inputs, handoff_split, vae_fixture_labels, mpu_inputs, checksum
from tests.util import relerr, oracle_doctree, digest, pin_rows, GOLDEN, UNCOND, COND, SMALL


@pytest.fixture(scope='module')
def pins():
    return np.load(os.path.join(GOLDEN, 'oracle_vs_reference.npz'))


def _close(pins, key, got, tol):
    """`got` has the reference output's shape and its pinned row sample agrees within `tol`"""
    assert tuple(got.shape) == tuple(pins[key + '_shape']), key
    assert relerr(pin_rows(got), torch.from_numpy(pins[key])) < tol, key


def _same(pins, key, got):
    assert digest(got) == str(pins[key]), key


@pytest.mark.parametrize('batch,seed', PIN_GRAPHS)
def test_dual_graph_equals_reference(pins, batch, seed):
    dg, _ = oracle_doctree(batch, seed)
    pre = 'graph_b%d_s%d_' % (batch, seed)
    for d in range(4, 7):
        k, c = R.edge_set(dg.graph[d])
        _same(pins, pre + 'key%d' % d, k)
        _same(pins, pre + 'col%d' % d, c)
        _same(pins, pre + 'node_type%d' % d, dg.graph[d]['node_type'])
        _same(pins, pre + 'batch_id%d' % d, dg.batch_id(d))
    _same(pins, pre + 'nnum', dg.nnum)
    _same(pins, pre + 'lnum', dg.lnum)


@pytest.mark.parametrize('name', ['small', 'uncond', 'cond'])
def test_full_unet_equals_reference(pins, name):
    """the reference's HR forward with the seeded state_dict of its own net is tests/golden/unet_<name>.npz
    (UNET_TS / UNET_LABEL begin with the time steps [1.5, -0.5] and labels [1, 3] used here)"""
    cfg = {'uncond': UNCOND, 'cond': COND, 'small': SMALL}[name]
    sd = R.seeded_state_dict(json.loads(str(pins['unet_shapes_' + name])), 1)
    batch = 1 if name != 'small' else 2
    want = torch.from_numpy(np.load(os.path.join(GOLDEN, 'unet_%s.npz' % name))['y'])
    dg, _ = oracle_doctree(batch, 0)
    g = torch.Generator().manual_seed(7)
    x = torch.randn(dg.total_num, 3, generator=g)
    ts = torch.tensor([1.5, -0.5])[:batch]
    label = torch.tensor([1, 3])[:batch] if cfg.get('num_classes') else None
    lr_cfg, hr_cfg = R.split_cfg(cfg)
    got = R.hr_forward(x, dg, ts, sd, hr_cfg, lr_cfg, label=label)
    assert float(want.abs().max()) > 0.1          # the seeded weights must not leave the net at zero
    assert relerr(got, want) < 2e-5


def test_operators_equal_reference(pins):
    dg, _ = oracle_doctree(2, 0)
    inp = operator_inputs(dg.batch_id(5).shape[0], dg.batch_id(6).shape[0])
    # config-1 analogue: GraphConv 8->8 on the depth-4 full layer
    _close(pins, 'conv4_y', R.graph_conv(inp['conv4_x'], dg.graph[4], inp['conv4_w'], 0), 1e-6)
    _close(pins, 'conv6_y', R.graph_conv(inp['conv6_x'], dg.graph[6], inp['conv6_w'], 5), 1e-6)
    for c in (24, 64, 384):
        y = R.doctree_group_norm(inp['gn%d_x' % c], dg.batch_id(5), 2, inp['gn%d_w' % c], inp['gn%d_b' % c])
        _close(pins, 'gn%d_y' % c, y, 1e-5)
    _close(pins, 'attn_y', R.qkv_attention(inp['qkv']), 1e-6)
    t = torch.tensor([9.2, -2.3, 0.1])
    assert relerr(R.timestep_embedding(t, 128), torch.from_numpy(pins['temb'])) < 1e-6
    assert abs(float(R.beta_linear_log_snr(torch.tensor(0.3))) - float(pins['log_snr'])) < 1e-6


def test_vae_decode_equals_reference(pins):
    """GraphVAE (SURVEY.md 8f rank 1): state_dict parity of the product class and decode_code(update_octree=True) of
    the oracle against the reference on two shapes; the oracle grows its octree with the reference's labels."""
    from tests import util as U
    assert {k: tuple(v) for k, v in json.loads(str(pins['vae_shapes'])).items()} == U.vae_shapes()
    sd = U.vae_state_dict(5)
    dg, _ = oracle_doctree(2, 3)
    code = U.vae_code(dg.total_num, 2)
    assert abs(checksum(code) - float(pins['vae_dec_code_sum'])) < 1e-6 * float(pins['vae_dec_code_sum'])
    labels = {d: torch.from_numpy(np.unpackbits(pins['vae_dec_label%d' % d])[: int(pins['vae_dec_logit%d_shape' % d][0])]
                                  .astype(np.int64)) for d in (6, 7, 8)}
    mine = R.DualGraph(U.oracle_child_octree(dg.octree))
    logits, regs, octree = R.vae_decode(code, mine, sd, 6, 8, 2, update_octree=True, labels=labels)
    _same(pins, 'vae_dec_nnum', octree.nnum)
    for d in (6, 7, 8):
        _same(pins, 'vae_dec_keys%d' % d, octree.keys[d])
        _same(pins, 'vae_dec_children%d' % d, octree.children[d])
        _close(pins, 'vae_dec_logit%d' % d, logits[d], 1e-5)
        _close(pins, 'vae_dec_reg%d' % d, regs[d], 1e-5)


def test_vae_encode_equals_reference(pins):
    """GraphVAE.octree_encoder_step + KL_conv on given input features (the reference builds them from point clouds
    with ocnn InputFeature, which is outside the path: `_get_input_feature` was replaced by a seeded tensor)."""
    from tests import util as U
    sd = U.vae_state_dict()
    octree = U.oracle_grown_octree(vae_fixture_labels())
    dg = R.DualGraph(octree)
    data = torch.randn(dg.total_num, 4, generator=torch.Generator().manual_seed(9))
    assert abs(checksum(data) - float(pins['vae_enc_data_sum'])) < 1e-6 * float(pins['vae_enc_data_sum'])
    _close(pins, 'vae_enc', R.vae_encode(data, dg, sd, 8, 6, 2), 1e-5)


def test_split_octree_handoff_equals_reference(pins):
    """stage-1 -> stage-2 handoff (SURVEY.md 8f rank 2): split2octree_small / octree2split_small of the product
    (device-agnostic index ops) against the reference's, on a random split signal and its round trip."""
    from octfusion_b200 import octree as P
    got = P.split2octree_small(handoff_split(), 6, 4)
    assert got.depth == int(pins['split_depth']) == 6
    for d in range(4, 7):
        _same(pins, 'split_keys%d' % d, got.keys[d])
        _same(pins, 'split_children%d' % d, got.children[d])
    assert got.nnum.tolist() == pins['split_nnum'].tolist()
    assert got.nnum_nempty.tolist() == pins['split_nnum_nempty'].tolist()
    back = P.octree2split_small(got, 4)
    _same(pins, 'split_back', back)
    # round trip: the octree built from its own split signal is the same octree
    again = P.split2octree_small(back, 6, 4)
    for d in range(4, 7):
        assert torch.equal(again.keys[d], got.keys[d]) and torch.equal(again.children[d], got.children[d])


def test_neural_mpu_equals_reference(pins):
    """NeuralMPU (SURVEY.md 8f rank 4, oracle only): per-point restatement against reference mpu.py on the octree and
    regression values of the VAE fixture case."""
    from tests import util as U
    octree = U.oracle_grown_octree(vae_fixture_labels())
    # query points: near occupied depth-8 cells (so that every depth contributes) plus uniform ones (mostly coarse)
    pos, reg = mpu_inputs(octree, 4000)
    mine = R.mpu_eval(pos, reg, octree, 4, 6, 8)
    for d in (6, 7, 8):
        _same(pins, 'mpu_flag%d' % d, mine[d][1])
        _close(pins, 'mpu_fval%d' % d, mine[d][0], 1e-5)
    assert bool(mine[8][1].any()) and not bool(mine[8][1].all())
