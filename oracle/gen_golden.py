"""TEST INFRASTRUCTURE.  Regenerates tests/golden/*.npz by running the UNMODIFIED reference
(/root/reference, imported under the ocnn shim) on seeded inputs.  Run in the build container:

    python -m oracle.gen_golden
    python -m oracle.gen_golden pins      # only tests/golden/oracle_vs_reference.npz

The fixtures travel to the GPU box (where the reference tree does not exist) and pin both the oracle
(`-m "not gpu"`) and the CUDA path (`-m gpu`).  Inputs are regenerated from seeds by the tests; the stored
input checksums guard against a drifting generator.
"""
import os
import sys
import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_import, restate as R                      # noqa: E402
from oracle.octree_util import octree_from_splits                # noqa: E402
from octfusion_b200.synth import synth_splits                    # noqa: E402
from tests.util import UNCOND, SMALL, COND                       # noqa: E402

OUT = os.path.join(ROOT, 'tests', 'golden')


def checksum(t: torch.Tensor) -> float:
    return float(t.double().abs().sum())


def seeded_inputs(n, c, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, c, generator=g)


def mpu_inputs(octree, npts=2000, seed=21):
    """seeded query points (half near occupied depth-8 cells, half uniform) and regression values for mpu tests."""
    gen = torch.Generator().manual_seed(seed)
    reg = {d: torch.randn(int(octree.nnum[4:d + 1].sum()), 4, generator=gen) for d in (6, 7, 8)}
    x, y, z, b = octree.xyzb(8)
    pick = torch.randperm(x.numel(), generator=gen)[:npts]
    near = (torch.stack([x, y, z], 1)[pick].float() + torch.rand(npts, 3, generator=gen)) / 128.0 - 1.0
    uni = torch.rand(npts, 3, generator=gen) * 2 - 1
    pos = torch.cat([torch.cat([near, uni]), torch.zeros(2 * npts, 1)], 1)
    return pos, reg


def mpu_fixture():
    """outputs of the unmodified reference NeuralMPU (mpu.py:143-155; its hard-coded `.cuda()` patched to identity)."""
    import importlib
    from tests import util as U
    ref_import.load()
    mpu = importlib.import_module('models.networks.dualoctree_networks.mpu')
    g = np.load(os.path.join(OUT, 'vae_decode.npz'))
    labels = {d: torch.from_numpy(np.unpackbits(g['label%d' % d])[: int(g['nnum'][d])].astype(np.int64)) for d in (6, 7, 8)}
    octree = U.oracle_grown_octree(labels)
    pos, reg = mpu_inputs(octree)
    orig = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self
    try:
        out = mpu.NeuralMPU(4, 6, 8)(pos, reg, octree)
    finally:
        torch.Tensor.cuda = orig
    fx = {'pos_sum': checksum(pos), 'reg_sum': sum(checksum(v) for v in reg.values())}
    for d in (6, 7, 8):
        fx['fval%d' % d] = out[d][0].numpy()
        fx['flag%d' % d] = np.packbits(out[d][1].numpy())
    return fx


# round-2 additions to UNET_CASES (tests/util.py): the benchmarked 8-channel config and the cond config at the shard
# size of BASELINE.json configs[4] (B = 4 per GPU)
from tests.util import UNET_CASES, UNET_TS, UNET_LABEL           # noqa: E402


def _ref_doctree(ref, batch, seed):
    l4, l5 = synth_splits(batch, seed)
    doc = ref.dual_octree.DualOctree(octree_from_splits(l4, l5, batch))
    doc.post_processing_for_docnn()
    return doc


def unet_fixture(ref, name):
    """full HR forward of the unmodified reference on seeded inputs -> tests/golden/unet_<name>.npz"""
    cfg, batch, cc = UNET_CASES[name]
    net = ref.union.UNet3DModel('hr', **cfg).eval()
    sd = R.seeded_state_dict({k: tuple(v.shape) for k, v in net.state_dict().items()}, 1)
    net.load_state_dict(sd)
    d = _ref_doctree(ref, batch, 0)
    x = seeded_inputs(d.total_num, cc, 7)
    ts = torch.tensor(UNET_TS)[:batch]
    label = torch.tensor(UNET_LABEL)[:batch] if cfg.get('num_classes') else None
    y = net(unet_type='hr', x=x, doctree=d, timesteps=ts, unet_lr=net.unet_lr, label=label)
    np.savez_compressed(os.path.join(OUT, 'unet_%s.npz' % name), y=y.numpy(), x_sum=checksum(x),
                        w_sum=sum(checksum(v) for v in sd.values()), batch=batch)
    print(name, 'out absmax', float(y.abs().max()), 'N', d.total_num)


def state_shapes(ref):
    """state_dict shapes of the unmodified reference nets -> tests/golden/state_shapes.json (lets bench.py's CPU arm
    build seeded weights on hosts without the reference tree and without importing the product package)."""
    import json
    out = {}
    for name in ('uncond', 'uncond8', 'cond'):
        cfg = UNET_CASES[name][0]
        with torch.device('meta'):
            net = ref.union.UNet3DModel('hr', **cfg)
        out[name] = {k: list(v.shape) for k, v in net.state_dict().items()}
    with open(os.path.join(OUT, 'state_shapes.json'), 'w') as f:
        json.dump(out, f)
    print('state_shapes.json', {k: len(v) for k, v in out.items()})


# ---- tests/golden/oracle_vs_reference.npz: what the unmodified reference returns in tests/test_oracle_vs_reference.py.
# Integer and exactly compared results are stored as digests (tests/util.py `digest`), float results as a fixed row
# sample (`pin_rows`) beside their full shape.  The input builders below are shared with the tests.
PIN_GRAPHS = [(1, 0), (2, 0), (3, 5)]


def operator_inputs(rows5, rows6):
    """seeded inputs and parameters of the operator pins on the batch-2 dual graph: GraphConv 8->8 on the full depth-4
    layer, GraphConv 16->24 with 5 node types at depth 6, group norms at depth 5, attention"""
    g = torch.Generator().manual_seed(3)
    r = lambda *s: torch.randn(*s, generator=g)                  # noqa: E731
    inp = {'conv4_x': r(2 * 4096, 8), 'conv4_w': r(7 * 8, 8) / np.sqrt(7 * 8.0),
           'conv6_x': r(rows6, 16), 'conv6_w': r(7 * 21, 24) / np.sqrt(7 * 21.0)}
    for c in (24, 64, 384):
        inp['gn%d_w' % c], inp['gn%d_b' % c] = 1 + 0.1 * r(1, c), 0.1 * r(1, c)
        inp['gn%d_x' % c] = r(rows5, c) * 2 + 0.5
    inp['qkv'] = r(8, 96, 64)
    return inp


def handoff_split():
    """random stage-1 split signal [2, 8, 16, 16, 16], sparse like a surface"""
    g = torch.Generator().manual_seed(4)
    split = torch.randn(2, 8, 16, 16, 16, generator=g)
    split[torch.rand(split.shape, generator=g) < 0.6] = -1.0
    return split


def vae_fixture_labels():
    """per-depth split labels the reference's GraphVAE decoder chose in tests/golden/vae_decode.npz"""
    g = np.load(os.path.join(OUT, 'vae_decode.npz'))
    return {d: torch.from_numpy(np.unpackbits(g['label%d' % d])[: int(g['nnum'][d])].astype(np.int64)) for d in (6, 7, 8)}


def reference_pins(ref):
    import importlib
    import json
    from tests import util as U
    P = {}

    def pin(key, t):
        P[key], P[key + '_shape'] = U.pin_rows(t).numpy(), np.array(t.shape)

    for b, s in PIN_GRAPHS:                                       # dual graphs
        doc, pre = _ref_doctree(ref, b, s), 'graph_b%d_s%d_' % (b, s)
        for d in range(4, 7):
            k, c = R.edge_set(doc.graph[d])
            P[pre + 'key%d' % d], P[pre + 'col%d' % d] = U.digest(k), U.digest(c)
            P[pre + 'node_type%d' % d] = U.digest(doc.graph[d]['node_type'])
            P[pre + 'batch_id%d' % d] = U.digest(doc.batch_id(d))
        P[pre + 'nnum'], P[pre + 'lnum'] = U.digest(doc.nnum), U.digest(doc.lnum)
    for name, cfg in (('small', SMALL), ('uncond', UNCOND), ('cond', COND)):    # nets of the unet_<name>.npz forwards
        with torch.device('meta'):
            net = ref.union.UNet3DModel('hr', **cfg)
        P['unet_shapes_' + name] = json.dumps({k: list(v.shape) for k, v in net.state_dict().items()}, sort_keys=True)

    m, doc = ref.modules, _ref_doctree(ref, 2, 0)                 # operators
    inp = operator_inputs(doc.batch_id(5).shape[0], doc.batch_id(6).shape[0])
    for name, conv, d in (('conv4', m.GraphConv(8, 8, 7, 7, 0), 4), ('conv6', m.GraphConv(16, 24, 7, 7, 5), 6)):
        conv.weights.data.copy_(inp[name + '_w'])
        pin(name + '_y', conv(inp[name + '_x'], doc, d))
    for c in (24, 64, 384):
        gn = m.DualOctreeGroupNorm(c)
        gn.weights.data.copy_(inp['gn%d_w' % c]); gn.bias.data.copy_(inp['gn%d_b' % c])
        pin('gn%d_y' % c, gn(inp['gn%d_x' % c], doc, 5))
    pin('attn_y', m.QKVAttention()(inp['qkv']))
    P['temb'] = ref.util.timestep_embedding(torch.tensor([9.2, -2.3, 0.1]), 128).numpy()
    P['log_snr'] = float(ref.util.beta_linear_log_snr(torch.tensor(0.3)))

    gv = importlib.import_module('models.networks.dualoctree_networks.graph_vae')
    net = gv.GraphVAE(**U.VAE).eval()                             # GraphVAE decoder, growing its octree
    P['vae_shapes'] = json.dumps({k: list(v.shape) for k, v in net.state_dict().items()}, sort_keys=True)
    net.load_state_dict(U.vae_state_dict(5))
    doc = _ref_doctree(ref, 2, 3)
    code = U.vae_code(doc.total_num, 2)
    out = net.decode_code(code, doc, update_octree=True)
    P['vae_dec_code_sum'], P['vae_dec_nnum'] = checksum(code), U.digest(out['octree_out'].nnum)
    for d in (6, 7, 8):
        P['vae_dec_label%d' % d] = np.packbits(out['logits'][d].argmax(1).numpy().astype(np.uint8))
        P['vae_dec_keys%d' % d] = U.digest(out['octree_out'].keys[d])
        P['vae_dec_children%d' % d] = U.digest(out['octree_out'].children[d])
        pin('vae_dec_logit%d' % d, out['logits'][d])
        pin('vae_dec_reg%d' % d, out['reg_voxs'][d])

    net = gv.GraphVAE(**U.VAE).eval()                             # GraphVAE encoder on given input features
    net.load_state_dict(U.vae_state_dict())
    octree = U.oracle_grown_octree(vae_fixture_labels())
    doc = ref.dual_octree.DualOctree(octree)
    doc.post_processing_for_docnn()
    data = torch.randn(doc.total_num, 4, generator=torch.Generator().manual_seed(9))
    net._get_input_feature = lambda doctree: data
    P['vae_enc_data_sum'] = checksum(data)
    pin('vae_enc', net.KL_conv(net.octree_encoder_step(octree, doc)[6]))

    util = ref_import.load_util()                                 # stage-1 -> stage-2 handoff
    want = util.split2octree_small(handoff_split(), 6, 4)
    P['split_depth'], P['split_nnum'], P['split_nnum_nempty'] = want.depth, want.nnum.numpy(), want.nnum_nempty.numpy()
    for d in range(4, 7):
        P['split_keys%d' % d], P['split_children%d' % d] = U.digest(want.keys[d]), U.digest(want.children[d].int())
    P['split_back'] = U.digest(util.octree2split_small(want, 4))

    mpu = importlib.import_module('models.networks.dualoctree_networks.mpu')
    octree = U.oracle_grown_octree(vae_fixture_labels())          # NeuralMPU, its `.cuda()` patched to identity
    pos, reg = mpu_inputs(octree, 4000)
    orig = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self
    try:
        out = mpu.NeuralMPU(4, 6, 8)(pos, reg, octree)
    finally:
        torch.Tensor.cuda = orig
    for d in (6, 7, 8):
        pin('mpu_fval%d' % d, out[d][0])
        P['mpu_flag%d' % d] = U.digest(out[d][1])
    np.savez_compressed(os.path.join(OUT, 'oracle_vs_reference.npz'), **P)


def main():
    ref = ref_import.load()
    os.makedirs(OUT, exist_ok=True)
    torch.set_grad_enabled(False)
    if 'shapes' in sys.argv[1:]:
        state_shapes(ref)
        return
    if 'pins' in sys.argv[1:]:
        reference_pins(ref)
        return
    only = [a for a in sys.argv[1:] if a in UNET_CASES]
    if only:                                   # python -m oracle.gen_golden uncond8 cond_b4: just these fixtures
        for name in only:
            unet_fixture(ref, name)
        return

    def ref_doctree(batch, seed):
        return _ref_doctree(ref, batch, seed)

    # 1. dual graph of one shape: canonical sorted (row*7+dir, col) per depth
    doc = ref_doctree(1, 0)
    g = {}
    for d in range(4, 7):
        k, c = R.edge_set(doc.graph[d])
        g['key%d' % d], g['col%d' % d] = k.numpy().astype(np.int32), c.numpy().astype(np.int32)
        g['node_type%d' % d] = doc.graph[d]['node_type'].numpy().astype(np.uint8)
        g['batch_id%d' % d] = doc.batch_id(d).numpy().astype(np.int32)
    g['nnum'], g['lnum'] = doc.nnum.numpy(), doc.lnum.numpy()
    np.savez_compressed(os.path.join(OUT, 'dual_graph_b1_s0.npz'), **g)

    # 2. BASELINE.json configs[0] analogue: one GraphConv 8->8 on the depth-4 full layer of one octree
    conv = ref.modules.GraphConv(8, 8, 7, 7, 0)
    w = seeded_inputs(56, 8, 11) / np.sqrt(56.0)
    conv.weights.data.copy_(w)
    x = seeded_inputs(4096, 8, 12)
    np.savez_compressed(os.path.join(OUT, 'graphconv_config1.npz'), x=x.numpy(), w=w.numpy(),
                        y=conv(x, doc, 4).numpy())

    # 3. operators at depth 6 with node types / ragged norm / attention
    conv = ref.modules.GraphConv(64, 32, 7, 7, 5)
    w = seeded_inputs(7 * 69, 32, 13) / np.sqrt(7 * 69.0)
    conv.weights.data.copy_(w)
    n6 = doc.total_num
    x = seeded_inputs(n6, 64, 14)
    ops = {'conv_y': conv(x, doc, 6)[::16].numpy(),      # every 16th row keeps the fixture small
            'conv_x_sum': checksum(x), 'conv_w_sum': checksum(w)}
    gn = ref.modules.DualOctreeGroupNorm(64)
    gam, bet = 1 + 0.1 * seeded_inputs(1, 64, 15), 0.1 * seeded_inputs(1, 64, 16)
    gn.weights.data.copy_(gam); gn.bias.data.copy_(bet)
    doc2 = ref_doctree(2, 0)
    x2 = seeded_inputs(doc2.batch_id(5).shape[0], 64, 17) * 2 + 0.5
    ops['gn_y'] = gn(x2, doc2, 5)[::16].numpy()
    qkv = seeded_inputs(8 * 96, 64, 18).reshape(8, 96, 64)
    ops['attn_y'] = ref.modules.QKVAttention()(qkv).numpy()
    np.savez_compressed(os.path.join(OUT, 'operators.npz'), **ops)

    # 4. full U-Net forwards (weights from the shared seeded_state_dict)
    for name in UNET_CASES:
        unet_fixture(ref, name)
    state_shapes(ref)
    # 5. GraphVAE decoder (SURVEY.md 8f rank 1): decode_code(update_octree=True) of the unmodified reference
    import importlib
    from tests import util as U
    gv = importlib.import_module('models.networks.dualoctree_networks.graph_vae')
    vae = gv.GraphVAE(**U.VAE).eval()
    sd = U.vae_state_dict()
    vae.load_state_dict(sd)
    d_in = ref_doctree(1, 0)
    code = U.vae_code(d_in.total_num)
    out = vae.decode_code(code, d_in, update_octree=True)
    fx = {'code_sum': checksum(code), 'w_sum': sum(checksum(v) for v in sd.values()),
          'nnum': out['octree_out'].nnum.numpy(), 'nnum_nempty': out['octree_out'].nnum_nempty.numpy()}
    for d in (6, 7, 8):
        lg = out['logits'][d]
        fx['label%d' % d] = np.packbits(lg.argmax(1).numpy().astype(np.uint8))
        fx['margin%d' % d] = float((lg[:, 0] - lg[:, 1]).abs().min())
        fx['logit%d' % d] = lg[::16].numpy()
        fx['reg%d' % d] = out['reg_voxs'][d][::16].numpy()
    np.savez_compressed(os.path.join(OUT, 'vae_decode.npz'), **fx)
    print('vae nnum', fx['nnum'].tolist(), 'margins', [fx['margin%d' % d] for d in (6, 7, 8)])
    # 6. NeuralMPU (SURVEY.md 8f rank 4) on the octree grown above, random per-node regression values
    fx = mpu_fixture()
    np.savez_compressed(os.path.join(OUT, 'mpu_eval.npz'), **fx)
    # 7. the results tests/test_oracle_vs_reference.py compares the oracle with (reads vae_decode.npz written above)
    reference_pins(ref)
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)) // 1024, 'KB')


if __name__ == '__main__':
    main()
