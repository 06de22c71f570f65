"""Shared helpers of the parity tests: seeded inputs built once for the oracle (CPU) and the product
(CUDA) from the same synthetic split labels."""
from __future__ import annotations
import functools
import hashlib
import os
import numpy as np
import torch

from octfusion_b200.synth import synth_splits
from oracle import restate as R
from oracle.octree_util import octree_from_splits as oracle_octree

UNCOND = dict(
    image_size=[16, 64], input_depth=[4, 6], unet_type=['lr', 'hr'], df_type=['x0', 'eps'], full_depth=4,
    input_channels=[8, 3], out_channels=[8, 3], model_channels=[64, 128], num_res_blocks=[[1, 1, 1], [1, 1, 0]],
    attention_resolutions=[2, 4], channel_mult=[[1, 2, 4], [1, 2, 4]], num_heads=4, use_checkpoint=False, dims=3)
COND = dict(UNCOND, num_res_blocks=[[1, 1, 1], [2, 2, 0]], attention_resolutions=[2, 4, 8],
            channel_mult=[[1, 2, 4, 8], [1, 2, 4]], num_classes=5)
# a narrow net with the same topology: fast enough for CPU-side tests and golden fixtures
SMALL = dict(UNCOND, model_channels=[64, 64], channel_mult=[[1, 2], [1, 1, 2]], attention_resolutions=[2])
# the benchmarked configuration (bench.py: 8 latent channels, BASELINE.json "8 feature channels")
UNCOND8 = dict(UNCOND, input_channels=[8, 8], out_channels=[8, 8])
# golden full-forward cases (oracle/gen_golden.py UNET_CASES): name -> (config, batch, latent channels)
UNET_CASES = {'small': (SMALL, 2, 3), 'uncond': (UNCOND, 1, 3), 'cond': (COND, 1, 3),
              'uncond8': (UNCOND8, 2, 8), 'cond_b4': (COND, 4, 3)}
UNET_TS = [1.5, -0.5, 0.3, 2.2]
UNET_LABEL = [1, 3, 0, 4]


def relerr(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def digest(t) -> str:
    """fingerprint for exact comparison with a stored reference tensor: dtype, shape and bytes (SHA-256), so that
    large integer outputs (graphs, octree keys) are pinned bit for bit without storing them"""
    a = np.ascontiguousarray(t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else t)
    h = hashlib.sha256(('%s %s ' % (a.dtype.str, a.shape)).encode())
    h.update(a.tobytes())
    return h.hexdigest()


PIN_VALUES = 2048


def pin_rows(t):
    """every k-th row of `t` (rows = all but the last dimension), k chosen from t's shape so that about PIN_VALUES
    values remain: the sample of a large reference output kept under golden/, and the same sample of the
    output it is compared with"""
    t = t.reshape(-1, t.shape[-1]) if t.dim() > 1 else t
    return t[:: max(1, -(-t.numel() // PIN_VALUES))]


@functools.lru_cache(maxsize=8)
def oracle_doctree(batch, seed=0):
    l4, l5 = synth_splits(batch, seed)
    oct_ = oracle_octree(l4, l5, batch)
    return R.DualGraph(oct_), (l4, l5)


def product_doctree(batch, seed=0, device='cuda'):
    from octfusion_b200 import octree_from_splits, DualOctree
    l4, l5 = synth_splits(batch, seed)
    return DualOctree(octree_from_splits(l4, l5, batch, device=device))


def model_shapes(cfg, stage='hr'):
    """state_dict shapes of the product model (== the reference's; checked by test_state_dict_parity)."""
    from octfusion_b200 import graph_unet_union
    with torch.device('meta'):
        net = graph_unet_union.UNet3DModel(stage, **cfg)
    return {k: tuple(v.shape) for k, v in net.state_dict().items()}


def build_product(cfg, sd, device='cuda', stage='hr'):
    from octfusion_b200 import graph_unet_union
    net = graph_unet_union.UNet3DModel(stage, **cfg)
    net.load_state_dict(sd)
    return net.to(device).eval()


GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


# ---- GraphVAE decoder (SURVEY.md 8f rank 1; reference configs/vae_snet_train.yaml) ----
VAE = dict(depth=8, channel_in=4, nout=4, full_depth=4, depth_stop=6, depth_out=8, resblk_type='basic', bottleneck=4,
           resblk_num=2, code_channel=16, embed_dim=3)
VAE_SPLIT_BIAS = 0.15      # keeps the grown octree small enough for the CPU oracle (~15-25 % of the nodes split)


def vae_shapes():
    from octfusion_b200 import graph_vae
    with torch.device('meta'):
        net = graph_vae.GraphVAE(**VAE)
    return {k: tuple(v.shape) for k, v in net.state_dict().items()}


def vae_state_dict(seed=3):
    sd = R.seeded_state_dict(vae_shapes(), seed)
    for i in range(3):
        sd['predict.%d.1.linear.bias' % i] = torch.tensor([VAE_SPLIT_BIAS, -VAE_SPLIT_BIAS])
    return sd


def vae_code(rows, seed=1):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(rows, 3, generator=g)


def build_vae(sd, device='cuda'):
    from octfusion_b200 import graph_vae
    net = graph_vae.GraphVAE(**VAE)
    net.load_state_dict(sd)
    return net.to(device).eval()


def oracle_child_octree(octree_in, depth_out=8):
    """GraphVAE.create_child_octree (graph_vae.py:235-244) on the shim octree."""
    from oracle.ref_import import ensure_shim
    ensure_shim()
    from ocnn.octree import Octree
    fd, ds = octree_in.full_depth, octree_in.depth
    out = Octree(depth_out, fd, octree_in.batch_size, 'cpu')
    for d in range(fd + 1):
        out.octree_grow_full(d)
    out.depth = fd
    for d in range(fd, ds):
        out.octree_split((octree_in.children[d] >= 0).long(), d)
        out.octree_grow(d + 1)
        out.depth += 1
    return out


def oracle_grown_octree(labels, batch=1, seed=0):
    """depth-8 shim octree: the depth-6 child octree split with the given per-depth labels."""
    dg, _ = oracle_doctree(batch, seed)
    octree = oracle_child_octree(dg.octree)
    for d in (6, 7, 8):
        octree.octree_split(labels[d].int(), d)
        if d < 8:
            octree.octree_grow(d + 1)
            octree.depth += 1
    return octree
