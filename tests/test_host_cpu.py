"""CPU tests (-m "not gpu") of everything that does not need a device: the C-ABI library loads and
exports every symbol include/octfusion_b200.h declares, state_dict parity with the reference, the synthetic
workload generator, the sharding rule, and the loud failure when no CUDA device is present."""
import ctypes
import os
import re
import subprocess
import sys
import pytest
import torch

from tests.util import UNCOND, COND, SMALL, model_shapes, GOLDEN
from oracle import restate as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from octfusion_b200 import _lib, build
    hdr = open(os.path.join(ROOT, 'include', 'octfusion_b200.h')).read()
    hdr = re.sub(r'/\*.*?\*/', '', hdr, flags=re.S)
    declared = set(re.findall(r'\b(of_[a-z0-9_]+)\s*\(', hdr))
    assert len(declared) >= 25
    lib = ctypes.CDLL(build.LIB)
    for name in declared:
        assert hasattr(lib, name), 'library does not export %s' % name
    assert declared == set(_lib.EXPORTED_SYMBOLS), declared ^ set(_lib.EXPORTED_SYMBOLS)
    assert lib.of_version() == 4


def test_argument_validation_without_gpu():
    """negative return + error text, no launch, no crash."""
    from octfusion_b200 import _lib
    g = _lib.GemmArgs()
    assert _lib.lib.of_gather_gemm_simt(ctypes.byref(g), None) == -1
    assert b'of_gather_gemm_simt' in _lib.lib.of_last_error()
    assert _lib.lib.of_pack_weight_tc_bytes(7, 100, 5, 128) == -1          # c not a multiple of 64
    assert _lib.lib.of_pack_weight_tc_bytes(7, 128, 5, 128) == (7 * 2 + 1) * 128 * 64 * 2


def test_splitk_plan_host_logic():
    """of_tc_splitk_plan is pure host arithmetic (148 SMs assumed without a device): split only launches whose 128-row
    tiles cannot fill half of the SMs, into whole K blocks, at least 4 per range, at most one wave of CTAs"""
    from octfusion_b200 import _lib
    def plan(m, n, c, taps, ntype=0, out_rows=None):
        g = _lib.GemmArgs()
        g.M, g.N, g.c0, g.c1, g.taps, g.ntype, g.dtype = m, n, c, 0, taps, ntype, 1          # dtype 1 = bf16
        g.out_rows = out_rows
        return _lib.lib.of_tc_splitk_plan(ctypes.byref(g))
    if torch.cuda.is_available() and torch.cuda.get_device_properties(0).multi_processor_count != 148:
        pytest.skip('the expected plans below are for 148 SMs')
    assert plan(2048, 256, 256, 27) == 9          # 108 K blocks, 16 tiles: 9 ranges of 12 (144 CTAs)
    assert plan(2048, 128, 512, 27) == 9          # 216 K blocks, 16 tiles
    assert plan(2048, 128, 128, 27) == 9          # 54 K blocks: 9 ranges of 6
    assert plan(2048, 256, 256, 1) == 1           # 4 K blocks: nothing to split
    assert plan(16384, 128, 128, 27) == 1         # 128 tiles already fill the SMs
    assert plan(907484, 128, 128, 7, 5) == 1
    assert plan(2048, 250, 256, 27) == 1          # N must be a multiple of 32
    assert plan(2048, 256, 100, 27) == 1          # c must be a multiple of 64 (tcgen05 path)
    assert _lib.lib.of_tc_splitk_plan(None) == 1


def test_no_cpu_fallback():
    if torch.cuda.is_available():
        pytest.skip('only meaningful on a host without a GPU')
    from octfusion_b200 import octree_from_splits, DualOctree
    from octfusion_b200.modules import GraphConv
    from octfusion_b200.synth import synth_splits
    l4, l5 = synth_splits(1, 0)
    with pytest.raises(RuntimeError):
        DualOctree(octree_from_splits(l4, l5, 1, device='cpu'))
    conv = GraphConv(8, 8, 7, 7, 0)

    class _Plan:  # a plan on the CPU must be refused, not silently computed
        tap = None
        node_type = None
    with pytest.raises(Exception):
        conv.run(torch.zeros(4, 8), _Plan())


@pytest.mark.parametrize('cfg', [UNCOND, COND, SMALL])
def test_hr_layout_matches_module_tree(cfg):
    shapes = model_shapes(cfg)
    _, hr = R.split_cfg(cfg)
    seq_in, _, seq_out = R.hr_layout(hr)
    for kind, p, _, _ in seq_in + seq_out:
        key = {'conv': 'weights', 'res': 'conv1.weights', 'down': 'downsample.weights', 'up': 'upsample.weights'}[kind]
        assert 'unet_hr.' + p + key in shapes


@pytest.mark.parametrize('cfg', [UNCOND, COND])
def test_state_dict_parity_with_reference(cfg):
    """against the reference nets' state_dict shapes stored by oracle/gen_golden.py"""
    import json
    with open(os.path.join(GOLDEN, 'state_shapes.json')) as f:
        table = json.load(f)
    want = {k: tuple(v) for k, v in table['cond' if cfg is COND else 'uncond'].items()}
    assert want == model_shapes(cfg)


def test_synth_is_deterministic_and_shapenet_sized():
    from octfusion_b200.synth import synth_splits
    a, b = synth_splits(4, 3), synth_splits(4, 3)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    l4, l5 = synth_splits(8, 0)
    n5, n6 = 8 * int(l4.sum()) / 8, 8 * int(l5.sum()) / 8
    assert 4000 < n5 < 12000 and 10000 < n6 < 40000


def test_shard_rules():
    from octfusion_b200.shard import shard_range, strided_indices
    for n, w in ((32, 8), (32, 3), (5, 8)):
        cover = []
        for r in range(w):
            lo, hi = shard_range(n, r, w)
            cover += list(range(lo, hi))
        assert cover == list(range(n))
        assert sorted(sum((strided_indices(n, r, w) for r in range(w)), [])) == list(range(n))


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from octfusion_b200.shard import all_gather_latents, shard_range
    lo, hi = shard_range(5, rank, world)
    x = torch.arange(lo * 3, hi * 3, dtype=torch.float32).reshape(-1, 3)      # ragged: 3 vs 2 rows
    out = torch.cat(all_gather_latents(x), 0)
    q.put((rank, out.tolist()))
    dist.destroy_process_group()


def test_ragged_all_gather_gloo_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    ps = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in ps:
        p.start()
    res = [q.get(timeout=120) for _ in ps]
    for p in ps:
        p.join(60)
    want = torch.arange(15, dtype=torch.float32).reshape(5, 3).tolist()
    assert all(r[1] == want for r in res)


def test_split_octree_round_trip_host():
    """stage-1 -> stage-2 handoff (reference utils/util_dualoctree.py:198-250): split signal -> octree -> split signal
    reproduces the sign pattern, and the octree built from it again is the same octree (index ops only: any device)."""
    import torch
    from octfusion_b200 import octree as P
    g = torch.Generator().manual_seed(11)
    s = torch.randn(2, 8, 16, 16, 16, generator=g)
    s[torch.rand(s.shape, generator=g) < 0.7] = -0.5
    a = P.split2octree_small(s, 6, 4)
    assert a.depth == 6 and int(a.nnum[5]) == 8 * int(a.nnum_nempty[4]) and int(a.nnum[6]) == 8 * int(a.nnum_nempty[5])
    assert int(a.nnum_nempty[5]) == int((s > 0).sum())
    back = P.octree2split_small(a, 4)
    assert torch.equal(back, 2.0 * (s > 0).float() - 1.0)
    b = P.split2octree_small(back, 6, 4)
    for d in range(4, 7):
        assert torch.equal(a.keys[d], b.keys[d]) and torch.equal(a.children[d], b.children[d])


def test_header_is_plain_c_and_struct_layouts_match_ctypes(tmp_path):
    """include/octfusion_b200.h compiles as C (gcc, no CUDA headers) and the struct layouts it declares are the ones
    octfusion_b200/_lib.py hands to ctypes (a field added on one side only would silently shift every pointer)."""
    import ctypes as C
    import os
    import shutil
    import subprocess
    from octfusion_b200 import _lib
    cc = shutil.which('gcc') or shutil.which('cc')
    if cc is None:
        import pytest
        pytest.skip('no host C compiler')
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / 'abi_check')
    subprocess.run([cc, '-std=c99', '-Wall', '-Werror', '-I', os.path.join(root, 'include'),
                    os.path.join(root, 'tests', 'c_abi_check.c'), '-o', exe], check=True)
    out = dict(l.split() for l in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.splitlines())
    g, o = _lib.GemmArgs, _lib.OctreeLevels
    assert int(out['sizeof_gemm_args']) == C.sizeof(g)
    for f in ('tap_tab', 'w', 'out', 'M', 'a_multi', 'nt_block', 'reverse', 'stat_out', 'stat_rows_per_sample'):
        assert int(out['off_' + f]) == getattr(g, f).offset, f
    assert int(out['sizeof_octree_levels']) == C.sizeof(o)
    assert int(out['off_nnum']) == o.nnum.offset and int(out['off_full_depth']) == o.full_depth.offset


@pytest.mark.parametrize('steps', [4, 10, 50, 100, 200, 1000])
def test_stage1_truncation_compares_in_float32_like_the_reference(steps):
    """reference octfusion_model_union.py:324 / :339 compare float32 time tensors against the Python scalar 0.7
    (cast to float32 by torch); linspace(1, 0, steps+1) contains float32(0.7) exactly for these step counts, where a
    float64 compare decides the other way (ADVICE round 1)."""
    from octfusion_b200.sampler import truncation_flags
    times = torch.linspace(1.0, 0.0, steps + 1)
    pairs = torch.stack((times[:-1], times[1:]), 0).unbind(-1)        # get_sampling_timesteps (:292-298), one sample
    do_sign, add_noise = truncation_flags(steps, 0.7)
    for i, (t, tn) in enumerate(pairs):
        assert do_sign[i] == bool(t < 0.7) and add_noise[i] == bool(tn > 0.7), i
    if steps >= 10:
        k = [i for i in range(steps) if float(times[i]) < 0.7 and not do_sign[i]]
        assert len(k) == 1          # the one step a double-precision compare would get wrong


def test_stat_plan_segment_tables():
    """ops.StatPlan (host/torch logic of the deterministic norm statistics): 32-row chunks split into per-sample
    segments, against a brute-force walk; covers samples smaller than a chunk, one sample only, and the dense layout."""
    from octfusion_b200.ops import StatPlan

    def brute(bid):
        rows = len(bid)
        chunk_seg, seg_sample = [], []
        for r in range(rows):
            if r % 32 == 0:
                chunk_seg.append(len(seg_sample))
            if r % 32 == 0 or bid[r] != bid[r - 1]:
                seg_sample.append(bid[r])
        chunk_seg.append(len(seg_sample))
        return chunk_seg, seg_sample

    g = torch.Generator().manual_seed(0)
    cases = []
    # three "sections" (leaves of two depths + nodes), each batch-sorted, with tiny and empty samples
    for counts in ([[5, 0, 40, 3], [70, 1, 1, 33], [100, 31, 64, 2]], [[4096], [100], [1000]], [[1, 1, 1]]):
        bid = []
        for sec in counts:
            for b, n in enumerate(sec):
                bid += [b] * n
        cases.append((bid, len(counts[0])))
    for bid, batch in cases:
        sp = StatPlan(len(bid), batch, sample_id=torch.tensor(bid, dtype=torch.int32))
        cs, ss = brute(bid)
        assert sp.n_seg == len(ss) and sp.chunk_seg.tolist() == cs
        off, idx = sp.sample_seg_off.tolist(), sp.sample_seg_idx.tolist()
        assert off[0] == 0 and off[-1] == len(ss)
        for b in range(batch):
            mine = idx[off[b]:off[b + 1]]
            assert mine == [k for k, s in enumerate(ss) if s == b]          # in row order
        slot = sp.seg_slot.tolist()
        assert sorted(slot) == list(range(len(ss))) and all(slot[s] == k for k, s in enumerate(idx))
    for rows_per_sample, batch in ((8, 5), (64, 3), (4096, 2)):
        sp = StatPlan(rows_per_sample * batch, batch, rows_per_sample=rows_per_sample, device='cpu')
        cs, ss = brute([r // rows_per_sample for r in range(rows_per_sample * batch)])
        assert sp.chunk_seg.tolist() == cs and sp.n_seg == len(ss)


def test_slice_splits_shards_the_batch():
    """bench.py --gpus N: every rank generates the same B shapes and keeps a contiguous block (strong scaling,
    BASELINE.json configs[2]).  The blocks partition the label arrays and each block builds the octree of exactly its
    shapes (per-shape node counts unchanged)."""
    from octfusion_b200.synth import synth_splits, slice_splits
    from octfusion_b200 import shard
    from oracle.octree_util import octree_from_splits
    b = 6
    l4, l5 = synth_splits(b, 0)
    full = octree_from_splits(l4, l5, b)
    per_shape = lambda oc, d, n: torch.bincount(oc.keys[d] >> 48, minlength=n)            # noqa: E731
    parts4, parts5, lo_all = [], [], 0
    for rank in range(4):
        lo, hi = shard.shard_range(b, rank, 4)
        assert lo == lo_all
        lo_all = hi
        a4, a5 = slice_splits(l4, l5, lo, hi)
        parts4.append(a4); parts5.append(a5)
        if hi > lo:
            oc = octree_from_splits(a4, a5, hi - lo)
            for d in (5, 6):
                assert torch.equal(per_shape(oc, d, hi - lo), per_shape(full, d, b)[lo:hi])
    assert lo_all == b and torch.equal(torch.cat(parts4), l4) and torch.equal(torch.cat(parts5), l5)
