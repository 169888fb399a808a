"""CPU-side checks (no GPU): the C-ABI library loads and exports every declared symbol, the host
mirror refuses to run without CUDA, the pair sharder works over gloo with world_size 2, and the
bench reference arm prints a well-formed line."""
import json
import os
import re
import subprocess
import sys
from argparse import Namespace

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    import __graft_entry__ as ge
    ge.build()
    from patch2pix_b200 import _lib
    hdr = open(os.path.join(ROOT, 'include', 'p2p_b200.h')).read()
    declared = re.findall(r'P2P_API\s+[\w\s\*]+?\b(p2p_\w+)\s*\(', hdr)
    assert len(declared) >= 18
    lib = _lib.load()
    for name in declared:
        assert hasattr(lib, name), f'{name} declared in include/p2p_b200.h but not exported'
        assert name in _lib.EXPORTED_SYMBOLS, f'{name} has no ctypes signature'
    assert lib.p2p_version() == 100
    assert lib.p2p_last_error() is not None


def test_c_abi_rejects_bad_arguments_without_a_gpu():
    from patch2pix_b200 import _lib
    lib = _lib.load()
    assert lib.p2p_destroy(None) == 0
    assert lib.p2p_set_option(None, b'mid_passes', 3) == -1
    assert b'null' in lib.p2p_last_error()
    import ctypes as C
    h = C.c_void_p()
    rc = lib.p2p_create(0, C.byref(h))
    if not torch.cuda.is_available():
        assert rc != 0 and lib.p2p_last_error()


def test_host_mirror_has_no_cpu_fallback():
    from patch2pix_b200.model import Patch2PixB200, filter_coarse
    cfg = Namespace(training=False, device='cpu', regr_batch=1200, backbone='ResNet34', feat_idx=[0, 1, 2, 3],
                    weights_dict=None, change_stride=True, regressor_config=None)
    with pytest.raises(RuntimeError, match='CUDA'):
        Patch2PixB200(cfg)
    with pytest.raises(RuntimeError):
        filter_coarse([torch.zeros(4, 4, dtype=torch.int64)], [torch.zeros(4)])
    cfg.training = True
    with pytest.raises(RuntimeError, match='inference'):
        Patch2PixB200(cfg)


def test_seeded_state_dict_matches_reference_names(seeded_sd):
    sd = seeded_sd
    assert tuple(sd['ncn.conv.0.weight'].shape) == (3, 16, 1, 3, 3, 3)
    assert tuple(sd['ncn.conv.2.weight'].shape) == (3, 1, 16, 3, 3, 3)
    assert tuple(sd['regress_mid.conv.0.weight'].shape) == (512, 518, 3, 3)
    assert tuple(sd['regress_fine.fc.6.weight'].shape) == (5, 256)
    assert 'extract.layer3.0.downsample.1.running_var' in sd
    from patch2pix_b200.synth import make_seeded_state_dict, synthetic_pair
    sd2 = make_seeded_state_dict(0)
    assert all(torch.equal(sd[k], sd2[k]) for k in sd)
    a, b = synthetic_pair(3, 96, 128)
    a2, _ = synthetic_pair(3, 96, 128)
    assert a.shape == (1, 3, 96, 128) and torch.equal(a, a2) and not torch.equal(a, b)


def test_backbone_matches_oracle_on_cpu(seeded_sd):
    from oracle import p2p_oracle as O
    from patch2pix_b200.backbone import ResNet34Features
    from patch2pix_b200.synth import synthetic_pair
    net = ResNet34Features(True).eval()
    sd = {k[len('extract.'):]: v for k, v in seeded_sd.items() if k.startswith('extract.')}
    missing, unexpected = net.load_state_dict(sd, strict=False)
    assert not unexpected and all('num_batches_tracked' in m for m in missing)
    im, _ = synthetic_pair(1, 64, 96)
    with torch.no_grad():
        got = net.forward_all(im, [], True)
        ref = O.backbone_forward_all(im, seeded_sd)
    assert [tuple(t.shape) for t in got] == [(1, 3, 64, 96), (1, 64, 32, 48), (1, 64, 16, 24), (1, 128, 8, 12), (1, 256, 8, 12)]
    for g, r in zip(got, ref):
        torch.testing.assert_close(g, r, rtol=1e-4, atol=1e-5)


def _shard_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from patch2pix_b200.sharding import PairSharder
    sh = PairSharder(rank, world, 'cpu')
    src = torch.arange(100, 112) if rank == 0 else torch.zeros(3, dtype=torch.int64)   # only rank 0's list counts
    mine = sh.scatter_pair_indices(src)
    local = torch.stack([torch.full((4, 5), float(p)) for p in mine.tolist()])          # [steps, patches, 5]
    stacked = sh.gather_results(local)
    flat = PairSharder.interleave(stacked)
    q.put((rank, mine.tolist(), flat[:, 0, 0].tolist()))
    dist.destroy_process_group()


def test_pair_sharding_gloo_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_shard_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    outs = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert outs[0][1] == list(range(100, 112, 2)) and outs[1][1] == list(range(101, 112, 2))
    assert outs[0][2] == [float(v) for v in range(100, 112)] == outs[1][2]


def test_bench_reference_arm_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0',
                        '--height', '96', '--width', '128', '--ptmax', '6', '--cpu-sample-patches', '8'],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line['impl'] == 'reference' and line['value'] > 0 and line['cpu_baseline']['kind'] == 'port'
    assert line['e2e']['h2d_bytes_per_step'] == 0 and line['unit'] == 'pairs/s'


def test_bench_dump_outputs_files(tmp_path):
    """bench.py --dump-outputs: one .npy per returned array, float32 / float64, values as given; a fixed seeded row sample
    past the size cap."""
    import numpy as np
    code = ('import sys, torch; import bench; d = sys.argv[1]; g = torch.Generator().manual_seed(0); '
            'res = torch.randn(300, 5, generator=g); anc = torch.randint(-8, 640, (300, 4), generator=g); '
            'bench.dump_outputs(d + "/all", res, anc); bench.DUMP_MAX_BYTES = 60 * 50; '
            'bench.dump_outputs(d + "/cut", res, anc, rank=1); bench.dump_outputs(d + "/cut2", res, anc, rank=1); '
            'torch.save((res, anc), d + "/in.pt")')
    r = subprocess.run([sys.executable, '-c', code, str(tmp_path)], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    res, anc = torch.load(tmp_path / 'in.pt')
    full = {f.name: np.load(f) for f in (tmp_path / 'all').iterdir()}
    assert sorted(full) == ['anchors.npy', 'fine_matches.npy', 'fine_scores.npy']
    assert full['fine_matches.npy'].dtype == np.float32 and np.array_equal(full['fine_matches.npy'], res[:, :4].numpy())
    assert full['fine_scores.npy'].dtype == np.float32 and np.array_equal(full['fine_scores.npy'], res[:, 4].numpy())
    assert full['anchors.npy'].dtype == np.float64 and np.array_equal(full['anchors.npy'], anc.numpy())
    rows = np.load(tmp_path / 'cut' / 'rows_rank1.npy').astype(np.int64)
    assert len(rows) == 50 and np.array_equal(rows, np.load(tmp_path / 'cut2' / 'rows_rank1.npy'))
    assert np.array_equal(np.load(tmp_path / 'cut' / 'fine_matches_rank1.npy'), res[rows, :4].numpy())
    assert np.array_equal(np.load(tmp_path / 'cut' / 'anchors_rank1.npy'), anc[rows].numpy())


def test_load_checkpoint_parses_the_released_file_format(tmp_path, seeded_sd):
    """utils/eval/model_helper.py:28-62: released checkpoints are pickled dicts holding a Namespace; the loader
    must read them (weights_only=False), reject other architectures, and -- with no GPU here -- stop at the
    constructor's 'no CPU fallback' error rather than silently building a CPU model."""
    from patch2pix_b200.eval_helper import load_checkpoint
    rc = Namespace(conv_dims=[512, 512], conv_kers=[3, 3], conv_strs=[2, 1], fc_dims=[512, 256], feat_comb='pre',
                   psize=[16, 16], pshift=8, panc=8, shared=False)
    good = tmp_path / 'p2p.pth'
    torch.save({'backbone': 'ResNet34', 'feat_idx': [0, 1, 2, 3], 'state_dict': seeded_sd, 'regressor_config': rc,
                'last_epoch': 24}, good)
    lines = []
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        load_checkpoint(str(good), device='cpu', lprint=lines.append)
    assert any('epochs:25' in ln for ln in lines)
    bad = tmp_path / 'r50.pth'
    torch.save({'backbone': 'ResNet50', 'feat_idx': [0, 1, 2, 3], 'state_dict': {}, 'regressor_config': rc}, bad)
    with pytest.raises(RuntimeError, match='released ResNet34'):
        load_checkpoint(str(bad), device='cpu', lprint=lines.append)
    nc = tmp_path / 'nc.pth'
    torch.save({k: v for k, v in seeded_sd.items() if not k.startswith('regress')}, nc)
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        load_checkpoint(str(nc), device='cpu', method='nc', lprint=lines.append)
    with pytest.raises(ValueError):
        load_checkpoint(str(nc), device='cpu', method='other', lprint=lines.append)


def test_preprocess_oracle_is_pinned_against_pillow():
    """SURVEY s8 f4: the numpy restatement of Pillow's 8-bit bicubic resampling (oracle/preprocess_oracle.py) equals
    Pillow bit for bit on down-, up- and mixed scaling, and the whole load_im_flexible tensor equals the reference's
    torchvision formulation."""
    PIL = pytest.importorskip('PIL')
    from PIL import Image
    import numpy as np
    from oracle import preprocess_oracle as PO
    rng = np.random.RandomState(0)
    for ho, wo, ht, wt in ((97, 131, 48, 64), (60, 80, 96, 128), (120, 160, 120, 80), (75, 100, 75, 100), (333, 500, 208, 320)):
        img = (rng.rand(ho, wo, 3) * 255).astype(np.uint8)
        ref = np.array(Image.fromarray(img).resize((wt, ht), Image.BICUBIC))
        assert np.array_equal(PO.resize_bicubic_u8(img, wt, ht), ref), (ho, wo, ht, wt)
    img = (rng.rand(375, 500, 3) * 255).astype(np.uint8)
    got, scale = PO.load_im_flexible_array(img, 2, 16, 320)
    wt, ht = PO.target_size(500, 375, 2, 16, 320)
    assert (wt, ht) == (320, 224) and scale == (500 / 320, 375 / 224)
    t = torch.from_numpy(np.array(Image.fromarray(img).resize((wt, ht), Image.BICUBIC))).permute(2, 0, 1).float().div(255)
    t = (t - torch.tensor([0.485, 0.456, 0.406]).view(3, 1, 1)) / torch.tensor([0.229, 0.224, 0.225]).view(3, 1, 1)
    assert np.array_equal(got, t.numpy())
    from patch2pix_b200.preprocess import cal_rescale_size
    for w, h, s in ((500, 375, 320), (1024, 768, 1024), (640, 480, 1000), (123, 457, 300)):
        assert cal_rescale_size(s, w, h, 2, 1 / 16) == PO.cal_rescale_size(s, w, h, 2, 1 / 16)


def test_shipped_library_is_blackwell_native_sass():
    """The hot kernels of the built library contain the sm_100a tensor-core / TMA mnemonics (tcgen05.mma = UTC*MMA incl.
    the cta_group::2 form, cp.async.bulk.tensor = UTMALDG / UTMASTG, cp.async.bulk = UBLKCP, tcgen05.ld = LDTM) and no
    legacy mma.sync (HMMA); profiles/r02_sass_summary.md is generated by the same scan (tools/sass_summary.py)."""
    import shutil
    if shutil.which('cuobjdump') is None:
        pytest.skip('cuobjdump not on PATH')
    import __graft_entry__ as ge
    ge.build()
    from patch2pix_b200 import _lib
    sass = subprocess.run(['cuobjdump', '-sass', _lib.LIB_PATH], capture_output=True, text=True, timeout=600).stdout
    per, cur = {}, None
    for ln in sass.splitlines():
        m = re.search(r'Function : (\S+)', ln)
        if m:
            cur = m.group(1)
            per[cur] = ''
        elif cur is not None:
            per[cur] += ln + '\n'

    def body(tag):
        hits = [v for k, v in per.items() if tag in k]
        assert hits, tag
        return '\n'.join(hits)
    assert re.search(r'(?<![A-Z])HMMA', sass) is None          # UTCHMMA is tcgen05; a bare HMMA would be mma.sync
    l1, l2 = body('nc_l1_umma_kernel'), body('nc_l2_umma_kernel')
    assert l1.count('UTCHMMA') == 12 and 'UBLKCP' in l1 and 'UTMASTG' in l1 and 'LDTM' in l1
    assert l2.count('UTCHMMA') >= 36 and 'UTMALDG' in l2 and 'LDTM' in l2
    c1 = body('umma_conv1_tma_kernel')
    assert 'UTCHMMA.2CTA' in c1 and 'UTMALDG' in c1
    gemm = body('umma_gemm_kernel')
    assert 'UTCHMMA.2CTA' in gemm and 'UTMALDG' in gemm and 'UTCBAR' in gemm
