"""Generate golden vectors by running the LIVE reference (a checkout of
https://github.com/GrumpyZhou/patch2pix) on CPU:

    PATCH2PIX_REFERENCE=/path/to/patch2pix python tests/golden/make_golden.py

Writes tests/golden/*.npz; the tests only read those files, never the reference.
The reference is imported unmodified except for the
two import-time shims documented in SURVEY.md Appendix B (skip the ResNet
checkpoint download; do not .cuda() the NC net on a CPU-only host).
"""
import os
import sys
import warnings
from argparse import Namespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
if not os.environ.get('PATCH2PIX_REFERENCE'):
    sys.exit('set PATCH2PIX_REFERENCE to a checkout of the reference patch2pix repository')
sys.path.insert(0, os.environ['PATCH2PIX_REFERENCE'])
warnings.filterwarnings('ignore')

import networks.resnet as resnet                                   # noqa: E402
resnet.ResNet.load_pretrained_ = lambda self, ignore='fc': None     # shim 1
import networks.ncn.model as ncm                                    # noqa: E402
_orig_init = ncm.NeighConsensus.__init__
ncm.NeighConsensus.__init__ = lambda self, use_cuda=True, **kw: _orig_init(self, use_cuda=False, **kw)  # shim 2
from networks.patch2pix import Patch2Pix                            # noqa: E402
from networks.modules import maxpool4d, L2Normalize                 # noqa: E402
from networks.ncn.model import MutualMatching                       # noqa: E402
from networks.utils import filter_coarse                            # noqa: E402

from patch2pix_b200.synth import make_seeded_state_dict, synthetic_pair, synthetic_pair_shifted  # noqa: E402
sys.path.insert(0, HERE)
from filter_cases import FILTER_CASES, filter_case_inputs           # noqa: E402


def build_ref(sd, panc):
    cfg = Namespace(training=False, device='cpu', regr_batch=1200, backbone='ResNet34',
                    feat_idx=[0, 1, 2, 3], weights_dict=sd, change_stride=True,
                    regressor_config=Namespace(conv_dims=[512, 512], conv_kers=[3, 3], conv_strs=[2, 1],
                                               fc_dims=[512, 256], feat_comb='pre', psize=[16, 16],
                                               pshift=8, panc=panc, shared=False))
    return Patch2Pix(cfg).eval()


def np_(t):
    return t.detach().cpu().numpy()


def case_stages(net, name, pair_idx, H, W, ksize=2, gen=synthetic_pair):
    """predict_fine path with every intermediate of the coarse stage."""
    im1, im2 = gen(pair_idx, H, W)
    out = {'pair_idx': pair_idx, 'H': H, 'W': W, 'ksize': ksize}
    with torch.no_grad():
        f1s, f2s = [], []
        net.extract.forward_all(im1, f1s, early_feat=True)
        net.extract.forward_all(im2, f2s, early_feat=True)
        for lvl in (1, 2, 3, 4):
            out[f'feat1_l{lvl}_sub'] = np_(f1s[lvl][0, ::7, ::3, ::3])   # sparse probe of the backbone
        a = L2Normalize(f1s[-1], dim=1)
        b = L2Normalize(f2s[-1], dim=1)
        corr = net.combine(a, b)
        pooled, mi, mj, mk, ml = maxpool4d(corr, k_size=ksize)
        out['pooled'] = np_(pooled)
        out['delta'] = np.stack([np_(mi), np_(mj), np_(mk), np_(ml)]).astype(np.int8)
        m1 = MutualMatching(pooled)
        out['mutual1'] = np_(m1)
        nc = net.ncn(m1)
        out['ncn'] = np_(nc)
        corr4d, delta4d = net.forward_coarse_match(f1s[-1], f2s[-1], ksize=ksize)
        out['corr4d'] = np_(corr4d)
        cm, sc = net.cal_coarse_matches(corr4d, delta4d, ksize=ksize, upsample=net.upsample, center=True)
        out['cand_matches'] = np_(cm)
        out['cand_scores'] = np_(sc)
        fm, fs = filter_coarse(cm, sc, 0.0, True)
        out['mutual_matches'] = np_(fm[0])
        out['mutual_scores'] = np_(fs[0])
        fine, fine_p, mid, mid_p, coarse = net.predict_fine(im1, im2, ksize=ksize, return_all=True)
        out['fine'] = np_(fine[0]).reshape(-1, 4)
        out['fine_p'] = np_(fine_p[0]).reshape(-1)
        out['mid'] = np_(mid[0]).reshape(-1, 4)
        out['mid_p'] = np_(mid_p[0]).reshape(-1)
        out['coarse'] = np_(coarse[0])
        pc_m, pc_s = net.predict_coarse(im1, im2, ksize=ksize, ncn_thres=0.0, mutual=False)
        out['predict_coarse_nomutual_matches'] = np_(pc_m[0])
        out['predict_coarse_nomutual_scores'] = np_(pc_s[0])
    np.savez_compressed(os.path.join(HERE, name + '.npz'), **out)
    print(name, 'mutual', out['mutual_matches'].shape, 'fine', out['fine'].shape)


def reference_tie_rows(net, corr4d, feat1, feat2, ksize, tie_eps=1e-6, margin_eps=2e-5):
    """Candidate rows of the reference's own output that are ambiguous under fp32 rounding: the selected cell's 2^4
    pooling window has a top-2 gap <= tie_eps, or the argmax of its corr4d row / column has a top-2 margin
    <= margin_eps * max(corr4d).  Computed from the LIVE reference's tensors (same rule as tests/_tie_masks)."""
    mm = corr4d[0, 0].reshape(corr4d.shape[2] * corr4d.shape[3], -1)
    nA, nB = mm.shape
    scale = mm.max().clamp_min(1e-30)
    tA, tB = mm.topk(2, dim=0)[0], mm.topk(2, dim=1)[0]
    fragile = torch.cat([(tA[0] - tA[1]) <= margin_eps * scale, (tB[:, 0] - tB[:, 1]) <= margin_eps * scale])
    corr = net.combine(L2Normalize(feat1, dim=1), L2Normalize(feat2, dim=1))
    k = ksize
    sl = torch.cat([corr[:, :, i::k, j::k, a::k, b::k] for i in range(k) for j in range(k) for a in range(k) for b in range(k)], 1)
    top2 = sl.topk(2, dim=1)[0]
    tie = ((top2[:, 0] - top2[:, 1]) <= tie_eps)[0].reshape(nA, nB)
    ia, ib = mm.argmax(0), mm.argmax(1)
    return fragile | torch.cat([tie[ia, torch.arange(nB)], tie[torch.arange(nA), ib]])


def case_train_sequence(net8, name, pair_idx, H, W, ptmax, np_seed, gen=synthetic_pair):
    """train_patch2pix.py:97-118 forward sequence under eval()/no_grad (ptmax, panc=8)."""
    im1, im2 = gen(pair_idx, H, W)
    out = {'pair_idx': pair_idx, 'H': H, 'W': W, 'ptmax': ptmax, 'np_seed': np_seed}
    with torch.no_grad():
        corr4d, delta4d, feats1, feats2 = net8.forward(im1, im2, ksize=2, return_feats=True)
        cm, sc = net8.cal_coarse_matches(corr4d, delta4d, ksize=2, upsample=net8.upsample, center=True)
        out['cand_matches'] = np_(cm)
        out['cand_scores'] = np_(sc)
        out['cand_fp32_tie'] = np_(reference_tie_rows(net8, corr4d, feats1[-1], feats2[-1], 2))
        np.random.seed(np_seed)
        cm, sc = filter_coarse(cm, sc, 0.0, True, ptmax=ptmax)
        out['sampled'] = np_(cm[0])
        out['sampled_scores'] = np_(sc[0])
        cm = net8.shift_to_anchors(cm)
        out['anchors'] = np_(cm[0])
        mid, mid_p = net8.forward_fine_match(feats1, feats2, cm, psize=16, ptype='center', regressor=net8.regress_mid)
        fine, fine_p = net8.forward_fine_match(feats1, feats2, mid, psize=16, ptype='center', regressor=net8.regress_fine)
        out['mid'] = np_(mid[0])
        out['mid_p'] = np_(mid_p[0])
        out['fine'] = np_(fine[0])
        out['fine_p'] = np_(fine_p[0])
    np.savez_compressed(os.path.join(HERE, name + '.npz'), **out)
    print(name, 'anchors', out['anchors'].shape)


def case_refine_only(net, name, pair_idx, H, W, n):
    """Patch2Pix.refine_matches with float coarse matches incl. border / out-of-range rows."""
    im1, im2 = synthetic_pair(pair_idx, H, W)
    g = torch.Generator().manual_seed(77)
    cm = torch.rand(n, 4, generator=g) * torch.tensor([W, H, W, H]) * 1.1 - 0.05 * torch.tensor([W, H, W, H])
    cm[0] = torch.tensor([0.0, 0.0, W - 1.0, H - 1.0])
    cm[1] = torch.tensor([W + 3.0, -2.5, 7.999, 8.0])
    with torch.no_grad():
        refined, scores, coarse = net.refine_matches(im1, im2, cm.clone(), io_thres=0.0)
        refined_t, scores_t, coarse_t = net.refine_matches(im1, im2, cm.clone(), io_thres=0.5)
    np.savez_compressed(os.path.join(HERE, name + '.npz'), pair_idx=pair_idx, H=H, W=W, coarse_in=np_(cm),
                        refined=refined, scores=scores, coarse=coarse,
                        refined_t=refined_t, scores_t=scores_t, coarse_t=coarse_t)
    print(name, refined.shape, refined_t.shape)


def case_filter_quirks(name='filter_quirks'):
    """networks/utils.py:38-72 on crafted candidate lists: every branch of filter_coarse (SURVEY s8 a8 quirks 1-6)."""
    out = {}
    for cname, kind, thres, mutual, ptmax, seed in FILTER_CASES:
        rows, scores = filter_case_inputs(kind)
        np.random.seed(seed)
        fm, fs = filter_coarse([rows.clone()], [scores.clone()], thres, mutual, ptmax=ptmax)
        out[cname + '_matches'] = np_(fm[0])
        out[cname + '_scores'] = np_(fs[0])
        print(cname, tuple(fm[0].shape))
    np.savez_compressed(os.path.join(HERE, name + '.npz'), **out)


if __name__ == '__main__':
    if len(sys.argv) > 1 and sys.argv[1] == 'filter':      # only the (network-free) filter_coarse fixture
        case_filter_quirks()
        sys.exit(0)
    torch.manual_seed(0)
    if not (len(sys.argv) > 1 and sys.argv[1] == 'shift'):
        sd = make_seeded_state_dict(0)
        net1 = build_ref(dict(sd), panc=1)
        net8 = build_ref(dict(sd), panc=8)
        missing = [k for k in net1.state_dict() if k not in sd and 'layer4' not in k and 'num_batches' not in k]
        assert not missing, missing
        case_stages(net1, 'stages_96x128', 3, 96, 128)
        case_stages(net1, 'stages_128x96', 5, 128, 96)
        case_train_sequence(net8, 'trainseq_96x128', 3, 96, 128, ptmax=12, np_seed=123)
        case_refine_only(net1, 'refine_128x160', 9, 128, 160, 40)
        case_filter_quirks()
    # round 2: the benchmark workload family -- 'consensus' NC weights + 16-px-shifted views (hundreds of distinct
    # mutual matches instead of a dozen), so that proposal / refine parity is pinned on many distinct windows.
    # Pair indices were picked so that the reference's own candidate list has no fp32-tie rows (reference_tie_rows).
    sdc = make_seeded_state_dict(0, nc_init='consensus')
    netc1 = build_ref(dict(sdc), panc=1)
    netc8 = build_ref(dict(sdc), panc=8)
    case_stages(netc1, 'stages_shift_128x160', 1, 128, 160, gen=synthetic_pair_shifted)
    case_train_sequence(netc8, 'trainseq_shift_160x240', 12, 160, 240, ptmax=60, np_seed=321, gen=synthetic_pair_shifted)
