#!/usr/bin/env python
"""Benchmark: image-pairs/sec of the Patch2Pix correlate-and-refine hot path at 640x480,
ptmax=400, panc=8 (BASELINE.json configs[2]; training-loop forward sequence under eval,
train_patch2pix.py:97-118), on N B200s of one node.

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference algorithm (CPU oracle port) on host cores
    python bench.py ... --dump-outputs DIR    # also write the last timed step's matches / scores / anchors as .npy

One "step" = one image pair per GPU through the whole hot path (weak scaling: pair p of step s
goes to rank p % N; no data-path collective, NCCL only broadcasts the pair indices and gathers
the matches).  `value` times the hot path with the feature pyramids already in HBM;
`e2e` times pinned-host images -> H2D -> cuDNN backbone -> hot path -> D2H of the matches.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True       # the benchmark leaves the source tree as it found it (it may be read-only)

H_DEF, W_DEF, PTMAX_DEF, PANC_DEF = 480, 640, 400, 8
MAC_CONV1, MAC_CONV2 = 152764416, 150994944        # per patch, dense count (SURVEY.md s8d)
N_DISTINCT = 8                                      # distinct synthetic pairs cycled per rank


def workload_string(W, H, ptmax):
    """Identical in both arms (the driver compares the strings)."""
    cfgno = {(640, 480, 400): 2, (480, 320, 200): 1, (1024, 768, 1000): 3}.get((W, H, ptmax))
    tag = f' (BASELINE configs[{cfgno}])' if cfgno is not None else ''
    return (f'{W}x{H} pair, ptmax={ptmax} panc={PANC_DEF} -> {ptmax * PANC_DEF} patches/stage{tag}; synthetic '
            f'16-px-shifted views + consensus NC weights (distinct proposals)')


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--height', type=int, default=H_DEF)
    ap.add_argument('--width', type=int, default=W_DEF)
    ap.add_argument('--ptmax', type=int, default=PTMAX_DEF)
    ap.add_argument('--mid-passes', type=int, default=None)
    ap.add_argument('--fine-passes', type=int, default=None)
    ap.add_argument('--corr-passes', type=int, default=None)
    ap.add_argument('--seg-len', type=int, default=None)
    ap.add_argument('--mid-band', type=int, default=None)
    ap.add_argument('--fuse-gather', type=int, default=None)
    ap.add_argument('--gemm-pair', type=int, default=None, help='bitmask of GEMM launches on the CTA-pair kernel')
    ap.add_argument('--nc-impl', type=int, default=None, help='1: tensor-core NeighConsensus (default), 0: fp32 CUDA-core kernels')
    ap.add_argument('--backbone-fp32', action='store_true', help='keep cuDNN TF32 off in the e2e backbone')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--e2e-overlap', type=int, default=0, help='1: backbone graph of the next pair on a side stream (overlaps the hot path)')
    ap.add_argument('--e2e-modes', default='tf32,fp16,fp32', help='backbone variants timed end to end (the first is the headline)')
    ap.add_argument('--pairs', type=int, default=0,
                    help='strong-scaling mode (BASELINE configs[4]): this many pairs in total, sharded over the ranks; '
                         'rank 0 re-computes a sample of the other ranks\' pairs and checks bit-equality')
    ap.add_argument('--depth', type=int, default=3, help='pairs in flight per GPU (coarse stages enqueued ahead of the host sync)')
    ap.add_argument('--legacy-workload', action='store_true', help="round-1 generator (13-17 mutual matches per pair)")
    ap.add_argument('--cpu-sample-patches', type=int, default=200)
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the hot path returned in the last timed step as DIR/<name>.npy '
                         '(fine_matches, fine_scores float32; anchors float64); with more than one GPU, each rank writes '
                         'its own pair with a _rank<r> suffix')
    args = ap.parse_args()
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of the CUDA path (--impl ours)')
    return args


def model_config(device, panc):
    from argparse import Namespace
    rc = Namespace(conv_dims=[512, 512], conv_kers=[3, 3], conv_strs=[2, 1], fc_dims=[512, 256], feat_comb='pre',
                   psize=[16, 16], pshift=8, panc=panc, shared=False)
    return Namespace(training=False, device=device, regr_batch=1200, backbone='ResNet34', feat_idx=[0, 1, 2, 3],
                     weights_dict=None, change_stride=True, regressor_config=rc)


def load_traffic():
    """DRAM bytes (read + write) per launch from the committed `ncu --set full` capture of the round
    (profiles/r02_traffic.json: kernel kind -> bytes), or {}."""
    p = os.path.join(ROOT, 'profiles', 'r02_traffic.json')
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f)
    return {}


def load_peaks():
    """Burst peak for a kernel whose timed region is short (clocks near max), sustained for seconds-long regions."""
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {'hbm_gbs': d['hbm_gbs'], 'tflops_burst': d['bf16_tflops'],
                'tflops_sustained': d.get('bf16_tflops_sustained', d['bf16_tflops']), 'src': 'measured'}
    return {'hbm_gbs': 6650.0, 'tflops_burst': 1590.0, 'tflops_sustained': 1400.0, 'src': 'fallback'}


_SAMPLER_SRC = r"""
import sys, time
import pynvml as N
N.nvmlInit()
h = N.nvmlDeviceGetHandleByIndex(int(sys.argv[1]))
reasons = getattr(N, 'nvmlDeviceGetCurrentClocksEventReasons', None) or N.nvmlDeviceGetCurrentClocksThrottleReasons
print('ready', N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM), flush=True)
sys.stdin.readline()                      # 'go'
import select
i, pw, slow = 0, 0.0, 0.0
while not select.select([sys.stdin], [], [], 0.01)[0]:
    t0 = time.perf_counter()
    if i % 8 == 0:
        pw = N.nvmlDeviceGetPowerUsage(h) / 1e3
    c, r = N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM), int(reasons(h))
    slow = max(slow, time.perf_counter() - t0)
    print(c, pw, r, flush=False)
    i += 1
print('slowest', slow * 1e3)
sys.stdout.flush()
"""


class ClockSampler:
    """Samples SM clock / power / throttle reasons through NVML every ~10 ms while the timed region runs -- in a separate
    PROCESS (a sampler thread in this interpreter contends for the GIL with the launch loop and shows up as launch gaps;
    nvidia-smi's own start-up would miss a 0.5 s region)."""

    def __init__(self, index):
        self.index, self.proc, self.sm_max, self.err, self.slowest_ms = index, None, None, None, None
        try:
            vis = os.environ.get('CUDA_VISIBLE_DEVICES')
            phys = int(vis.split(',')[index]) if vis and vis.split(',')[index].isdigit() else index
            self.proc = subprocess.Popen([sys.executable, '-u', '-c', _SAMPLER_SRC, str(phys)], stdin=subprocess.PIPE,
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            line = self.proc.stdout.readline().split()
            if len(line) == 2 and line[0] == 'ready':
                self.sm_max = float(line[1])
            else:
                raise RuntimeError('sampler did not start')
        except Exception as e:       # no sampler process: fall back to a thread in this interpreter (still real NVML samples)
            self.err, self.proc = repr(e), None
        self.thread = None

    def _thread_loop(self):
        try:
            import pynvml as N
            N.nvmlInit()
            vis = os.environ.get('CUDA_VISIBLE_DEVICES')
            phys = int(vis.split(',')[self.index]) if vis and vis.split(',')[self.index].isdigit() else self.index
            h = N.nvmlDeviceGetHandleByIndex(phys)
            self.sm_max = float(N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM))
            reasons = getattr(N, 'nvmlDeviceGetCurrentClocksEventReasons', None) or N.nvmlDeviceGetCurrentClocksThrottleReasons
            while not self._halt.is_set():
                self._rows.append((float(N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)), N.nvmlDeviceGetPowerUsage(h) / 1e3,
                                   int(reasons(h))))
                self._halt.wait(0.02)
        except Exception as e:
            self.err = repr(e)

    def start(self):
        if self.proc:
            self.proc.stdin.write('go\n')
            self.proc.stdin.flush()
        else:
            self._rows, self._halt = [], threading.Event()
            self.thread = threading.Thread(target=self._thread_loop, daemon=True)
            self.thread.start()

    def finish(self):
        rows = []
        if self.thread is not None:
            self._halt.set()
            self.thread.join(timeout=5)
            rows = list(self._rows)
        if self.proc:
            try:
                out, _ = self.proc.communicate('stop\n', timeout=10)
                for ln in out.splitlines():
                    p = ln.split()
                    if len(p) == 3:
                        rows.append((float(p[0]), float(p[1]), int(p[2])))
                    elif len(p) == 2 and p[0] == 'slowest':
                        self.slowest_ms = float(p[1])
            except Exception as e:
                self.err = repr(e)
                self.proc.kill()
        if not rows:
            return {'sm_mhz': None, 'sm_max_mhz': self.sm_max, 'reasons': ['unavailable: ' + str(self.err)]}
        bits = {'hw_slowdown': 0x8, 'hw_thermal_slowdown': 0x40, 'sw_thermal_slowdown': 0x20, 'sw_power_cap': 0x4,
                'hw_power_brake_slowdown': 0x80}
        allbits = 0
        for r in rows:
            allbits |= r[2]
        return {'sm_mhz': statistics.median(r[0] for r in rows), 'sm_min_mhz': min(r[0] for r in rows),
                'sm_max_mhz': self.sm_max, 'power_w_max': max(r[1] for r in rows), 'samples': len(rows),
                'interval_ms': 10 if self.proc else 20, 'slowest_nvml_query_ms': self.slowest_ms,
                'source': 'nvml (separate process)' if self.proc else 'nvml (thread)', 'reasons': [n for n, b in bits.items() if allbits & b]}


# --------------------------------------------------------------------------------------------------
# CPU arm: the reference algorithm restated in oracle/p2p_oracle.py (the Python reference itself
# cannot travel to the GPU box).  One step = the full coarse stage of one pair + the two refine
# stages on a bounded subset of the 3200 patches, extrapolated to the full pair.
# --------------------------------------------------------------------------------------------------
def cpu_threads():
    """Threads for the CPU arm: every host core up to 32 (torch's CPU kernels for this path -- hundreds of
    small conv3d / index ops -- get slower, not faster, beyond that; measured on the 128-core GPU box).
    Override with P2P_CPU_THREADS."""
    cores = os.cpu_count() or 1
    return int(os.environ.get('P2P_CPU_THREADS', min(cores, 32)))


def cpu_step(O, sd, im1, im2, ptmax, panc, n_sample, nc_slices=None):
    """One bounded sample of the reference algorithm on the CPU for one pair: full backbone, full
    correlation / max-pool / mutual matching / proposals, the NC 4D conv on `nc_slices` of its
    first-dimension output slices (all if None) and the two refine stages on `n_sample` patches;
    the sampled parts are scaled to the full pair."""
    t0 = time.perf_counter()
    with torch.no_grad():
        f1 = O.backbone_forward_all(im1, sd)
        f2 = O.backbone_forward_all(im2, sd)
        t1 = time.perf_counter()
        a, b = O.l2_normalize(f1[-1], 1), O.l2_normalize(f2[-1], 1)
        corr, mi, mj, mk, ml = O.maxpool4d(O.feat_correlation_4d(a, b), 2)
        corr = O.mutual_matching(corr)
        t2 = time.perf_counter()
        hA = corr.shape[2]
        sl = None if (nc_slices is None or nc_slices >= hA) else list(range(0, hA, max(1, hA // nc_slices)))[:nc_slices]
        nc = O.neigh_consensus(corr, sd, sl)
        t3 = time.perf_counter()
        nc_scale = 1.0 if sl is None else hA / len(sl)
        corr4d = O.mutual_matching(nc if sl is None else corr)
        cm, sc = O.cal_coarse_matches(corr4d, (mi, mj, mk, ml), 2, upsample=O.UPSAMPLE, center=True)
        np.random.seed(0)
        cm, sc = O.filter_coarse(cm, sc, 0.0, True, ptmax=ptmax)
        anch = O.shift_to_anchors(cm, panc)
        t4 = time.perf_counter()
        n_full = anch[0].shape[0]
        sub = [anch[0][:n_sample]]
        mid, _ = O.forward_fine_match(f1, f2, sub, sd, 'regress_mid.')
        fine, _ = O.forward_fine_match(f1, f2, mid, sd, 'regress_fine.')
        t5 = time.perf_counter()
    n_sub = sub[0].shape[0]
    t_nc = (t3 - t2) * nc_scale
    t_refine = (t5 - t4) * n_full / max(n_sub, 1)
    hot = (t2 - t1) + t_nc + (t4 - t3) + t_refine
    return {'backbone_s': t1 - t0, 'coarse_s': (t2 - t1) + t_nc + (t4 - t3), 'nc_s_extrapolated': t_nc,
            'refine_s_extrapolated': t_refine, 'hot_path_s': hot, 'e2e_s': (t1 - t0) + hot, 'wall_s': t5 - t0,
            'n_sample': n_sub, 'n_full': n_full, 'nc_slices': 'all' if sl is None else f'{len(sl)}/{hA}'}


def make_workload(args):
    """(state_dict, pair generator): the benchmark workload family unless --legacy-workload."""
    from patch2pix_b200.synth import make_seeded_state_dict, synthetic_pair, synthetic_pair_shifted
    if args.legacy_workload:
        return make_seeded_state_dict(0), synthetic_pair
    return make_seeded_state_dict(0, nc_init='consensus'), synthetic_pair_shifted


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, res, anchors, rank=None):
    """Write one pair's hot-path outputs (`res` [patches, 5] = fine matches x1 y1 x2 y2 + confidence, `anchors` [patches, 4]
    int64) as .npy files, so that two builds can be compared output for output.  Past DUMP_MAX_BYTES a fixed seeded sample
    of the rows is written, with their indices in rows.npy."""
    os.makedirs(out_dir, exist_ok=True)
    out = {'fine_matches': res[:, :4].float(), 'fine_scores': res[:, 4].float(), 'anchors': anchors.double()}
    n = res.shape[0]
    cap = DUMP_MAX_BYTES // (4 * 4 + 4 + 4 * 8 + 8)
    if n > cap:
        rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:cap].sort().values
        out = {k: v[rows.to(v.device)] for k, v in out.items()}
        out['rows'] = rows.double()
    sfx = '' if rank is None else f'_rank{rank}'
    for name, t in out.items():
        np.save(os.path.join(out_dir, name + sfx + '.npy'), t.cpu().numpy())


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from oracle import p2p_oracle as O
    threads = cpu_threads()
    torch.set_num_threads(threads)
    sd, gen = make_workload(args)
    H, W = args.height, args.width
    pairs = [gen(p, H, W) for p in range(2)]
    # bounded sample per step (tier rule: the whole --steps/--warmup run must end within a few minutes): the NC 4D
    # conv runs on a subset of its output slices and the refine stages on a subset of the patches; both are scaled
    # to the full pair and the line says so ("extrapolated", with the sampled fractions)
    budget = 150.0 / max(args.steps + min(args.warmup, 1), 1)
    nc_slices, n_sample = (None, args.cpu_sample_patches) if budget > 12 else ((8, 96) if budget > 4 else (3, 32))
    for i in range(min(args.warmup, 1)):
        cpu_step(O, sd, *pairs[i % 2], args.ptmax, PANC_DEF, n_sample, nc_slices)
    rs = [cpu_step(O, sd, *pairs[i % 2], args.ptmax, PANC_DEF, n_sample, nc_slices) for i in range(args.steps)]
    hot = sum(r['hot_path_s'] for r in rs) / len(rs)
    e2e = sum(r['e2e_s'] for r in rs) / len(rs)
    wall = sum(r['wall_s'] for r in rs) / len(rs)
    hA = H // 16
    nc_frac = 1.0 if rs[0]['nc_slices'] == 'all' else int(rs[0]['nc_slices'].split('/')[0]) / hA
    sample = (f'per step, one {W}x{H} pair: full backbone + correlation/max-pool/mutual/proposals, NC 4D conv on '
              f'{rs[0]["nc_slices"]} output slices, mid+fine refine on {rs[0]["n_sample"]} of {rs[0]["n_full"]} patches; '
              f'sampled parts scaled to the full pair (measured wall {wall:.2f} s/step, extrapolated {e2e:.2f} s/pair)')
    line = {'impl': 'reference', 'metric': 'image-pairs/sec', 'value': 1.0 / e2e, 'unit': 'pairs/s', 'n_gpus': 0,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': e2e * 1e3, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'extrapolated': True, 'measured_wall_ms_per_step': wall * 1e3,
            'sampled_fractions': {'nc_output_slices': nc_frac, 'refine_patches': rs[0]['n_sample'] / rs[0]['n_full']},
            'config': {'workload': workload_string(W, H, args.ptmax),
                       'sequence': 'train_patch2pix.py:97-118 under eval/no_grad', 'includes_backbone': True},
            'cpu_baseline': {'value': 1.0 / e2e, 'unit': 'pairs/s', 'cores': threads, 'kind': 'port', 'sample': sample,
                             'host_cores': os.cpu_count(), 'hot_path_only_pairs_per_s': 1.0 / hot},
            'e2e': {'value': 1.0 / e2e, 'unit': 'pairs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    from patch2pix_b200.model import Patch2PixB200
    from patch2pix_b200.sharding import PairSharder

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise RuntimeError('bench.py (impl ours) needs a CUDA device: there is no CPU fallback')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    sharder = PairSharder(rank, world, dev)

    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    H, W, K, Wm = args.height, args.width, args.steps, args.warmup
    strong = args.pairs > 0
    if strong:
        K = (args.pairs + world - 1) // world            # steps per rank; ranks past the end of the list idle
    sd, gen = make_workload(args)
    cfg = model_config(dev, PANC_DEF)
    cfg.weights_dict = sd
    net = Patch2PixB200(cfg)
    for key, v in (('mid_passes', args.mid_passes), ('fine_passes', args.fine_passes), ('corr_passes', args.corr_passes),
                   ('seg_len', args.seg_len), ('mid_band', args.mid_band), ('fuse_gather', args.fuse_gather),
                   ('gemm_pair', args.gemm_pair), ('nc_impl', args.nc_impl)):
        if v is not None:
            net.set_option(key, v)
    opts = {k: net._handle.get_option(k) for k in ('mid_passes', 'fine_passes', 'corr_passes', 'seg_len', 'mid_band', 'fuse_gather',
                                                    'gemm_pair', 'nc_impl')}

    # pair indices: rank 0 decides, NCCL broadcasts (the "scatter pair indices" step); global pair p -> rank p % world
    total_steps = K + Wm
    n_global = args.pairs if strong else total_steps * world
    mine = sharder.scatter_pair_indices(torch.arange(n_global, dtype=torch.int64)).tolist()
    if strong:
        mine = mine[:1] * Wm + mine                       # warm-up on the first pair of the shard
    n_distinct = N_DISTINCT if not strong else min(64, max(len(set(mine)), 1))
    slot_of = {}                                           # synthetic image id -> resident pyramid slot
    imgs, feats = [], []
    with torch.no_grad():
        for p in mine:
            key = p % 64
            if key in slot_of or len(slot_of) >= n_distinct:
                continue
            slot_of[key] = len(imgs)
            a, b = gen(key, H, W)
            imgs.append((a, b))
            feats.append((net.extract.forward_all(a.to(dev), [], True), net.extract.forward_all(b.to(dev), [], True)))
    slots = [slot_of.get(p % 64, i % max(len(imgs), 1)) for i, p in enumerate(mine)]
    pinned = [(a.pin_memory(), b.pin_memory()) for a, b in imgs]
    n_patches = args.ptmax * PANC_DEF
    results = torch.zeros(max(K, 1), n_patches, 5, device=dev)
    last_anchors = torch.zeros(n_patches, 4, dtype=torch.int64, device=dev) if args.dump_outputs else None

    # Two pairs are kept in flight: the coarse stage of pair i is enqueued before the host waits for the
    # mutual-match count of pair i-1 (filter_coarse's host sync), so the GPU never idles on that sync.
    def hot_submit(i):
        f1, f2 = feats[slots[i]]
        return (i, net.submit_coarse(f1, f2, 2, True))

    step_events = [torch.cuda.Event(enable_timing=True) for _ in range(max(K, 1))]   # created before the timed region

    host_stamps = [0.0] * max(K, 1)

    def hot_finish(tk, out_slot=None, keep=None, stamp=False):
        i, ticket = tk
        np.random.seed(mine[i] % (2 ** 31))               # the reference's global numpy RNG, seeded per pair
        fine, fine_p, cm = net.finish_match(ticket, 0.0, args.ptmax)
        if out_slot is not None:
            results[out_slot, :, :4] = fine[0]
            results[out_slot, :, 4] = fine_p[0]
            if last_anchors is not None and out_slot == min(K, n_mine) - 1:
                last_anchors.copy_(cm[0])                  # the last timed step's anchors, for --dump-outputs
            if stamp:
                step_events[out_slot].record()
                host_stamps[out_slot] = time.perf_counter()
        if keep is not None and out_slot is not None and out_slot < keep.shape[0]:
            keep[out_slot].copy_(cm[0])                    # into a buffer allocated before the timed region: holding on to
                                                           # the per-step tensors makes the caching allocator cudaMalloc mid-region

    depth = max(1, args.depth)

    def hot_loop(first, steps, record, keep=None, stamp=False):
        # `depth` pairs in flight: the coarse stages of the next pairs are already queued when the host waits for the
        # mutual-match count of the oldest one, so the GPU always has more than a coarse stage of work ahead of the host
        from collections import deque
        q = deque()
        for j in range(steps):
            q.append((hot_submit(first + j), j if record else None))
            if len(q) >= depth:
                tk, slot = q.popleft()
                hot_finish(tk, slot, keep, stamp)
        while q:
            tk, slot = q.popleft()
            hot_finish(tk, slot, keep, stamp)

    def e2e_submit(i):
        a, b = pinned[slots[i]]
        f1, f2 = net.extract_pair(a, b, slot=i)    # pinned host images: H2D into the graph's input, then the backbone
        return (i, net.submit_coarse(f1, f2, 2, True))

    def e2e_finish(tk, host_out):
        i, ticket = tk
        np.random.seed(mine[i] % (2 ** 31))
        fine, fine_p, _ = net.finish_match(ticket, 0.0, args.ptmax)
        host_out[:, :4].copy_(fine[0], non_blocking=True)          # D2H read of this step's result
        host_out[:, 4].copy_(fine_p[0], non_blocking=True)

    def e2e_loop(first, steps, host_outs):
        from collections import deque
        q = deque()
        for j in range(steps):
            q.append((e2e_submit(first + j), j))
            if len(q) >= depth:
                tk, jj = q.popleft()
                e2e_finish(tk, host_outs[jj % len(host_outs)])
        while q:
            tk, jj = q.popleft()
            e2e_finish(tk, host_outs[jj % len(host_outs)])
        torch.cuda.current_stream().synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, sampler=None):
        import gc
        barrier()
        if sampler:
            sampler.start()
            time.sleep(0.01)
        gc.collect()
        gc.disable()          # a generational collection of this process's heap is a 10-40 ms host stall mid-region
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()             # ranks leave the preparations above (sampler start-up on rank 0, collection) together: a rank
        e0.record()           # that starts early only waits for the late one in the gather that closes the region
        fn(steps)
        e1.record()
        torch.cuda.synchronize()
        gc.enable()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return ms.item()

    n_mine = len(mine) - Wm                                # timed steps of this rank (strong mode: may be < K)
    with torch.no_grad():
        # ---- hot path, features resident in HBM -------------------------------------------------
        hot_loop(0, Wm, False)
        anchors_seen = torch.zeros(min(8, max(K, 1)), n_patches, 4, dtype=torch.int64, device=dev) if rank == 0 else None
        # spare cached segments in both pools of the caching allocator: no cudaMalloc (device-synchronising, and slow on a
        # shared driver) inside a timed region whatever the per-pair tensor sizes turn out to be
        spare = [torch.empty(1 << 19, dtype=torch.uint8, device=dev) for _ in range(64)] + \
                [torch.empty(16 << 20, dtype=torch.uint8, device=dev) for _ in range(8)]
        del spare
        hot_loop(0, min(Wm, K), True, anchors_seen, stamp=True)   # the recorded path itself (result stores,
        sharder.gather_results(results)                  # step events); warm-up of the collective (NCCL sets up channels lazily)
        l0 = net._handle.launch_count()
        sampler = ClockSampler(local) if rank == 0 else None

        def hot_region(steps):
            hot_loop(Wm, min(steps, n_mine), True, anchors_seen, stamp=True)
            sharder.gather_results(results)              # NCCL gather of the matches (inside the timed region)
        ms_hot = timed(hot_region, K, sampler)
        launches = net._handle.launch_count() - l0
        clocks = sampler.finish() if sampler else None
        nst = min(K, n_mine)
        if args.dump_outputs and nst > 0:
            dump_outputs(args.dump_outputs, results[nst - 1], last_anchors, rank if world > 1 else None)
        step_raw = [step_events[j].elapsed_time(step_events[j + 1]) for j in range(nst - 1)]
        step_ms = sorted(step_raw)
        worst = max(range(len(step_raw)), key=lambda j: step_raw[j]) if step_raw else None
        worst_step = None if worst is None else {'step': worst + 1, 'gpu_ms': step_raw[worst],
                                                 'host_ms': (host_stamps[worst + 1] - host_stamps[worst]) * 1e3}
        # ---- per-kernel breakdown: a SEPARATE, untimed-for-the-headline pass with an event pair around every launch
        # group (the event bookkeeping of the profiler stays out of the headline number) ----
        Kp = max(min(K, n_mine, 20), 1)
        net.set_option('profile', 1)
        net._handle.profile_read()
        net._handle.get_option('band_calls_rows_total')  # reset the running band totals
        ms_prof = timed(lambda steps: hot_loop(Wm, steps, False), Kp)
        prof = net._handle.profile_read()
        net.set_option('profile', 0)
        band_rows_total = net._handle.get_option('band_rows_total')
        mid_rows_total = net._handle.get_option('band_calls_rows_total')
        gathered = sharder.gather_results(results)       # [world, K, patches, 5]
        distinct = [int(torch.unique(a, dim=0).shape[0]) for a in anchors_seen] if anchors_seen is not None else []

        # ---- strong-scaling mode: rank 0 re-computes a sample of the other ranks' pairs, bit-equality ----------
        cross = None
        if strong and rank == 0:
            cross = {'checked_pairs': [], 'bit_equal': True}
            for r in range(1, world):
                for step in (0, K // 2):
                    p = step * world + r
                    if p >= args.pairs:
                        continue
                    a, b = gen(p % 64, H, W)
                    f1 = net.extract.forward_all(a.to(dev), [], True)
                    f2 = net.extract.forward_all(b.to(dev), [], True)
                    np.random.seed(p % (2 ** 31))
                    fine, fine_p, _ = net.match_from_feats(f1, f2, 2, ptmax=args.ptmax)
                    ok = bool(torch.equal(fine[0], gathered[r, step, :, :4]) and torch.equal(fine_p[0], gathered[r, step, :, 4]))
                    cross['checked_pairs'].append(p)
                    cross['bit_equal'] = cross['bit_equal'] and ok
            if not cross['bit_equal']:
                raise RuntimeError(f'cross-rank check failed: {cross}')

        # ---- refine-only arm: refine_matches (networks/patch2pix.py:278-318) on 3200 distinct random float matches ----
        refine_only = None
        if not strong:
            g = torch.Generator().manual_seed(99)
            rm = (torch.rand(n_patches, 4, generator=g) * torch.tensor([W, H, W, H], dtype=torch.float32)).to(dev)
            f1, f2 = feats[0]

            def refine_once():
                net._prepare_pair(f1, f2, 0)
                mid, _ = net.forward_fine_match(f1, f2, [rm], 16, 'center', net.regress_mid, _prepared=0)
                return net.forward_fine_match(f1, f2, mid, 16, 'center', net.regress_fine, _prepared=0)
            for _ in range(3):
                refine_once()
            ms_ref = timed(lambda steps: [refine_once() for _ in range(steps)], K)
            refine_only = {'ms_per_step': ms_ref / K, 'pairs_per_s': K / (ms_ref / 1e3),
                           'input': f'{n_patches} distinct uniform-random float matches, mid + fine stage'}

        # ---- end to end: pinned host images -> matches on the host ------------------------------
        # backbone in PyTorch's default cuDNN mode (TF32 convolutions allowed, as the reference would run on a GPU);
        # the fp32-backbone variant is measured beside it (parity: tests/test_gpu_parity.py::test_backbone_graph_tf32_path)
        e2e_ms = {}
        host_outs = [torch.empty(n_patches, 5).pin_memory() for _ in range(depth + 1)]
        for mode in (['fp32'] if args.backbone_fp32 else [m for m in args.e2e_modes.split(',') if m in ('tf32', 'fp16', 'fp32')]):
            if strong and mode != 'tf32' and not args.backbone_fp32:
                continue
            torch.backends.cudnn.allow_tf32 = mode != 'fp32'
            torch.backends.cudnn.benchmark = True
            net.enable_backbone_graphs(H, W, instances=depth + 1, fast=mode == 'fp16', overlap=bool(args.e2e_overlap))
            e2e_loop(0, max(min(Wm, 3), 1), host_outs)

            def e2e_region(steps):
                e2e_loop(Wm, min(steps, n_mine), host_outs)
            e2e_ms[mode] = timed(e2e_region, K)
            if mode == 'tf32' and not strong:           # the backbone share of the end-to-end step (H2D + graph replay alone)
                nb = min(K, 30)
                e2e_ms['backbone_only'] = timed(lambda steps: [net.extract_pair(*pinned[slots[i % len(slots)]], slot=i)
                                                               for i in range(steps)], nb) / nb
        torch.backends.cudnn.allow_tf32 = False

    if rank == 0:
        peaks = load_peaks()
        pairs = args.pairs if strong else K * world
        value = pairs / (ms_hot / 1e3)
        # a seconds-long region under the power cap is compared with the sustained cuBLAS peak, a short one with the burst
        sustained = ms_hot > 2000.0
        peak = peaks['tflops_sustained'] if sustained else peaks['tflops_burst']
        # dominant kernel: the conv implicit GEMMs of the refine stage
        kern = {k: {'ms_per_launch': v[0] / v[1], 'launches': v[1]} for k, v in prof.items() if v[1] > 0}
        banded = opts['mid_passes'] == 3 and opts['mid_band'] > 0
        macs = {'conv1': MAC_CONV1, 'conv2': MAC_CONV2}
        for k in list(kern):
            base, _, stage = k.partition('_')
            if base not in macs:
                continue
            # rows per launch: band launches process the band rows (running device-side total / launches)
            rows = band_rows_total / max(kern[k]['launches'], 1) if stage == 'band' else n_patches
            ps = 3 if stage == 'band' else (opts['fine_passes'] if stage == 'fine' else (1 if banded else opts['mid_passes']))
            fl = 2.0 * macs[base] * rows
            kern[k].update({'rows_per_launch': rows, 'tensor_passes': ps,
                            'algorithmic_tflops': fl / (kern[k]['ms_per_launch'] * 1e-3) / 1e12})
            kern[k]['issued_tflops'] = kern[k]['algorithmic_tflops'] * ps
        gemm_names = [k for k in kern if k.startswith('conv')]
        dom = max(gemm_names, key=lambda k: kern[k]['ms_per_launch'] * kern[k]['launches'], default=None)
        ksum = sum(v['ms_per_launch'] * v['launches'] for v in kern.values())
        roofline = None
        if dom:
            ach = kern[dom]['algorithmic_tflops']
            gemm_ms = sum(kern[k]['ms_per_launch'] * kern[k]['launches'] for k in gemm_names)
            kname = ('umma_conv1_tma_kernel' if opts['fuse_gather'] == 3 else 'umma_conv1_fused_kernel') if (dom.startswith('conv1') and not dom.endswith('band') and opts['fuse_gather'] in (1, 3)) \
                else 'umma_gemm_kernel'
            traffic = load_traffic().get(dom if kname == 'umma_gemm_kernel' else 'conv1_fused')
            roofline = {'kernel': f'{kname} ({dom})', 'bound': 'tensor', 'achieved': ach, 'peak': peak,
                        'unit': 'TFLOP/s', 'frac': ach / peak, 'traffic': traffic,
                        'traffic_unit': 'bytes of DRAM read+write per launch (ncu --set full, profiles/)',
                        'peak_source': f"{peaks['src']} cuBLAS bf16 {'sustained' if sustained else 'burst'} (fp16 runs at the same "
                                       f"tensor rate); timed region {ms_hot / 1e3:.2f} s -> {'sustained' if sustained else 'burst'} denominator",
                        'frac_vs_burst': ach / peaks['tflops_burst'], 'frac_vs_sustained': ach / peaks['tflops_sustained'],
                        'tensor_passes': kern[dom]['tensor_passes'],
                        'issued_frac': kern[dom]['issued_tflops'] / peak,
                        'share_of_step': kern[dom]['ms_per_launch'] * kern[dom]['launches'] / Kp / (ms_hot / K),
                        'all_umma_gemm_share_of_step': gemm_ms / Kp / (ms_hot / K),
                        'kernel_event_sum_ms_per_step': ksum / Kp,
                        'gap_ms_per_step': ms_hot / K - ksum / Kp if world == 1 else None,
                        'breakdown_pass': f'{Kp} steps with an event pair around every launch group, run after the timed '
                                          f'region ({ms_prof / Kp:.3f} ms/step with the event bookkeeping)',
                        'band_rows_fraction': band_rows_total / mid_rows_total if (banded and mid_rows_total) else None}
        cpu = None
        if world == 1 and not args.no_cpu_baseline and not strong:
            from oracle import p2p_oracle as O
            threads = cpu_threads()
            torch.set_num_threads(threads)
            cpu_step(O, sd, *imgs[0], args.ptmax, PANC_DEF, 16, 2)          # warm-up
            r = cpu_step(O, sd, *imgs[0], args.ptmax, PANC_DEF, args.cpu_sample_patches, None)
            cpu = {'value': 1.0 / r['hot_path_s'], 'unit': 'pairs/s', 'cores': threads, 'host_cores': os.cpu_count(),
                   'kind': 'port',
                   'sample': (f'oracle port of the reference, {threads} threads: full coarse stage of one {W}x{H} pair '
                              f'({r["coarse_s"]:.2f} s) + mid/fine refine on {r["n_sample"]} of {r["n_full"]} patches scaled to '
                              f'the full pair ({r["refine_s_extrapolated"]:.2f} s); backbone excluded ({r["backbone_s"]:.2f} s)'),
                   'with_backbone_pairs_per_s': 1.0 / r['e2e_s']}
        head = 'fp32' if args.backbone_fp32 else next(m for m in args.e2e_modes.split(',') if m in e2e_ms)
        e2e = {'value': pairs / (e2e_ms[head] / 1e3), 'unit': 'pairs/s', 'ms_per_step': e2e_ms[head] / K,
               'h2d_bytes_per_step': 2 * 3 * H * W * 4, 'd2h_bytes_per_step': n_patches * 5 * 4,
               'backbone_overlap': bool(args.e2e_overlap),
               'path': 'pinned host images -> H2D -> cuDNN ResNet34 pyramid, both images as one batch, CUDA graph ('
                       + {'fp32': 'fp32', 'tf32': 'TF32 convs, PyTorch default', 'fp16': 'fp16 channels-last'}[head] + ') -> hot path -> D2H matches+scores'}
        if 'fp32' in e2e_ms and head != 'fp32':
            e2e['fp32_backbone_value'] = pairs / (e2e_ms['fp32'] / 1e3)
        if 'fp16' in e2e_ms:
            e2e['fp16_channels_last_backbone_value'] = pairs / (e2e_ms['fp16'] / 1e3)
        if 'backbone_only' in e2e_ms:
            e2e['backbone_h2d_ms_per_pair'] = e2e_ms['backbone_only']
        line = {
            'metric': 'image-pairs/sec', 'value': value, 'unit': 'pairs/s', 'n_gpus': world, 'steps': K, 'warmup': Wm,
            'ms_per_step': ms_hot / K, 'higher_is_better': True, 'scaling': 'strong' if strong else 'weak', 'vs_baseline': None,
            'dtype': f'f16 tensor-core operands (mid: {opts["mid_passes"]}-pass hi/lo split'
                     f'{" on the risk band, 1-pass elsewhere" if opts["mid_band"] and opts["mid_passes"] == 3 else ""}, '
                     f'fine: {opts["fine_passes"]}-pass, correlation + NC conv: 3-pass), f32 accumulate',
            'data': 'synthetic',
            'config': {'workload': workload_string(W, H, args.ptmax),
                       'hot_path': 'correlation .. fine matches, features resident in HBM',
                       'sequence': 'train_patch2pix.py:97-118 under eval/no_grad', 'pairs_per_step': world,
                       'total_pairs': pairs, 'distinct_proposals_first_pairs': distinct,
                       'step_ms_quantiles': ({'p10': step_ms[len(step_ms) // 10], 'p50': step_ms[len(step_ms) // 2],
                                              'p90': step_ms[(len(step_ms) * 9) // 10], 'max': step_ms[-1],
                                              'slowest_step': worst_step} if step_ms else None),
                       'l2': f'{len(imgs)} distinct pairs cycled per rank; per-step working set (~3 GB of scratch written and '
                             f're-read) >> 126 MB L2',
                       'pipelining': f'{depth} pairs in flight per GPU (the coarse stages of the next pairs are enqueued before the host sync of the oldest)',
                       'options': opts},
            'e2e': e2e, 'gpu_launches': launches, 'roofline': roofline, 'kernels': kern, 'clocks': clocks,
            'cpu_baseline': cpu, 'refine_only': refine_only, 'cross_rank_check': cross,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    a = parse()
    if a.impl == 'reference':
        run_reference(a)
    else:
        run_ours(a)
