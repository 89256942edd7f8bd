#!/usr/bin/env python
"""bench.py -- headline benchmark of the L3C encode/decode hot path (see BASELINE.json).

  python bench.py --gpus N --steps K --warmup W                 (our sm_100a path, one process per GPU)
  python bench.py --impl reference --gpus N --steps K --warmup W (reference CPU algorithm, host cores)
  python bench.py --workload rgb_shared | crops                  (BASELINE configs 4 and 5; default: 2/3)

One "step" = one lossless round trip (encode -> decode) of one batch of synthetic images per GPU:
  l3c         16 x 3x512x512, L3C cr.cf                 (BASELINE configs[1] at N=1, configs[2] at N=8)
  rgb_shared  32 x 3x256x256, cr_rgb_shared.cf, f16x2   (configs[3])
  crops       1 x 3x3000x2000 per GPU -> 4 crops of 1500x1000 padded to 1504x1000 (configs[4], --gpus 4)
Prints ONE JSON line (rank 0).  `value` = Mpixels/s with inputs resident in HBM; `e2e` = the same
round trip through the public `Bitcoding` API from pinned host buffers (H2D of the images and the
containers, D2H of the containers and the decoded images inside the timed region).  By default the K
steps are software-pipelined (the encode of batch k+1 runs beside the latency-bound decodes of earlier
batches); the strictly sequential figures are reported beside them (`sequential`,
`e2e.sequential_value`) and `--no-pipeline` makes them the headline.  Timing: CUDA events on the stream
all work forks from and joins, barrier + synchronize on both sides, max over ranks.
`--dump-outputs DIR` also writes what the last timed step computed as DIR/<name>.npy; the inputs are seeded, so
two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# several decodes in flight = dozens of streams full of event-dependent launches: give them their own hardware
# queues (default 8: a ready kernel waits behind another decode's queued, not-yet-ready ones)
os.environ.setdefault('CUDA_DEVICE_MAX_CONNECTIONS', '32')

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'Mpixels/s encode+decode (lossless round-trip)'
# --dump-outputs: elements per array (16 MB as float32), so that a dump stays far below 64 MB
DUMP_MAX_ELEMENTS = 1 << 22

# conv FLOPs per pixel of a round trip (SURVEY.md 8d): encode forward + decoder-side re-run
WORKLOADS = {
    'l3c': dict(cfg='cr', n_img=16, H=512, W=512, precision='f16', golden='l3c_512x512',
                flop_per_px=2.230e6,
                name='L3C cr.cf (3 scales, seed-0 default init), %d x 3x512x512 uint8 noise images per GPU, '
                     'encode+decode round trip, byte-compatible .l3c containers'),
    'rgb_shared': dict(cfg='cr_rgb_shared', n_img=32, H=256, W=256, precision='f16x2', golden='rgbs_256x256',
                       flop_per_px=1.309e6, lanes=1,    # its decode is short (25 ms): more lanes only take SMs away
                       name='RGB-shared baseline cr_rgb_shared.cf (bicubic thumbnail + 1 scale), %d x 3x256x256 '
                            'uint8 noise images per GPU, encode+decode round trip'),
    'crops': dict(cfg='cr', n_img=1, H=3000, W=2000, precision='f16', golden=None, flop_per_px=2.230e6,
                  name='L3C cr.cf, adaptive-crop path: %d x 3x3000x2000 uint8 noise image per GPU -> 4 crops of '
                       '1500x1000 (auto_crop) padded to 1504x1000, coded as one batch, decoded and stitched'),
}


def make_images(first, n, h, w=None):
    import torch
    w = h if w is None else w
    out = []
    for i in range(first, first + n):
        g = torch.Generator().manual_seed(1000 + i)
        out.append((torch.rand(3, h, w, generator=g) * 255).round().to(torch.uint8))
    return torch.stack(out)


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler(object):
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '200'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for (t, line) in self.lines:
            if t < t0 or t > t1 + 0.3:
                continue
            f = [x.strip() for x in line.split(',')]
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except (ValueError, IndexError):
                continue
            for name, val in zip(['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'],
                                 f[4:8]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': mx, 'reasons': sorted(reasons),
                'samples': len(sm)}


# ------------------------------------------------------------------------------------------------
# reference arm: the reference's CPU algorithm on the host cores.  NOTHING of the product package is
# imported in this arm (nor in its worker processes): weights come from oracle/weights.py (plain torch
# module tree, same seeded default init as the reference), the algorithm from oracle/model.py.
# ------------------------------------------------------------------------------------------------
_REF = {}


def _ref_init(threads):
    import torch
    torch.set_num_threads(max(1, threads))
    torch.set_grad_enabled(False)


def _ref_roundtrip(task):
    """One lossless round trip of ONE image with the reference's CPU algorithm as restated in
    oracle/model.py (byte-identical to the unmodified reference on the golden fixtures): PyTorch fp32 CPU
    convs, PyTorch CPU CDF tables (torchac.py:174-213), the reference's coder loop.  -> (bytes, seconds)"""
    workload, seed_idx, h, w = task
    import torch
    from oracle import model as om, weights
    cfg = om.CFG_RGB_SHARED if workload == 'rgb_shared' else om.CFG_L3C
    if workload not in _REF:
        _REF[workload] = weights.default_init_state_dict(cfg)
    sd = _REF[workload]
    img = make_images(seed_idx, 1, h, w)[0]
    t0 = time.perf_counter()
    with torch.no_grad():
        data = om.encode_image(sd, cfg, img, 'torch')
        dec = om.decode_image(sd, cfg, data, 'torch')
    dt = time.perf_counter() - t0
    # (the CPU path is not bit-reproducible between its encoder-side and decoder-side network passes on every
    # host: oneDNN may choose other blockings under load.  The reference has the same property; it is reported,
    # not hidden, and does not change the amount of work that was timed.)
    return len(data), dt, bool((dec[0] == img.long()).all())


def _host_cores():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def _reference_sample(workload):
    """(h, w, description) of the bounded per-step sample of the reference arm."""
    wl = WORKLOADS[workload]
    if workload == 'crops':
        # one 1504x1000 crop needs ~15 GB of CDF temporaries per channel on the CPU path: time the same
        # algorithm on one 512x512 tile instead (its per-pixel rate is size-stable to ~2 %)
        return 512, 512, 'one 3x512x512 tile (of a 1504x1000 crop) per step'
    return wl['H'], wl['W'], 'one 3x%dx%d image of the %d-image batch per step' % (wl['H'], wl['W'], wl['n_img'])


def cpu_roundtrips(workload, n_tasks, n_warm, first_seed=0):
    """`n_tasks` independent round trips on ALL host cores: a pool of P worker processes with
    cores/P torch threads each (the CPU path is bound by its PyTorch CDF materialisation, which scales
    poorly past ~8 threads; independent images in parallel is how the reference would use a big host).
    Returns dict(value Mpx/s, seconds, cores, workers, threads, bpsp, sample)."""
    import multiprocessing as mp
    h, w, sample = _reference_sample(workload)
    cores = _host_cores()
    workers = max(1, min(8, cores // 8, n_tasks))
    threads = max(1, cores // workers)
    ctx = mp.get_context('spawn')
    # fixed thread teams in the workers: with dynamic teams (the OpenMP / MKL default under oversubscription) a conv
    # may be split differently in the encoder-side and the decoder-side pass of the same image
    os.environ.setdefault('OMP_DYNAMIC', 'FALSE')
    os.environ.setdefault('MKL_DYNAMIC', 'FALSE')
    with ctx.Pool(workers, initializer=_ref_init, initargs=(threads,)) as pool:
        if n_warm:
            pool.map(_ref_roundtrip, [(workload, first_seed + i, h, w) for i in range(n_warm)])
        t0 = time.perf_counter()
        res = pool.map(_ref_roundtrip, [(workload, first_seed + i, h, w) for i in range(n_tasks)], chunksize=1)
        dt = time.perf_counter() - t0
    px = n_tasks * h * w
    return {'value': px / 1e6 / dt, 'seconds': dt, 'cores': workers * threads, 'workers': workers,
            'threads_per_worker': threads, 'bpsp': sum(r[0] for r in res) * 8.0 / (3 * px),
            'mean_image_seconds': sum(r[1] for r in res) / n_tasks, 'sample': sample,
            'lossless': '%d of %d CPU round trips decoded bit-exactly' % (sum(1 for r in res if r[2]), n_tasks)}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return 0
    wl = WORKLOADS[args.workload]
    steps, warm = args.steps, args.warmup
    cores = _host_cores()
    workers = max(1, min(8, cores // 8, steps))
    # warm-up: every worker imports torch and runs the real sample once (at most one wave)
    r = cpu_roundtrips(args.workload, steps, min(warm, workers))
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': r['value'], 'unit': 'Mpixels/s', 'n_gpus': args.gpus,
        'steps': steps, 'warmup': warm, 'ms_per_step': 1e3 * r['seconds'] / steps, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': wl['name'] % wl['n_img'], 'bench_workload': args.workload,
                   'sample': '%s; steps run %d at a time on a pool of %d worker processes x %d torch threads '
                             '(= all %d host cores); warm-up = %d such round trip(s)'
                             % (r['sample'], r['workers'], r['workers'], r['threads_per_worker'], r['cores'],
                                min(warm, workers))},
        'cpu_baseline': {'value': r['value'], 'unit': 'Mpixels/s', 'cores': r['cores'], 'kind': 'port',
                         'sample': '%d round trip(s), %s: oracle/model.py with the reference\'s PyTorch-CPU CDF path '
                                   '(byte-identical to the unmodified reference on tests/golden), weights from '
                                   'oracle/weights.py; %.1f s per image per worker'
                                   % (steps, r['sample'], r['mean_image_seconds']),
                         'lossless': r['lossless']},
        'e2e': {'value': r['value'], 'unit': 'Mpixels/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'bpsp': r['bpsp'],
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def _profile_json(name):
    try:
        with open(os.path.join(ROOT, 'profiles', name)) as f:
            return json.load(f)
    except (OSError, ValueError):
        return None


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import l3c_pytorch_b200 as l3c
    from l3c_pytorch_b200 import auto_crop, config, dist as l3c_dist, engine as E, pad as l3c_pad

    wl = WORKLOADS[args.workload]
    precision = args.precision or wl['precision']
    rank, world, local_rank = l3c_dist.init_from_env()
    assert torch.cuda.is_available(), 'bench.py (our arm) needs a GPU; there is no CPU fallback'
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    E.set_conv_precision(precision)
    torch.manual_seed(0)
    bp = l3c.MultiscaleBlueprint(config.ms_config(wl['cfg']), device=dev).set_eval()
    bc = l3c.Bitcoding(bp)
    codec = bc.codec
    n_img = args.images_per_gpu or wl['n_img']
    n_global = n_img * world
    lo, hi = l3c_dist.shard_bounds(n_global, rank, world)
    H, W = wl['H'], wl['W']
    fac = 2 ** bp.net.config_ms.num_scales
    crops_mode = args.workload == 'crops'

    # a few distinct batches so consecutive steps do not see identical inputs; activations are ~1 GB per
    # layer at these batch sizes, far beyond the 126 MB L2
    n_sets = 2
    raw_sets = [make_images(lo + s * n_global, n_img, H, W) for s in range(n_sets)]      # [n_img,3,H,W] uint8

    def to_batch(raw):
        """host-side shape plumbing (auto_crop.py:44-75, pad.py:23-59): -> (uint8 batch, pad tuple)"""
        if not crops_mode:
            return raw, (0, 0, 0, 0)
        parts = []
        for i in range(raw.shape[0]):
            parts.extend(auto_crop.iter_crops(raw[i:i + 1]))
        pt = l3c_pad.padding_tuple(parts[0].shape[-2], parts[0].shape[-1], fac)
        return torch.nn.functional.pad(torch.cat(parts, 0), pt, 'constant').contiguous(), pt

    batches = [to_batch(r) for r in raw_sets]
    pad_tuple = batches[0][1]
    host_sets = [b.pin_memory() for (b, _) in batches]
    dev_sets = [h.to(dev) for h in host_sets]
    n_units = host_sets[0].shape[0]                      # images (or crops) per step per GPU
    Hp, Wp = host_sets[0].shape[-2:]
    px_step_global = n_global * H * W                    # unpadded pixels: what the user handed in

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def shapes_of(info):
        return [(C, h, w) for (_, C, h, w) in info['shapes']]

    TILE = {'v': tuple(args.tile) if args.tile else None}     # None: the reference's byte-compatible layout

    def step_resident(imgs):
        blob, info = codec.encode_batch(imgs, pad_tuple, to_host=False, tile=TILE['v'])
        S = codec.decode_device(blob, info['stream_offsets'], info['lens'], shapes_of(info), tile=TILE['v'])
        return S, info, blob

    tmpdir = None
    if crops_mode:
        import tempfile
        tmpdir = tempfile.mkdtemp(prefix='l3c_bench_', dir='/dev/shm' if os.path.isdir('/dev/shm') else None)

    def step_e2e(k):
        """the call a user makes.  l3c / rgb_shared: Bitcoding.encode_batch -> decode_batch from pinned host
        buffers; crops: Bitcoding.encode(img, file) -> .part0..3 -> Bitcoding.decode(file) (the reference's
        file API, auto_crop + pad + stitch inside), files on a RAM disk."""
        if crops_mode:
            outs = []
            for i in range(n_img):
                p = os.path.join(tmpdir, 'r%d_i%d.l3c' % (rank, i))
                for q in l3c.part_suffix_helper.existing_parts(p):
                    os.remove(q)
                bc.encode(raw_sets[k][i].long(), p)
                outs.append(bc.decode(p + '.part0').to(torch.uint8).cpu())
            return torch.cat(outs, 0), None
        datas, bpsps = bc.encode_batch(host_sets[k])
        dec = bc.decode_batch(datas)
        back = torch.cat(dec, 0).to(torch.uint8).cpu()        # D2H of the result
        return back, datas

    # Software pipelining over steps (the default): a decode is bound by the serial range decoder and
    # leaves most SMs idle, so the encode of the NEXT batch runs beside it, on a stream confined to the SMs
    # the decoders do not own.  K complete round trips -- including the un-overlapped first encode and last
    # decode -- lie inside the timed region.
    # args.lanes decodes are in flight at any time (each on its own set of streams; the range decoders of all
    # of them share one group of SMs), and two encodes are queued ahead on the lowest-priority stream.
    if args.lanes is None:
        args.lanes = int(os.environ.get('L3C_BENCH_LANES', wl.get('lanes', 4)))
    n_lanes = max(1, args.lanes)
    lanes, side_stream = codec.lanes(dev, 3 * n_units, n_lanes)[:2] if args.pipeline else (None, None)
    enc_streams = codec.encode_streams(dev, 3 * n_units, n_lanes) if args.pipeline else None
    ENC_DEPTH = int(os.environ.get('L3C_BENCH_ENC_DEPTH', len(enc_streams) if enc_streams else 2))

    def run_resident(steps, first_set=0):
        if not args.pipeline:
            for s in range(steps):
                S, info, blob = step_resident(dev_sets[(first_set + s) % n_sets])
            return S, info, blob
        dbg = os.environ.get('L3C_BENCH_DEBUG')
        cur = torch.cuda.current_stream()
        for es in enc_streams:
            es.wait_stream(cur)                   # the timing events live on `cur`: fork from it ...
        for ln in lanes:
            ln.main.wait_stream(cur)
        jobs = {}
        tl = [] if dbg else None                      # timeline events (L3C_BENCH_DEBUG): where does a step go?

        def tick(stream):
            e = torch.cuda.Event(enable_timing=True)
            e.record(stream)
            return e

        def begin(i):
            if i < steps:
                es = enc_streams[i % len(enc_streams)]     # alternate: the latency-bound range-encoder launch of
                with torch.cuda.stream(es):                # batch i overlaps the convs of batch i+1
                    a = tick(es) if dbg else None
                    jobs[i] = codec.encode_begin(dev_sets[(first_set + i) % n_sets], pad_tuple, tile=TILE['v'])
                    if dbg:
                        tl.append(('enc', i, a, tick(es)))

        t_origin = tick(cur) if dbg else None
        only = os.environ.get('L3C_BENCH_ONLY')       # diagnosis: 'enc' / 'dec' = only that half of every step
        if only == 'dec':
            begin(0)
            blob0, info0 = jobs.pop(0).finish(to_host=False)
        else:
            for i in range(ENC_DEPTH):
                begin(i)
        for s in range(steps):
            t0 = time.perf_counter()
            if only == 'dec':
                blob, info = blob0, info0
            else:
                blob, info = jobs.pop(s).finish(to_host=False)
            t1 = time.perf_counter()
            if only != 'dec':
                begin(s + ENC_DEPTH)
            t2 = time.perf_counter()
            if only == 'enc':
                S = None
                continue
            ln = lanes[s % n_lanes]
            with torch.cuda.stream(ln.main):
                ln.main.wait_event(info['ready'])
                blob.record_stream(ln.main)
                a = tick(ln.main) if dbg else None
                if dbg:
                    codec.stage_events = []
                S = codec.decode_device(blob, info['stream_offsets'], info['lens'], shapes_of(info), lane=ln,
                                        tile=TILE['v'])
                if dbg:
                    tl.append(('dec', s, a, tick(ln.main), codec.stage_events))
                    codec.stage_events = None
            if dbg:
                print('pipelined step %d: finish %.1f ms, begin(next) %.1f ms, decode issue %.1f ms'
                      % (s, 1e3 * (t1 - t0), 1e3 * (t2 - t1), 1e3 * (time.perf_counter() - t2)), file=sys.stderr)
        for ln in lanes:
            cur.wait_stream(ln.main)              # ... and join it again
        for es in enc_streams:
            cur.wait_stream(es)
        if dbg:
            torch.cuda.synchronize()
            for rec in sorted(tl, key=lambda r: (r[1], r[0] == 'dec')):
                kind, i, a, b = rec[:4]
                line = '  %s %2d: start %7.1f  end %7.1f  (%.1f ms)' % (kind, i, t_origin.elapsed_time(a),
                                                                        t_origin.elapsed_time(b), a.elapsed_time(b))
                if kind == 'dec':
                    evs = rec[4]
                    line += '  stages: ' + ' '.join('%s=%.1f' % (n2, e1.elapsed_time(e2))
                                                     for (_, e1), (n2, e2) in zip(evs[:-1], evs[1:]))
                print(line, file=sys.stderr)
        return S, info, blob

    def run_e2e(steps, first_set=0):
        if not args.pipeline or crops_mode:
            for s in range(steps):
                back, datas = step_e2e((first_set + s) % n_sets)
            return back, datas
        cur = torch.cuda.current_stream()
        for es in enc_streams:
            es.wait_stream(cur)
        for ln in lanes:
            ln.main.wait_stream(cur)
        jobs = {}

        def begin(i):
            if i < steps:
                jobs[i] = bc.encode_batch_begin(host_sets[(first_set + i) % n_sets],
                                                stream=enc_streams[i % len(enc_streams)])

        for i in range(ENC_DEPTH):
            begin(i)
        # the decoded images come back through pinned buffers; the read-back of step s is awaited after
        # n_lanes more steps have been issued, so the host prepares the next decodes while this one runs
        bufs = [torch.empty_like(host_sets[0]).pin_memory() for _ in range(n_lanes + 1)]
        pending = []
        for s in range(steps):
            datas, _ = jobs.pop(s).finish()
            begin(s + ENC_DEPTH)
            ln = lanes[s % n_lanes]
            with torch.cuda.stream(ln.main):
                dec = bc.decode_batch(datas, lane=ln)          # containers -> GPU -> images (asynchronous)
                bufs[s % (n_lanes + 1)].copy_(torch.cat(dec, 0).to(torch.uint8), non_blocking=True)    # D2H of the result
                ev = torch.cuda.Event()
                ev.record(ln.main)
            pending.append(ev)
            if len(pending) > n_lanes:
                pending.pop(0).synchronize()
        for ev in pending:
            ev.synchronize()
        back = bufs[(steps - 1) % (n_lanes + 1)]
        for ln in lanes:
            cur.wait_stream(ln.main)
        for es in enc_streams:
            cur.wait_stream(es)
        return back, datas

    def check_lossless(S, k, what):
        if os.environ.get('L3C_BENCH_ONLY'):      # diagnosis runs time half a step: nothing to compare
            return
        assert torch.equal(S, dev_sets[k]), what + ': round trip is not lossless'
        if crops_mode:       # undo the padding, stitch the crops back (auto_crop.py:109-136): the user's image
            per = n_units // n_img
            for i in range(n_img):
                parts = [l3c_pad.undo_pad(S[i * per + j:i * per + j + 1], *pad_tuple) for j in range(per)]
                assert torch.equal(auto_crop.stitch(parts)[0].cpu(), raw_sets[k][i]), what + ': stitched image differs'

    def dump_outputs(out_dir, S, info, blob):
        """What the last timed step handed its caller, as out_dir/<name>.npy: the decoded images, the coded
        bytes of every stream (container order, concatenated), the container sizes and the stream lengths.
        An array of more than DUMP_MAX_ELEMENTS elements is cut to a fixed, seeded sample of its elements."""
        def sample(n):
            if n <= DUMP_MAX_ELEMENTS:
                return np.arange(n, dtype=np.int64)
            return np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_ELEMENTS, replace=False))

        lens = np.asarray(info['lens'], np.int64).reshape(-1)
        ends = np.cumsum(lens)
        pos = sample(int(ends[-1]))                       # positions in the concatenated streams
        j = np.searchsorted(ends, pos, side='right')
        at = np.asarray(info['stream_offsets'], np.int64).reshape(-1)[j] + pos - (ends[j] - lens[j])
        arrays = {'decoded': S.reshape(-1)[torch.from_numpy(sample(S.numel())).to(dev)],
                  'streams': blob[torch.from_numpy(at).to(dev)]}
        arrays = {k: v.cpu().numpy().astype(np.float32) for k, v in arrays.items()}
        arrays['container_bytes'] = np.asarray(info['sizes'], np.float64)
        arrays['stream_lens'] = np.asarray(info['lens'], np.float64)
        os.makedirs(out_dir, exist_ok=True)
        for name, a in arrays.items():
            np.save(os.path.join(out_dir, name + '.npy'), a)

    # ---- warm-up + correctness (outside the timed region)
    for w in range(max(args.warmup, 1)):
        S, info, _ = step_resident(dev_sets[w % n_sets])
    check_lossless(S, (max(args.warmup, 1) - 1) % n_sets, 'warm-up')
    if args.pipeline:                      # every lane / encode stream has its own allocator pool: warm them all up
        n_warm = max(args.warmup, n_lanes + 1)     # (a first use inside the timed region costs a 300 ms cudaMalloc stall)
        S, info, _ = run_resident(n_warm)
        check_lossless(S, (n_warm - 1) % n_sets, 'pipelined warm-up')
    sizes = info['sizes']
    counts = l3c_dist.gather_byte_counts(sizes, n_global * (n_units // n_img), rank, world)   # the one collective
    bpsp = l3c_dist.global_bpsp(counts, 3 * Hp * Wp)
    # parity with the reference's own torchac path on the same weights / images: EVERY image of rank 0's
    # batch against the container size the unmodified reference writes for it (tests/golden/batch_bytes.json)
    parity = None
    if wl['golden'] and rank == 0:
        try:
            with open(os.path.join(ROOT, 'tests', 'golden', 'batch_bytes.json')) as f:
                gold = json.load(f)[wl['golden']]
            _, info0 = codec.encode_batch(dev_sets[0], pad_tuple, to_host=False)
            n_cmp = min(n_units, len(gold))
            ours = [int(x) for x in info0['sizes'][:n_cmp]]
            ref = [g['ref_bytes'] for g in gold[:n_cmp]]
            d = [(a - b) * 8.0 / (3.0 * H * W) for a, b in zip(ours, ref)]
            parity = {'images': 'seeds 1000..%d, 3x%dx%d (all %d of rank 0\'s batch)' % (999 + n_cmp, H, W, n_cmp),
                      'reference': 'unmodified reference Bitcoding.encode on the CPU (oracle/gen_golden_batch.py)',
                      'mean_dbpsp': sum(d) / n_cmp, 'mean_abs_dbpsp': sum(abs(x) for x in d) / n_cmp,
                      'max_abs_dbpsp': max(abs(x) for x in d), 'bytes_minus_reference': [a - b for a, b in zip(ours, ref)],
                      'bytes': ours[0], 'reference_bytes': ref[0], 'abs_dbpsp': abs(d[0])}
        except (OSError, KeyError):
            pass

    # ---- timed: device-resident
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    barrier()
    t_wall0 = time.time()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    launches0 = E.LAUNCHES['n']
    S, info, blob = run_resident(args.steps)
    launches_timed = E.LAUNCHES['n'] - launches0
    e1.record()
    barrier()
    t_wall1 = time.time()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    clocks = sampler.stop(t_wall0, t_wall1)
    ms_total = float(ms)
    value = px_step_global * args.steps / 1e6 / (ms_total / 1e3)
    check_lossless(S, (args.steps - 1) % n_sets, 'timed run')
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, S, info, blob)

    def timed_sequential(fn):
        """the same K steps strictly one after the other (reported beside the pipelined numbers)"""
        barrier()
        tw = time.perf_counter()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for s in range(args.steps):
            fn(s % n_sets)
        b.record()
        barrier()
        t = torch.tensor([max(a.elapsed_time(b), 0.0), (time.perf_counter() - tw) * 1e3], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1])

    if args.value_only:                       # tuning sweeps: the device-resident figure only
        if rank == 0:
            print(json.dumps({'metric': METRIC, 'value': value, 'unit': 'Mpixels/s', 'ms_per_step': ms_total / args.steps,
                              'steps': args.steps, 'lanes': args.lanes, 'precision': precision, 'value_only': True,
                              'env': {k: v for k, v in os.environ.items() if k.startswith('L3C_')}}))
        if world > 1:
            dist.destroy_process_group()
        return 0

    seq_value = seq_e2e = None
    if args.pipeline:
        seq_ms, _ = timed_sequential(lambda i: step_resident(dev_sets[i]))
        seq_value = px_step_global * args.steps / 1e6 / (seq_ms / 1e3)

    # ---- the throughput (tiled-stream) layout beside it: same symbols, every channel plane cut into 64x64 tiles
    #      coded as independent streams (codec.ContainerLayout) -- not byte-compatible with the reference, a few
    #      bytes per tile larger; never the headline
    tiled = None
    if not crops_mode and TILE['v'] is None and not args.no_tiled:
        TILE['v'] = (64, 64)
        try:
            S, info_t, _ = step_resident(dev_sets[0])
            check_lossless(S, 0, 'tiled')
            t_seq, _ = timed_sequential(lambda i: step_resident(dev_sets[i]))
            t_pipe = None
            if args.pipeline:
                run_resident(n_lanes + 1)
                barrier()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                S, _, _ = run_resident(args.steps)
                b.record()
                barrier()
                t_pipe = a.elapsed_time(b)
                check_lossless(S, (args.steps - 1) % n_sets, 'tiled pipelined')
            bpsp_t = sum(int(x) for x in info_t['sizes']) * 8.0 / (n_units * 3 * Hp * Wp)
            bpsp_c = sum(int(x) for x in sizes) * 8.0 / (n_units * 3 * Hp * Wp)
            tiled = {'tile': [64, 64], 'streams_per_image': int(info_t['lens'].shape[1]),
                     'sequential_value': px_step_global / world * args.steps / 1e6 / (t_seq / 1e3),
                     'value': (px_step_global / world * args.steps / 1e6 / (t_pipe / 1e3)) if t_pipe else None,
                     'bpsp': bpsp_t, 'bpsp_minus_compat': bpsp_t - bpsp_c, 'unit': 'Mpixels/s (this rank)',
                     'note': 'not readable by the reference; lossless; same symbols and CDFs as the compat layout'}
        finally:
            TILE['v'] = None

    # ---- timed: end to end through the public API (host buffers, copies inside)
    back, datas = step_e2e(0)
    assert torch.equal(back, raw_sets[0] if crops_mode else host_sets[0]), 'e2e round trip is not lossless'
    if args.pipeline:
        run_e2e(n_lanes + 1)
    barrier()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    if os.environ.get('L3C_BENCH_PROFILE'):           # where does the host thread spend an e2e step?
        import cProfile
        import pstats
        prof = cProfile.Profile()
        back, datas = prof.runcall(run_e2e, args.steps)
        pstats.Stats(prof, stream=sys.stderr).sort_stats('cumulative').print_stats(35)
    else:
        back, datas = run_e2e(args.steps)
    e1.record()
    barrier()
    wall = time.perf_counter() - t0
    ms2 = torch.tensor([max(e0.elapsed_time(e1), wall * 1e3)], device=dev)
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    e2e_value = px_step_global * args.steps / 1e6 / (float(ms2) / 1e3)
    last = (args.steps - 1) % n_sets
    assert torch.equal(back, raw_sets[last] if crops_mode else host_sets[last]), 'timed e2e round trip is not lossless'
    if args.pipeline and not crops_mode:
        seq_ev, seq_wall = timed_sequential(step_e2e)
        seq_e2e = px_step_global * args.steps / 1e6 / (max(seq_ev, seq_wall) / 1e3)
    cont_bytes = sum(int(x) for x in sizes)
    img_bytes = n_img * 3 * H * W

    # ---- roofline of the FLOP-dominant kernel: the 3x3 64->64 convolution at 16 x 256 x 256 (34 of the
    #      ~120 conv launches of an L3C round trip and ~60 % of its FLOPs run on exactly this shape)
    peaks = {}
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            peaks = json.load(f)
    except OSError:
        pass
    peak_tf = peaks.get('bf16_tflops', 1590.0)
    peak_tf_sus = peaks.get('bf16_tflops_sustained', 1400.0)
    hbm_gbs = peaks.get('hbm_gbs', 6650.0)
    # The dominant conv kernel (conv_f16_kernel<0>: 102 of the ~125 conv launches of an L3C round trip and
    # ~85 % of its FLOPs) on its dominant shape, 16 x 256 x 256 x 64 -> 64, as the two launches of one ResBlock
    # (edsr.py:63-89): conv + ReLU writing only the FP16 operand image, then conv + fp32 residual writing fp32 +
    # operand image.  With FP16 operands and layer-granular fp32 activations the layer is HBM-bound on a B200
    # (73.7 kFLOP per 256 / 768 algorithmic bytes per pixel vs a ridge of ~260 FLOP/B): the roofline is
    # algorithmic bytes / time against the measured copy bandwidth; the tensor-pipe view is reported beside it.
    roof_prec = precision if precision in ('f16', 'tf32') else 'f16'
    E.set_conv_precision(roof_prec)
    blk = bp.net.nets[0].dec.body[0].body
    conv1, conv2 = blk[0], blk[2]
    cn = 16
    x = torch.randn(cn, 256, 256, 64, device=dev)
    res = torch.randn(cn, 256, 256, 64, device=dev)
    xa = E.as_operand(x)                              # Act carrying the operand image the tensor cores read
    reps = 10
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def time_launches(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        c0.record()
        for _ in range(reps):
            fn()
        c1.record()
        torch.cuda.synchronize()
        return c0.elapsed_time(c1) / reps

    mid = E.conv2d(conv1, xa, relu=True, want='round')
    ms1 = time_launches(lambda: E.conv2d(conv1, xa, relu=True, want='round'))
    ms2 = time_launches(lambda: E.conv2d(conv2, mid, residual=res, want='act'))
    op_b = 2 if roof_prec == 'f16' else 4             # bytes per element of the operand image
    px = cn * 256 * 256
    bytes1 = px * (64 * op_b + 64 * op_b)             # operand image in, operand image out
    bytes2 = px * (64 * op_b + 256 + 256 + 64 * op_b)   # operand image + fp32 residual in, fp32 + operand image out
    conv_flops = 2.0 * 9 * 64 * 64 * px               # per launch
    conv_ms = 0.5 * (ms1 + ms2)
    # the library conv the reference would run on this GPU (cuDNN through torch, channels_last), same shape:
    # a comparator, not part of the product path
    cudnn = {}
    try:
        if args.no_comparators:
            raise RuntimeError('skipped (--no-comparators)')
        xc = x.permute(0, 3, 1, 2)                    # NCHW view of the NHWC buffer = channels_last
        wc = conv1.weight.detach().contiguous(memory_format=torch.channels_last)
        for name, allow in (('tf32', True), ('fp32', False)):
            old = torch.backends.cudnn.allow_tf32
            torch.backends.cudnn.allow_tf32 = allow
            torch.backends.cudnn.benchmark = True
            try:
                cudnn[name + '_ms'] = time_launches(lambda: torch.nn.functional.conv2d(xc, wc, conv1.bias, padding=1))
                cudnn[name + '_tflops'] = conv_flops / (cudnn[name + '_ms'] / 1e3) / 1e12
            finally:
                torch.backends.cudnn.allow_tf32 = old
        xh, wh = xc.half(), wc.half()
        cudnn['fp16_ms'] = time_launches(lambda: torch.nn.functional.conv2d(xh, wh, conv1.bias.half(), padding=1))
        cudnn['fp16_tflops'] = conv_flops / (cudnn['fp16_ms'] / 1e3) / 1e12
        del xh, wh
    except RuntimeError as ex:                        # never let the comparator break the bench
        cudnn['error'] = str(ex)[:200]
    E.set_conv_precision(precision)
    achieved_tf = 2 * conv_flops / ((ms1 + ms2) / 1e3) / 1e12
    achieved_gbs = (bytes1 + bytes2) / ((ms1 + ms2) / 1e3) / 1e9
    step_tf = wl['flop_per_px'] * n_units * Hp * Wp * args.steps / (ms_total / 1e3) / 1e12
    traffic = _profile_json('conv3x3_traffic.json') or {}
    tr = traffic.get(roof_prec, {})
    roofline = {'bound': 'hbm', 'achieved': achieved_gbs, 'peak': hbm_gbs, 'unit': 'GB/s',
                'frac': achieved_gbs / hbm_gbs,
                # dram__bytes_read.sum + dram__bytes_write.sum of the two launches on THIS shape, parsed from the
                # `ncu --set full` capture summarised in profiles/conv3x3_traffic.json (records the commit)
                'traffic': tr.get('dram_bytes'), 'traffic_source': tr.get('source'),
                'algorithmic_bytes': bytes1 + bytes2,
                'kernel': 'conv3x3 64->64 (%s operands, fp32 accumulate), 16x256x256 NHWC, the two launches of one '
                          'ResBlock: conv+ReLU -> operand image only; conv + fp32 residual -> fp32 + operand image'
                          % roof_prec,
                'launches': {'conv_relu_operand_only': {'ms': ms1, 'GBps': bytes1 / (ms1 / 1e3) / 1e9,
                                                        'TFLOPs': conv_flops / (ms1 / 1e3) / 1e12},
                             'conv_residual_fp32_and_operand': {'ms': ms2, 'GBps': bytes2 / (ms2 / 1e3) / 1e9,
                                                                'TFLOPs': conv_flops / (ms2 / 1e3) / 1e12}},
                'ms': conv_ms,
                'peak_source': 'MEASURED_PEAKS.json hbm_gbs (copy bandwidth)' if peaks else 'fallback 6650 GB/s',
                'tensor': {'achieved': achieved_tf, 'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': achieved_tf / peak_tf,
                           'peak_source': 'MEASURED_PEAKS.json bf16 burst' if peaks else 'fallback 1.59 PFLOP/s'},
                'cudnn_same_shape': cudnn,
                # SURVEY 8(d): conv FLOPs of the whole round trip / step time, against the burst and the sustained peak
                'whole_round_trip': {'achieved': step_tf, 'frac_burst': step_tf / peak_tf,
                                     'frac_sustained': step_tf / peak_tf_sus,
                                     'flop_per_px': wl['flop_per_px']}}
    del x, res, xa, mid

    # ---- where the step goes (one extra, untimed-for-the-metric round trip with CUDA events): the dominant
    #      kernel by TIME is the serial range decoder, which is latency-bound (one warp per stream, a fixed
    #      number of ns per symbol whatever the number of streams), not HBM- or tensor-bound
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    bp.net(dev_sets[0])                                # untimed: the allocator re-grows its pools after the comparators
    torch.cuda.synchronize()
    ev[0].record()
    out_net = bp.net(dev_sets[0])
    ev[1].record()
    blob, info = codec.encode_batch(dev_sets[0], pad_tuple, out=out_net, to_host=False)
    ev[2].record()
    codec.stage_events = []
    codec.decode_device(blob, info['stream_offsets'], info['lens'], shapes_of(info))
    ev[3].record()
    torch.cuda.synchronize()
    n_sym_rgb = Hp * Wp
    dec_ms = ev[2].elapsed_time(ev[3])
    stages = codec.stage_ms()
    rgb_ms = stages.get('rgb')
    breakdown = {'forward_ms': ev[0].elapsed_time(ev[1]), 'entropy_encode_ms': ev[1].elapsed_time(ev[2]),
                 'decode_ms': dec_ms, 'decode_stage_ms': stages,
                 'serial_symbols_per_stream': {'rgb': n_sym_rgb},
                 'streams_in_flight': n_units * sum(C for (C, _, _) in shapes_of(info))}
    # decoder roofline: algorithmic bytes per RGB symbol = 480 B parameters /3 + 1 B symbol + ~2 B code; the
    # chain floor is the dependent-issue latency of one warp (DESIGN.md 4.4), not bandwidth
    if rgb_ms:
        ns_sym = rgb_ms * 1e6 / n_sym_rgb
        alg_bytes = n_units * n_sym_rgb * (480.0 + 3.0 + 3 * 2.3)
        roofline['decoder'] = {'kernel': 'RGB range decoder (one warp per stream, %d streams)' % (3 * n_units),
                               'ns_per_symbol': ns_sym, 'dependency_chain_floor_ns': 130 / 1.965,
                               'algorithmic_GBps': alg_bytes / (rgb_ms / 1e3) / 1e9,
                               'frac_of_hbm': alg_bytes / (rgb_ms / 1e3) / 1e9 / hbm_gbs, 'hbm_peak_GBps': hbm_gbs}

    # ---- CPU baseline beside it (rank 0, N=1 only, bounded sample)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = cpu_roundtrips(args.workload, max(1, min(8, _host_cores() // 8)), 0)
        cpu = {'value': r['value'], 'unit': 'Mpixels/s', 'cores': r['cores'], 'kind': 'port',
               'sample': '%d concurrent round trip(s) (%d worker processes x %d torch threads), %s (%.1f s wall): '
                         'oracle/model.py with the reference\'s PyTorch-CPU CDF path (byte-identical to the unmodified '
                         'reference on tests/golden)' % (r['workers'], r['workers'], r['threads_per_worker'],
                                                        r['sample'], r['seconds']),
               'bpsp': r['bpsp'], 'lossless': r['lossless']}

    if rank == 0:
        line = {
            'metric': METRIC, 'value': value, 'unit': 'Mpixels/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms_total / args.steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None,
            'dtype': {'f16': 'f16', 'tf32': 'tf32', 'fp32': 'f32', 'f16x2': 'f16x2'}[precision], 'data': 'synthetic',
            'config': {'workload': wl['name'] % n_img, 'bench_workload': args.workload,
                       'global_batch': n_global, 'parallelism': 'images sharded over %d GPU(s), no data-path '
                                                                'collective' % world,
                       'conv_precision': precision + {'f16': ': FP16 operand images (RN), fp32 accumulation in TMEM, fp32 '
                                                             'residual stream and DMLL parameters; integer range coder',
                                                      'tf32': ': TF32-RN operands, fp32 accumulation',
                                                      'f16x2': ': split-FP16 operands (hi + lo/2^11, 22 bits), three '
                                                               'tcgen05.mma per K step, fp32 accumulation (strict mode)',
                                                      'fp32': ': CUDA-core fp32'}[precision],
                       'pipelining': ('%d decodes in flight (range decoders of all of them on one SM partition) beside '
                                      'the encodes of the next batches; all %d round trips, incl. the un-overlapped '
                                      'first encode and last decodes, are inside the timed region; "sequential" = '
                                      'the same steps one after the other'
                                      % (n_lanes, args.steps)) if args.pipeline else 'none (sequential steps)',
                       'l2': 'working set >> L2 (>= 1 GB of activations per layer), inputs alternate between batches'},
            'bpsp': bpsp, 'bpsp_parity': parity,
            'e2e': {'value': e2e_value, 'unit': 'Mpixels/s', 'h2d_bytes_per_step': img_bytes + cont_bytes,
                    'd2h_bytes_per_step': cont_bytes + img_bytes, 'sequential_value': seq_e2e,
                    'api': 'Bitcoding.encode(file)/decode(file), files on a RAM disk' if crops_mode else
                           'Bitcoding.encode_batch_begin/finish -> decode_batch, pinned host buffers'},
            'sequential': {'value': seq_value, 'unit': 'Mpixels/s'},
            # kernels of libl3c_b200.so launched inside the timed (device-resident) region, counted at the
            # C-ABI call sites (engine.LAUNCHES)
            'gpu_launches': launches_timed,
            'clocks': clocks,
            'roofline': roofline,
            'breakdown': breakdown,
            'tiled': tiled,
            'cpu_baseline': cpu,
        }
        print(json.dumps(line))
    if tmpdir:
        import shutil
        shutil.rmtree(tmpdir, ignore_errors=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='l3c', choices=sorted(WORKLOADS),
                    help='l3c = BASELINE configs 2/3 (default), rgb_shared = config 4, crops = config 5')
    ap.add_argument('--precision', default=os.environ.get('L3C_CONV_PRECISION'),
                    choices=['fp32', 'tf32', 'f16', 'f16x2'],
                    help='conv mode (default: f16 = FP16-operand tensor cores for l3c/crops, f16x2 = split-FP16 strict mode for rgb_shared)')
    ap.add_argument('--images-per-gpu', type=int, default=None)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--value-only', action='store_true', help='tuning: print the device-resident value and stop')
    ap.add_argument('--tile', type=int, nargs=2, default=None, metavar=('TH', 'TW'),
                    help='run the whole bench on TILED containers (throughput layout, not reference-compatible)')
    ap.add_argument('--no-tiled', action='store_true', help='skip the extra tiled-layout measurement')
    ap.add_argument('--no-comparators', action='store_true',
                    help='skip the cuDNN timings of the roofline shape (their autotuning floods a profiler capture)')
    ap.add_argument('--lanes', type=int, default=None,
                    help='decodes in flight in the pipelined mode (default: 4; rgb_shared: 1)')
    ap.add_argument('--no-pipeline', dest='pipeline', action='store_false',
                    help='strictly sequential steps: encode(k), decode(k), encode(k+1), ...')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step computed (rank 0) as DIR/<name>.npy, float32/float64, '
                         'to compare two builds output for output')
    args = ap.parse_args()
    if args.impl == 'reference':
        return run_reference(args)
    return run_ours(args)


if __name__ == '__main__':
    sys.exit(main())
