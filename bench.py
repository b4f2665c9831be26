#!/usr/bin/env python
"""Benchmark of the C2-Matching restoration-forward hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    (N > 1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...)

--dump-outputs DIR writes what the timed path returned in its last timed step as DIR/<name>.npy (float32):
`sr` = the SR batch of the device-resident forward (`value`), `e2e_sr` = the host SR batch of the end-to-end
call (`e2e`), 19.7 MB each; rank 0's batch when N > 1; with --impl reference, `sr` of its one-image step.
Inputs and weights are seeded, so two builds run with the same arguments can be compared output for output.

Metric (BASELINE.json): SR images/s, LR 160x160 -> 640x640 with a 500x500 Ref (zero-padded to
640x640, as the reference dataset does).  A step = one full forward (extractor -> correlation /
index_map -> offsets -> restoration net with 3 fused DCNs) over a batch of 4 synthetic pairs per
GPU (BASELINE config 2), random-init weights of the real architecture.  Weak scaling: each rank
processes its own batch, no data-path collective; `value` = images of all ranks / max-over-ranks
time.

One JSON line on rank 0 (see the task contract): value (inputs resident in HBM; timed with the library's
profiling hook OFF), e2e (host pinned inputs -> H2D -> forward -> D2H of the SR images, through the public
RestorationPipeline.run_host call), roofline of the dominant kernel class (per-launch CUDA events recorded by
the library on the launching stream in a SEPARATE pass), cpu_baseline (the oracle port of the reference's CPU
path on this box's physical host cores, bounded sample), parity (image 0 of the timed batch: GPU pipeline vs
that same oracle run), micro (BASELINE configs 3 and 4), clocks, gpu_launches.
"""
import argparse
import atexit
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, 'c2-matching_b200'), os.path.join(ROOT, 'tests', 'golden')):
    if p not in sys.path:
        sys.path.insert(0, p)

# random-init (seeded) weights of the real architecture: no ImageNet VGG checkpoint exists on the box
os.environ.setdefault('C2M_VGG_PRETRAINED', '0')

import torch  # noqa: E402

LR, REF, BATCH, CH = 160, 500, 4, 256
WORKLOAD = 'config2: LR 160x160 -> SR 640x640, Ref 500x500 zero-padded to 640x640, batch 4 per GPU'


# ------------------------------------------------------------------------------- helpers
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region: one background `nvidia-smi -lms`
    process (a fresh nvidia-smi per sample takes ~0.5 s on these hosts and misses short runs)."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-i',
                                          str(self.index), '-lms', '100'], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.kill)      # no sampler left running if the benchmark fails before stop()
        except Exception:
            self.proc = None

    def stop(self):
        rows = []
        if self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()
            try:
                out, _ = self.proc.communicate(timeout=5)
            except Exception:
                self.proc.kill()
                out = ''
            rows = [[c.strip() for c in ln.split(',')] for ln in out.splitlines() if ln.strip()]
        num = lambda v: v.replace('.', '', 1).isdigit()
        # keep samples taken under load (power well above idle) when there are any
        sm = [float(r[0]) for r in rows if len(r) >= 7 and num(r[0])]
        mx = [float(r[1]) for r in rows if len(r) >= 7 and num(r[1])]
        pw = [float(r[2]) for r in rows if len(r) >= 7 and num(r[2])]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({n for r in rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith('active')})
        return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'power_w_max': max(pw) if pw else None, 'reasons': reasons, 'samples': len(rows)}


def seeded_weights():
    import seeding
    return (seeding.share_extractor_weights(seeding.seeded_state_dict(seeding.spec_extractor(), 11)),
            seeding.seeded_state_dict(seeding.spec_net_map(), 12),
            seeding.seeded_state_dict(seeding.spec_restoration_net(), 13))


def corr_algorithmic(batch):
    """SURVEY.md §8(d): per image FLOPs = 2*C*p^2*N_in*N_ref, bytes = 4*C*(HW_in+HW_ref) + 12*N_in."""
    n = (LR - 2) ** 2
    flops = 2.0 * CH * 9 * n * n * batch
    byts = (4.0 * CH * (LR * LR * 2) + 12.0 * n) * batch
    return flops, byts


def host_cores():
    """(physical, logical) core counts of this host; the CPU legs run on the physical ones (SURVEY §8d)."""
    logical = os.cpu_count() or 1
    try:
        import psutil
        physical = psutil.cpu_count(logical=False) or logical
    except Exception:
        physical = logical
    return physical, logical


def cpu_baseline(pair, timed_runs=3, b4_budget_s=120.0):
    """The reference's CPU path (oracle port, kind "port": the reference is Python and /root/reference does not
    exist on the GPU box) on a bounded sample of the SAME workload: image 0 of rank 0's timed batch, 1 warm-up +
    `timed_runs` runs at batch 1 (the reference's own validation batch size), and one batch-4 run when it fits
    the time budget.  Returns (record, (sr, idx) of the oracle on that image) — the latter feeds `parity`."""
    from oracle import ref_path
    physical, logical = host_cores()
    torch.set_num_threads(physical)
    sds = seeded_weights()
    one = [t[:1] for t in pair]
    t0 = time.perf_counter()
    want = ref_path.full_forward(*sds, *one, return_idx=True)          # warm-up run; its result is the parity oracle
    warm = time.perf_counter() - t0
    runs = []
    for _ in range(timed_runs):
        t0 = time.perf_counter()
        ref_path.full_forward(*sds, *one)
        runs.append(time.perf_counter() - t0)
    mean = sum(runs) / len(runs)
    rec = {'value': 1.0 / mean, 'unit': 'images/s', 'cores': physical, 'logical_cores': logical, 'kind': 'port',
           'runs_s': [round(r, 2) for r in runs], 'warmup_s': round(warm, 2),
           'sample': f'image 0 of the timed batch, full forward at batch 1, {timed_runs} timed runs after 1 warm-up, fp32 '
                     f'torch-CPU oracle port (oracle/ref_path.py), {physical} threads = physical cores'}
    if pair[0].shape[0] >= 4 and 4 * mean <= b4_budget_s:
        four = [t[:4] for t in pair]
        t0 = time.perf_counter()
        ref_path.full_forward(*sds, *four)
        dt = time.perf_counter() - t0
        rec['batch4'] = {'value': 4.0 / dt, 'unit': 'images/s', 'runs_s': [round(dt, 2)]}
    return rec, want


def dump_outputs(out_dir, arrays):
    """{name: tensor} -> out_dir/<name>.npy in float32 (see --dump-outputs)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + '.npy'), v.detach().float().cpu().numpy())


# ------------------------------------------------------------------------------- reference arm
def run_reference(args, rank):
    if rank != 0:
        return
    from c2m_b200.pipeline import synthetic_pair
    from oracle import ref_path
    threads, logical = host_cores()
    torch.set_num_threads(threads)
    sd_e, sd_m, sd_g = seeded_weights()
    img_lq, img_up, img_ref = [t[:1] for t in synthetic_pair(1234, BATCH, LR, REF)]     # bounded sample: image 0, 1 image per step
    ref_path.full_forward(sd_e, sd_m, sd_g, img_lq, img_up, img_ref)         # warm-up
    t0 = time.perf_counter()
    for _ in range(args.steps):
        sr = ref_path.full_forward(sd_e, sd_m, sd_g, img_lq, img_up, img_ref)
    dt = time.perf_counter() - t0
    v = args.steps / dt
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {'sr': sr})
    sample = (f'1 image per step (config-2 shapes), {args.steps} timed steps after 1 warm-up, '
              f'torch-CPU oracle port of the reference path, {threads} threads = physical cores ({logical} logical)')
    print(json.dumps({
        'impl': 'reference', 'metric': 'SR images/sec (160x160->640x640, 500x500 Ref)', 'value': v, 'unit': 'images/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': 1, 'ms_per_step': dt / args.steps * 1e3, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'reference_arm': 'CPU, batch 1 per step'},
        'cpu_baseline': {'value': v, 'unit': 'images/s', 'cores': threads, 'kind': 'port', 'sample': sample},
        'e2e': {'value': v, 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }), flush=True)


# ------------------------------------------------------------------------------- our arm
def run_ours(args, rank, world, local_rank):
    import c2m_b200 as c2m
    from c2m_b200 import ops
    from c2m_b200.dist import max_over_ranks
    from c2m_b200.pipeline import RestorationPipeline, synthetic_pair
    import __graft_entry__ as entry

    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    dist_on = world > 1
    if dist_on:
        torch.distributed.init_process_group('nccl', device_id=dev)
        # one rank per node (re)builds the native library if it is stale; the others wait
        if local_rank == 0:
            entry.build()
        torch.distributed.barrier()
        if local_rank != 0:
            entry.build()
    else:
        entry.build()
    pipe = RestorationPipeline(dev, allow_tf32=bool(args.tf32), channels_last=bool(args.channels_last),
                               cuda_graph=bool(args.cuda_graph))
    pipe.load_state_dicts(*seeded_weights()).place()

    img_lq, img_up, img_ref = synthetic_pair(1234 + rank * 1000, BATCH, LR, REF)
    host = [t.pin_memory() for t in (img_lq, img_up, img_ref)]
    devt = [t.to(dev) for t in host]
    out_host = torch.empty(BATCH, 3, 4 * LR, 4 * LR, dtype=torch.float32).pin_memory()
    flush = torch.empty(192 * 1024 * 1024, dtype=torch.uint8, device=dev)       # > 126 MB L2
    h2d = sum(t.numel() * t.element_size() for t in host)
    d2h = out_host.numel() * out_host.element_size()

    def barrier():
        if dist_on:
            torch.distributed.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps):
        """K steps, each bracketed by events on the current stream, L2 flushed (untimed) between them.
        Returns (max-over-ranks ms, what the last step returned)."""
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        for e0, e1 in evs:
            out = None          # free the previous result first: each step allocates as if it had been discarded
            flush.fill_(1)
            e0.record()
            out = fn()
            e1.record()
        barrier()
        ms = sum(e0.elapsed_time(e1) for e0, e1 in evs)
        return max_over_ranks(ms, dev), out

    step_eager = lambda: pipe.forward(*devt)
    step_dev = (lambda: pipe.forward_graphed(*devt)) if args.cuda_graph else step_eager
    step_e2e = lambda: pipe.run_host(*host, out=out_host)

    for _ in range(max(args.warmup, 3)):
        step_eager()
    torch.cuda.synchronize(dev)
    n0 = c2m.launch_count()
    step_eager()                        # one eager step counts the launches of a step (a graph replay issues the same kernels)
    torch.cuda.synchronize(dev)
    launches_per_step = c2m.launch_count() - n0
    for _ in range(max(args.warmup, 3)):
        step_dev()                      # with --cuda-graph the first call captures
    step_e2e()
    torch.cuda.synchronize(dev)

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    # (1) the headline numbers: library profiling hook OFF, nothing but the step inside the events
    ops.profile_enable(False)
    ms_dev, sr_dev = timed(step_dev, args.steps)
    # copied out before anything else runs (a graph replay or a later forward may reuse the buffer); the device
    # batch is released right away, so the passes below allocate as if it had been discarded
    dumped = {'sr': sr_dev.cpu()} if args.dump_outputs and rank == 0 else None
    del sr_dev
    launches = launches_per_step * args.steps
    ms_e2e, sr_e2e = timed(step_e2e, args.steps)       # sr_e2e is out_host, the pinned buffer every e2e step fills
    if dumped is not None:
        dumped['e2e_sr'] = sr_e2e.clone()
    clocks = sampler.stop() if sampler else None
    # (2) separate pass for the per-kernel-class device times (2 cudaEventRecord per launch: not part of `value`)
    prof_steps = max(1, min(args.steps, 5))
    ops.profile_enable(True)
    for k in ops.PROF_KERNELS:
        ops.profile_collect(k)
    ms_prof = timed(step_eager, prof_steps)[0]
    prof = {k: ops.profile_collect(k) for k in ops.PROF_KERNELS}
    ops.profile_enable(False)

    imgs = BATCH * args.steps * world
    value = imgs / (ms_dev / 1e3)
    e2e = imgs / (ms_e2e / 1e3)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except Exception:
            pass
        peak = peaks.get('bf16_tflops_sustained')       # kernel timed inside a long step -> sustained figure
        peak_src = 'measured (MEASURED_PEAKS.json bf16_tflops_sustained)'
        if not peak:
            peak, peak_src = 1400.0, 'fallback (B200_PROFILING.md: ~1.4 PFLOP/s sustained)'
        # per kernel class: device time inside the timed steps (CUDA events on the launching stream,
        # recorded by the library), algorithmic flops / bytes per SURVEY.md §8(d)
        classes = {}
        for k, r in prof.items():
            if r['launches']:
                classes[k] = {'ms_per_step': r['ms'] / prof_steps, 'launches_per_step': r['launches'] / prof_steps,
                              'share_of_step': r['ms'] / ms_prof,
                              'algorithmic_tflops': r['flops'] / (r['ms'] / 1e3) / 1e12,
                              'algorithmic_gbps': r['bytes'] / (r['ms'] / 1e3) / 1e9}
        dom = max(prof, key=lambda k: prof[k]['ms'])
        r = prof[dom]
        name = {'corr_search': 'corr_umma_kernel', 'conv3x3': 'conv3x3_umma_kernel', 'dcn': 'dcn_umma_kernel'}[dom]
        achieved = r['flops'] / (r['ms'] / 1e3) / 1e12
        traffic, traffic_shape = None, None
        try:
            tj = json.load(open(os.path.join(ROOT, 'profiles', 'dominant_kernel_traffic.json')))
            traffic = tj.get(name)                      # ncu dram read+write per launch (null if shapes vary)
            if (tj.get('dominant_shape') or {}).get('kernel') == name:
                traffic_shape = tj['dominant_shape']
        except Exception:
            pass
        # conv / dcn: three split products per algorithmic product.  corr: only the three ROW taps are MMAs (1/3 of the
        # nine-tap flops), x2 products ((q_hi + q_lo) * r_hi), x(16/14)^2 for the halo columns of the 16-px blocks = 0.87
        issued = {'conv3x3': 3.0, 'corr_search': 2.0 / 3.0 * (16.0 / 14.0) ** 2, 'dcn': 3.0}[dom]
        roofline = {'bound': 'tensor', 'kernel': name, 'achieved': achieved, 'peak': peak, 'unit': 'TFLOP/s',
                    'frac': achieved / peak, 'traffic': traffic, 'traffic_dominant_shape': traffic_shape,
                    'peak_source': peak_src,
                    'ms_per_launch': r['ms'] / r['launches'], 'launches_timed': r['launches'],
                    'algorithmic_flops_per_launch': r['flops'] / r['launches'],
                    'algorithmic_bytes_per_launch': r['bytes'] / r['launches'],
                    'hbm_gbps_at_algorithmic_bytes': r['bytes'] / (r['ms'] / 1e3) / 1e9,
                    'issued_over_algorithmic_mma': issued,
                    'note': 'fp32-grade results from fp16 tensor cores: every product is issued as split hi/lo '
                            'partial products (conv / DCN: hi*hi + hi*lo + lo*hi = x3 issued MMA work; the search issues '
                            'only its row taps, as the two products (q_hi + q_lo) * r_hi, and sums the column taps in the '
                            'epilogue), so the tensor-pipe busy fraction is about `issued_over_algorithmic_mma` x `frac`',
                    'per_kernel_class': classes}
        cpu = parity = micro = None
        if world == 1 and not args.no_cpu_baseline:
            # same seeded pair for the CPU leg and the GPU: image 0 of the timed batch.  The oracle's result is
            # kept and the GPU pipeline is checked against it (checker use of oracle/, never on the timed path).
            from parity_util import full_forward_parity
            cpu, want = cpu_baseline((img_lq, img_up, img_ref))
            parity = full_forward_parity(pipe, seeded_weights(), img_lq[:1], img_up[:1], img_ref[:1], want=want)
            parity['note'] = ('image 0 of the timed batch vs oracle/ref_path.full_forward on the same inputs: idx_flips = '
                              'queries whose index differs from the oracle end to end (features from tcgen05 convs vs '
                              'oneDNN), max_gap64_of_flips = largest fp64 score difference between the two candidates of '
                              'a flipped query, sr_max_rel_err = SR vs the oracle restoration evaluated on this run\'s own '
                              'index map, psnr_delta_db = |PSNR(ours) - PSNR(oracle end to end)| with the reference metric')
        if world == 1 and not args.no_micro:
            sys.path.insert(0, os.path.join(ROOT, 'tools'))
            import microbench
            micro = {'peak_tflops': peaks.get('bf16_tflops') or 1590.0, 'peak_hbm_gbs': peaks.get('hbm_gbs') or 6650.0,
                     'peaks': 'MEASURED_PEAKS.json burst figures (kernels timed alone)' if peaks else 'fallback',
                     'rows': microbench.run_config3(dev, flush, peaks.get('bf16_tflops') or 1590.0) +
                             microbench.run_config4(dev, flush, peaks.get('hbm_gbs') or 6650.0)}
        print(json.dumps({
            'metric': 'SR images/sec (160x160->640x640, 500x500 Ref)', 'value': value, 'unit': 'images/s',
            'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
            'ms_per_step': ms_dev / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'global_batch': BATCH * world, 'parallelism': f'dp{world} (batch-sharded pairs, no data-path collective)',
                       'l2': 'flushed between timed steps (192 MiB fill)', 'profiling_hook': 'off while `value` / `e2e` are timed', 'cuda_graph': bool(args.cuda_graph), 'weights': 'random-init (seeded), real architecture',
                       'convs': 'hand-written tcgen05 3x3 kernel, split-fp16 operands, fp32 accumulate (fp32-grade); '
                                'cuDNN is not on the path', 'cudnn_tf32_allowed': bool(args.tf32)},
            'e2e': {'value': e2e, 'unit': 'images/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                    'ms_per_step': ms_e2e / args.steps, 'api': 'c2m_b200.pipeline.RestorationPipeline.run_host'},
            'gpu_launches': int(launches), 'roofline': roofline, 'cpu_baseline': cpu, 'parity': parity, 'micro': micro,
            'clocks': clocks,
        }), flush=True)
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped)
    if dist_on:
        torch.distributed.destroy_process_group()


# ------------------------------------------------------------------------------- config 5 (N1: sharded evaluation)
def run_config5(args, rank, world, local_rank):
    """BASELINE config 5: 126 synthetic CUFED5-shape pairs (config-2 shapes) through the model-level driver
    `RefRestorationModel.validation` — dataset decode + PIL resizes in loader workers, rank::world sharding at the
    index level, same-shape batches, forward, async D2H, PSNR/SSIM on a thread pool, final metric all-gather.
    value = pairs of ALL ranks / max-over-ranks wall time (barrier + sync on both sides)."""
    import __graft_entry__ as entry
    from c2m_b200.dist import max_over_ranks
    from mmsr.data import create_dataloader, create_dataset
    from mmsr.models.ref_restoration_model import RefRestorationModel
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    dist_on = world > 1
    if dist_on:
        torch.distributed.init_process_group('nccl', device_id=dev)
        if local_rank == 0:
            entry.build()
        torch.distributed.barrier()
    entry.build()
    opt = {'name': 'config5', 'suffix': None, 'scale': 4, 'crop_border': None, 'dist': dist_on, 'is_train': False,
           'post_workers': args.post_workers, 'metrics_device': args.metrics_device,
           'network_g': {'type': 'RestorationNet', 'ngf': 64, 'n_blocks': 16, 'groups': 8},
           'network_map': {'type': 'CorrespondenceGenerationArch', 'patch_size': 3, 'stride': 1,
                           'vgg_layer_list': ['relu1_1', 'relu2_1', 'relu3_1'], 'vgg_type': 'vgg19', 'vgg_pretrained': False},
           'network_extractor': {'type': 'ContrasExtractorSep'}, 'path': {}}
    model = RefRestorationModel(opt)
    for net, sd in zip((model.net_extractor, model.net_map, model.net_g), seeded_weights()):
        net.load_state_dict(sd, strict=True)
    dopt = {'name': 'config5_synth', 'type': 'SyntheticRefDataset', 'phase': 'test', 'num': args.pairs, 'gt_size': 4 * LR,
            'ref_size': REF, 'scale': 4, 'num_workers': args.loader_workers, 'batch_size': args.eval_batch,
            'prefetch_factor': 2, 'per_sample_workers': not args.per_batch_workers}
    dset = create_dataset(dopt)
    # warm-up on a few pairs (weight packing, allocator, loader worker start-up are not part of the metric)
    wopt = dict(dopt, num=max(2, args.eval_batch) * world)
    wloader = create_dataloader(create_dataset(wopt), wopt, dist=dist_on)
    model.validation(wloader, 0)
    getattr(wloader, 'close', lambda: None)()

    def barrier():
        if dist_on:
            torch.distributed.barrier()
        torch.cuda.synchronize(dev)

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    loader = create_dataloader(dset, dopt, dist=dist_on)
    barrier()
    t0 = time.perf_counter()
    res = model.validation(loader, 0)
    barrier()
    wall = max_over_ranks(time.perf_counter() - t0, dev)
    clocks = sampler.stop() if sampler else None
    getattr(loader, 'close', lambda: None)()
    stage = torch.tensor([res['rank_loader_wait_s'], res['rank_submit_s'], res['rank_wall_s'], float(res['rank_images']),
                          res['rank_gpu_busy_s']],
                         dtype=torch.float64, device=dev)
    if dist_on:
        stages = [torch.zeros_like(stage) for _ in range(world)]
        torch.distributed.all_gather(stages, stage)
    else:
        stages = [stage]
    if rank == 0:
        per_rank = [{'images': int(s[3]), 'wall_s': round(float(s[2]), 3), 'loader_wait_s': round(float(s[0]), 3),
                     'forward_submit_s': round(float(s[1]), 3), 'gpu_busy_s': round(float(s[4]), 3)} for s in stages]
        worst = max(per_rank, key=lambda r: r['wall_s'])
        limiting = ('GPU forward (device busy %d %% of the wall time)' % round(100 * worst['gpu_busy_s'] / worst['wall_s'])
                    if worst['gpu_busy_s'] > 0.7 * worst['wall_s'] else
                    'host loader (GPU waits for decoded pairs)' if worst['loader_wait_s'] > 0.3 * worst['wall_s'] else
                    'host post-processing / submit')
        physical, logical = host_cores()
        print(json.dumps({
            'metric': 'SR images/sec, sharded evaluation of 126 CUFED5-shape pairs (config 5)', 'value': args.pairs / wall,
            'unit': 'images/s', 'n_gpus': world, 'steps': 1, 'warmup': 1, 'ms_per_step': wall * 1e3, 'higher_is_better': True,
            'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': f'config5: {args.pairs} synthetic pairs (GT 640x640, Ref 500x500 zero-padded), RefRestorationModel.validation: '
                                   'dataset decode + PIL bicubic in loader workers ('
                                   + ('one batch' if args.per_batch_workers else 'one pair') + ' per worker task), rank::world index '
                                   'sharding, same-shape batches, forward, PSNR/PSNR_Y/SSIM_Y '
                                   + ('on the GPU (float64, reference definitions)' if args.metrics_device == 'cuda' else
                                      'on a host thread pool after an async D2H copy') + ', final all-gather of the metric rows',
                       'metrics_device': args.metrics_device, 'eval_batch': args.eval_batch, 'loader_workers_per_rank': args.loader_workers,
                       'post_workers_per_rank': args.post_workers, 'host_cores': {'physical': physical, 'logical': logical},
                       'parallelism': f'dp{world} (pair list sharded rank::world; collective = metric all-gather only)'},
            'validation': {k: res[k] for k in ('psnr', 'psnr_y', 'ssim_y', 'n')}, 'per_rank': per_rank,
            'limiting_stage': limiting, 'clocks': clocks,
        }), flush=True)
    if dist_on:
        torch.distributed.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None, help='timed steps of config2 (default 10)')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', choices=['ours', 'reference'], default='ours')
    ap.add_argument('--tf32', type=int, default=0, help='allow cuDNN TF32 for the plain convolutions (default: exact fp32)')
    ap.add_argument('--channels-last', type=int, default=0)
    ap.add_argument('--cuda-graph', type=int, default=0,
                    help='replay the forward from a CUDA graph captured per input shape (same kernels, bit-identical results; measured: no '
                         'gain, 100.7 vs 101.1 images/s — the step runs at the power cap, not at the launch rate)')
    ap.add_argument('--no-cpu-baseline', action='store_true', help='skip the CPU oracle leg (cpu_baseline + parity)')
    ap.add_argument('--no-micro', action='store_true', help='skip the config-3 / config-4 microbenchmarks')
    ap.add_argument('--workload', choices=['config2', 'config5'], default='config2',
                    help='config2 (default, the headline metric) or config5: sharded evaluation of 126 pairs')
    ap.add_argument('--pairs', type=int, default=126)
    ap.add_argument('--eval-batch', type=int, default=4)
    ap.add_argument('--loader-workers', type=int, default=10)
    ap.add_argument('--post-workers', type=int, default=6)
    ap.add_argument('--metrics-device', choices=['cuda', 'cpu'], default='cuda',
                    help="config5: where PSNR/SSIM run ('cpu' = the reference's numpy/cv2 arithmetic on a thread pool)")
    ap.add_argument('--per-batch-workers', action='store_true', help='config5: one BATCH per loader-worker task')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='config2: write the outputs of the last timed step to DIR/<name>.npy (float32)')
    args = ap.parse_args()
    if args.workload == 'config5' and args.steps is not None:
        ap.error('--steps applies to the config2 workload (config5 times one validation pass over --pairs pairs)')
    if args.steps is None:
        args.steps = 10
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.workload != 'config2':
        ap.error('--dump-outputs applies to the config2 workload')
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    if args.impl == 'reference':
        run_reference(args, rank)
    elif args.workload == 'config5':
        run_config5(args, rank, world, local_rank)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == '__main__':
    main()
