#!/usr/bin/env python
"""bench.py — headline benchmark of dust3r_b200 (contract in the task statement / DESIGN.md §Measurement).

    python bench.py --gpus 1 --steps 5 --warmup 3                       # our arm, 1 GPU
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W      # our arm, N GPUs (weak scaling)
    python bench.py --impl reference --gpus 1 --steps K --warmup W      # reference arm: CPU path on host cores
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs bench_outputs/RUN   # + the last timed step's outputs as .npy

Workload (BASELINE.json configs[1]): one step = forward of a batch of 32 synthetic 512x384 pairs through
ViT-L encoder / 2x ViT-B decoder / DPT heads ("ViTLarge_BaseDecoder_512_dpt"), random-init weights.  With
N>1 every rank runs its own 32 pairs (configs[3]: 256 pairs over 8 GPUs) and the step ends with the single
NCCL all-gather of the per-pair pointmaps the north_star prescribes before alignment.
`value` is device-timed with inputs resident in HBM; `e2e` goes through the public inference() API with
pinned HOST inputs and CPU outputs.  Extra key `cloud_opt`: BASELINE configs[2] (8 views -> 28 pairs,
PointCloudOptimizer, 300 iterations) iterations/s with its own HBM roofline.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GFLOP_PER_PAIR = 1856.8          # SURVEY §8d / BASELINE.md §2 (2*MAC, enc 1046.1 + dec 437.3 + heads 373.4)
H, W = 384, 512
PAIRS_PER_GPU = 32
METRIC = 'image-pairs/sec (512x384, ViT-L/B+DPT)'
DUMP_MAX_BYTES = 64 * 2**20      # --dump-outputs writes at most this much
DUMP_SAMPLE_PX = 2**20           # pixel positions kept when the whole result would not fit (32 bytes each)
DUMP_SEED = 0


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p['hbm_gbs'], tf_burst=p['bf16_tflops'], tf_sustained=p.get('bf16_tflops_sustained', p['bf16_tflops']),
                    source='measured (MEASURED_PEAKS.json)')
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source='fallback (B200_PROFILING.md)')


def host_threads(cap=64):
    """Threads the CPU legs may use: min(affinity mask, cgroup cpu.max quota, cap).  torchrun exports OMP_NUM_THREADS=1 and
    the affinity mask of a container is usually the whole host, so neither is a usable default: round 1's reference arm
    ran 5x oversubscribed and was killed by the driver's limit."""
    try:
        n = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        n = os.cpu_count() or 1
    for path in ('/sys/fs/cgroup/cpu.max', '/sys/fs/cgroup/cpu/cpu.cfs_quota_us'):
        try:
            txt = open(path).read().split()
            if path.endswith('cpu.max'):
                if txt[0] != 'max':
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
                    n = min(n, max(1, q // per))
            break
        except (OSError, ValueError, IndexError):
            continue
    return max(1, min(n, cap))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.idx, self.rows, self.stop = gpu_index, [], threading.Event()
        self.th = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-i', str(self.idx)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(',')])
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join(timeout=6)

    def summary(self):
        sm = [float(r[1]) for r in self.rows if len(r) > 2 and r[1].replace('.', '').isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace('.', '').isdigit()]
        reasons = set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            for k, nm in enumerate(names):
                if len(r) > 5 + k and r[5 + k].lower().startswith('active'):
                    reasons.add(nm)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(self.rows))


def build_model(device):
    from dust3r_b200.config import vitl_512_dpt
    from dust3r_b200.model import AsymmetricCroCo3DStereo
    from dust3r_b200.utils.synth import synth_state_dict
    cfg = vitl_512_dpt()
    net = AsymmetricCroCo3DStereo(pos_embed='RoPE100', img_size=(512, 512), head_type='dpt', output_mode='pts3d',
                                  depth_mode=('exp', -float('inf'), float('inf')), conf_mode=('exp', 1, float('inf')),
                                  enc_embed_dim=1024, enc_depth=24, enc_num_heads=16, dec_embed_dim=768, dec_depth=12,
                                  dec_num_heads=12, landscape_only=False)
    net.load_state_dict(synth_state_dict(cfg, seed=0))
    return net.to(device), cfg


def synth_pairs_host(n_pairs, seed, pin):
    """n_pairs distinct pairs (2*n_pairs images) in load_images' format, pinned host memory."""
    g = torch.Generator().manual_seed(seed)
    views = []
    for i in range(2 * n_pairs):
        img = torch.rand((1, 3, H, W), generator=g) * 2 - 1
        if pin:
            img = img.pin_memory()
        views.append(dict(img=img, true_shape=np.int32([[H, W]]), idx=i, instance=str(i)))
    return [(views[2 * k], views[2 * k + 1]) for k in range(n_pairs)]


def cloud_opt_section(device, pk, steps_iters=300):
    """BASELINE configs[2]: 8 views -> 28 pairs (symmetrize=False), PointCloudOptimizer, 300 iterations."""
    from dust3r_b200.utils.synth import synth_pair_predictions
    from dust3r_b200.cloud_opt import global_aligner
    n = 8
    edges = [(i, j) for i in range(n) for j in range(i)]
    out = synth_pair_predictions(n, edges, H, W, seed=0)
    # the predictions arrive the way inference() hands them over: CPU tensors in pinned memory
    for side in ('pred1', 'pred2'):
        out[side] = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in out[side].items()}
    torch.manual_seed(0)
    net = global_aligner(out, device, verbose=False)
    eng = net._get_engine()
    net._engine_push(eng)
    # warm-up: a 300-iteration run lasts ~15 ms, far too short for the GPU to leave the idle clocks it fell to while the host
    # prepared the problem (measured: 170 us/iter cold vs 59 warm) -- iterate for ~0.5 s first, then time 7 runs of 300
    # iterations back to back and report the median run
    t_w = time.perf_counter()
    while time.perf_counter() - t_w < 0.5:
        eng.run(steps_iters)
        torch.cuda.synchronize()
    runs = []
    for _ in range(7):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        losses = eng.run(steps_iters)
        e1.record()
        torch.cuda.synchronize()
        runs.append(e0.elapsed_time(e1))
    ms = float(np.median(runs))
    by = eng.algorithmic_bytes_per_iter()
    gbs = by / (ms / steps_iters) / 1e6
    tr = ncu_traffic().get('align_stream' if eng.kernel == 'stream' else 'align_iter')
    # e2e through the public API: host dict in -> global_aligner -> compute_global_alignment -> float loss (median of 3 after
    # one warm-up call: the first call also pays pinned-allocator and lazy-initialisation costs)
    api = []
    for k in range(4):
        t0 = time.perf_counter()
        torch.manual_seed(0)
        net2 = global_aligner(out, device, verbose=False)
        loss = net2.compute_global_alignment(init=None, niter=steps_iters, schedule='cosine', lr=0.01)
        torch.cuda.synchronize()
        if k > 0:
            api.append(time.perf_counter() - t0)
        del net2
    t_api = float(np.median(api))
    # the same public call on predictions that never left the GPU (inference(keep_on_device=True) / inference_sharded(
    # gather_device=cuda): SURVEY 8f rank 2): no upload, the aligner packs the four stacked tensors in place
    e2e_dev = None
    try:
        out_dev = dict(out)
        for side in ('pred1', 'pred2'):
            out_dev[side] = {k: (v.to(device) if torch.is_tensor(v) else v) for k, v in out[side].items()}
        torch.cuda.synchronize()
        api_dev = []
        for k in range(4):
            t0 = time.perf_counter()
            torch.manual_seed(0)
            net3 = global_aligner(out_dev, device, verbose=False)
            loss_dev = net3.compute_global_alignment(init=None, niter=steps_iters, schedule='cosine', lr=0.01)
            torch.cuda.synchronize()
            if k > 0:
                api_dev.append(time.perf_counter() - t0)
            del net3
        e2e_dev = dict(value=steps_iters / float(np.median(api_dev)), unit='iters/s', final_loss=loss_dev,
                       includes='predictions resident in HBM (inference(keep_on_device=True)): aligner construction, packing, 300 iters, loss readback')
        del out_dev
    except Exception as ex:          # an extra figure must never cost the section
        e2e_dev = dict(unavailable=f'{type(ex).__name__}: {ex}')
    # opt-in variant of the host-prediction call: the upload is issued before the scene object is built (global_aligner(...,
    # early_upload=True)) so that it runs under the constructor's host work -- measured here, off by default
    e2e_early = None
    try:
        api_early = []
        for k in range(4):
            t0 = time.perf_counter()
            torch.manual_seed(0)
            net4 = global_aligner(out, device, verbose=False, early_upload=True)
            loss_early = net4.compute_global_alignment(init=None, niter=steps_iters, schedule='cosine', lr=0.01)
            torch.cuda.synchronize()
            if k > 0:
                api_early.append(time.perf_counter() - t0)
            del net4
        e2e_early = dict(value=steps_iters / float(np.median(api_early)), unit='iters/s', final_loss=loss_early,
                         identical_to_default=bool(loss_early == loss),
                         includes='as e2e, with global_aligner(..., early_upload=True): upload issued before the scene constructor')
    except Exception as ex:
        e2e_early = dict(unavailable=f'{type(ex).__name__}: {ex}')
    return dict(metric='cloud_opt iters/sec', value=steps_iters / ms * 1e3, unit='iters/s',
                config=dict(workload='8 synthetic views -> 28 pairs (symmetrize=False) at 512x384, PointCloudOptimizer, '
                                     '300 iters, lr 0.01 cosine, dist l1, conf log, init=None'),
                ms_per_iter=ms / steps_iters, runs_ms=[round(r, 3) for r in runs], kernel=eng.kernel, loss_first=float(losses[0]), loss_last=float(losses[-1]),
                roofline=dict(bound='hbm', achieved=gbs, peak=pk['hbm'], unit='GB/s', frac=gbs / pk['hbm'],
                              # dram__bytes_read+write per align_iter launch from the committed ncu --set full record
                              traffic=tr['bytes'] if tr else None,
                              traffic_source=f"{tr['capture']} @ {tr['commit']}" if tr else None,
                              algorithmic_bytes_per_iter=by, peak_source=pk['source']),
                e2e=dict(value=steps_iters / t_api, unit='iters/s', includes='H2D of 28 pairs of predictions (pinned host memory, as returned by inference()), packing, 300 iters, loss readback',
                         final_loss=loss, device_resident_inputs=e2e_dev, early_upload=e2e_early))


def cloud_opt_config5_section(device, pk, n=50, niter=300):
    """Alignment leg of BASELINE configs[4] on ONE GPU (alignment does not shard: replicas only): 50 views -> 1225 pairs at
    512x384, predictions synthesised in HBM (where the all-gather of the sharded forward leaves them), global_aligner in
    ModularPointCloudOptimizer mode, 300 iterations.  7.9 GB of algorithmic traffic per iteration: no cache effects."""
    from dust3r_b200.cloud_opt import global_aligner, GlobalAlignerMode
    edges = [(i, j) for i in range(n) for j in range(i)]
    g = torch.Generator(device=device).manual_seed(0)
    E = len(edges)
    off = torch.tensor([0.0, 0.0, 3.0], device=device)
    ts = torch.from_numpy(np.int32([[H, W]] * E))
    mk = lambda: torch.randn((E, H, W, 3), generator=g, device=device) + off
    cf = lambda: 1 + 5 * torch.rand((E, H, W), generator=g, device=device)
    out = dict(view1=dict(idx=[int(i) for i, j in edges], instance=[str(i) for i, j in edges], true_shape=ts),
               view2=dict(idx=[int(j) for i, j in edges], instance=[str(j) for i, j in edges], true_shape=ts),
               pred1=dict(pts3d=mk(), conf=cf()), pred2=dict(pts3d_in_other_view=mk(), conf=cf()), loss=None)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    torch.manual_seed(0)
    net = global_aligner(out, device, mode=GlobalAlignerMode.ModularPointCloudOptimizer, verbose=False)
    eng = net._get_engine()
    net._engine_push(eng)
    torch.cuda.synchronize()
    t_build = time.perf_counter() - t0
    eng.run(60)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    losses = eng.run(niter)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    by = eng.algorithmic_bytes_per_iter()
    gbs = by / (ms / niter) / 1e6
    tr5 = ncu_traffic().get('align_stream_config5')
    res = dict(metric='cloud_opt iters/sec', value=niter / ms * 1e3, unit='iters/s', ms_per_iter=ms / niter, kernel=eng.kernel,
               config=dict(workload=f'{n} synthetic views -> {E} pairs (symmetrize=False) at 512x384, ModularPointCloudOptimizer, '
                                    f'{niter} iters, lr 0.01 cosine, dist l1, conf log, init=None; predictions resident in HBM'),
               aligner_build_s=round(t_build, 3), loss_first=float(losses[0]), loss_last=float(losses[-1]),
               mem_GB=round(torch.cuda.max_memory_allocated() / 1e9, 1),
               roofline=dict(bound='hbm', achieved=gbs, peak=pk['hbm'], unit='GB/s', frac=gbs / pk['hbm'],
                             traffic=tr5['bytes'] if tr5 else None, traffic_source=f"{tr5['capture']} @ {tr5['commit']}" if tr5 else None,
                             algorithmic_bytes_per_iter=by, peak_source=pk['source']))
    del net, eng, out
    torch.cuda.empty_cache()
    return res


def load_images_section(device, pk, reps=20):
    """SURVEY 8f rank 4: the pixel work of load_images for one 12 Mpx photograph (4000x3000 -> 512x384): Pillow's two-pass
    resize + crop + ImgNorm on the GPU (d3r_image_resize_crop_normalize) against the same work done by PIL on a host core
    (what the reference does), checked bit for bit.  `value` has the decoded bytes resident in HBM, `e2e` uploads them
    (pageable numpy array, as PIL hands them over) inside the timed region."""
    import PIL.Image
    from dust3r_b200.utils import image as im
    from dust3r_b200.utils.synth import synth_photo
    h0, w0, size = 3000, 4000, 512
    photo = synth_photo(h0, w0, seed=0)
    plan = im.preprocess_plan(h0, w0, size)
    src = torch.from_numpy(photo).to(device)
    for _ in range(3):
        out = im.preprocess_image_u8(src, size, device=device)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = im.preprocess_image_u8(src, size, device=device)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    t0 = time.perf_counter()
    for _ in range(5):
        out_h = im.preprocess_image_u8(photo, size, device=device)
    torch.cuda.synchronize()
    ms_e2e = (time.perf_counter() - t0) / 5 * 1e3
    # host pipeline of the reference on the same decoded image
    pil = PIL.Image.fromarray(photo)
    t0 = time.perf_counter()
    for _ in range(3):
        r = im._rescale(pil, size)
        r = r.crop(im._crop_box(r.size[0], r.size[1], size, False))
        ref = ((torch.from_numpy(np.asarray(r, dtype=np.float32) / 255).permute(2, 0, 1) - 0.5) / 0.5)[None]
    ms_cpu = (time.perf_counter() - t0) / 3 * 1e3
    by = 3 * plan['rows'] * w0 + 2 * 3 * plan['rows'] * plan['w2'] + 12 * plan['h2'] * plan['w2']
    gbs = by / ms / 1e6
    return dict(metric='load_images pixel work, images/sec', value=1e3 / ms, unit='images/s', ms_per_image=ms,
                config=dict(workload=f'{w0}x{h0} RGB uint8 -> {plan["w2"]}x{plan["h2"]} fp32 CHW (Lanczos, crop, ImgNorm), decoded bytes resident in HBM'),
                bit_exact_vs_host_pipeline=bool(torch.equal(out.cpu(), ref) and torch.equal(out_h.cpu(), ref)),
                roofline=dict(bound='hbm', achieved=gbs, peak=pk['hbm'], unit='GB/s', frac=gbs / pk['hbm'], traffic=None,
                              algorithmic_bytes_per_image=by, peak_source=pk['source'],
                              note='two launches + host-side table lookup per image; timed with CUDA events over back-to-back calls'),
                e2e=dict(value=1e3 / ms_e2e, unit='images/s', ms_per_image=ms_e2e, h2d_bytes_per_image=int(photo.nbytes),
                         includes='H2D of the decoded uint8 image from pageable host memory'),
                cpu_baseline=dict(value=1e3 / ms_cpu, unit='images/s', ms_per_image=ms_cpu, cores=1, kind='reference',
                                  sample='PIL.Image.resize(LANCZOS) + crop + ImgNorm of the same image, 3 repeats (the library calls the reference makes)'))


def _oracle_forward_setup(threads):
    from dust3r_b200.config import vitl_512_dpt
    from dust3r_b200.utils.synth import synth_state_dict, synth_images
    from oracle.forward_oracle import forward_oracle
    torch.set_num_threads(threads)
    cfg = vitl_512_dpt()
    sd = synth_state_dict(cfg, seed=0)
    imgs = synth_images(2, H, W, seed=3)
    forward_oracle(sd, cfg, imgs[0]['img'][:, :, :64, :64], imgs[1]['img'][:, :, :64, :64])  # spin up the thread pool
    return lambda: forward_oracle(sd, cfg, imgs[0]['img'], imgs[1]['img'])


def cpu_baseline_forward(n_pairs=1):
    """Oracle port (CPU fp32 torch restatement of the reference forward) on the host cores."""
    threads = host_threads()
    one_pair = _oracle_forward_setup(threads)
    t0 = time.perf_counter()
    for _ in range(n_pairs):
        one_pair()
    dt = time.perf_counter() - t0
    return dict(value=n_pairs / dt, unit='image-pairs/s', cores=threads, kind='port',
                sample=f'{n_pairs} pair(s) of 512x384, batch 1, oracle/forward_oracle.py (fp32 torch CPU restatement of the reference, '
                       'bit-identical to it: tests/test_oracle.py)')


def cpu_baseline_align(n_iters=3, budget_s=60.0):
    """BASELINE.md §3, metric 2: the reference's alignment loop (autograd + torch.optim.Adam) on the host cores, as
    restated by oracle/align_oracle.py ("reference cloud_opt + local roma restatement": `roma` is not installable
    offline), on BASELINE configs[2] (8 views -> 28 pairs at 512x384), a few iterations after one warm-up iteration."""
    from dust3r_b200.utils.synth import synth_pair_predictions
    from oracle.align_oracle import AlignProblem, init_params, align_oracle
    threads = host_threads()
    torch.set_num_threads(threads)
    n = 8
    edges = [(i, j) for i in range(n) for j in range(i)]
    out = synth_pair_predictions(n, edges, H, W, seed=0)
    prob = AlignProblem.from_output(out)
    P0 = init_params(prob, seed=0)
    t0 = time.perf_counter()
    align_oracle(prob, P0, niter=1)                      # warm-up (allocator, thread pool, autograd graph caches)
    warm = time.perf_counter() - t0
    n_iters = max(1, min(n_iters, int(budget_s / max(warm, 1e-3))))
    t0 = time.perf_counter()
    losses, _ = align_oracle(prob, P0, niter=n_iters)
    dt = time.perf_counter() - t0
    return dict(value=n_iters / dt, unit='iters/s', cores=threads, kind='port', s_per_iter=dt / n_iters,
                sample=f'{n_iters} iterations (after 1 warm-up) of PointCloudOptimizer on 8 views / 28 pairs at 512x384, '
                       'oracle/align_oracle.py = reference cloud_opt loop + local roma restatement', loss_first=float(losses[0]))


REF_WARMUP_BUDGET_S = 60.0
REF_TIMED_BUDGET_S = 170.0


def run_reference_arm(args):
    """Reference arm: the reference's own CPU implementation of the path.  /root/reference does not exist on
    the GPU box and the reference has no compiled component for this path, so this times the oracle port
    (validated bit-for-bit against the live reference in tests/test_oracle.py) on the host cores this process
    may really use (host_threads()).  One step = a bounded sample (1 pair, batch 1) of the 32-pair workload.
    The whole run is bounded by wall clock: warm-up stops after REF_WARMUP_BUDGET_S, the timed loop stops
    (and the line is still printed, with `steps` = the steps completed) once REF_TIMED_BUDGET_S are used."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    threads = host_threads()
    one_pair = _oracle_forward_setup(threads)
    sample_pairs = 1
    t_w = time.perf_counter()
    done_w = 0
    for _ in range(args.warmup):
        one_pair()
        done_w += 1
        if time.perf_counter() - t_w > REF_WARMUP_BUDGET_S:
            break
    t0 = time.perf_counter()
    done = 0
    last = 0.0
    while done < args.steps:
        ts = time.perf_counter()
        for _ in range(sample_pairs):
            one_pair()
        done += 1
        last = time.perf_counter() - ts
        if done < args.steps and (time.perf_counter() - t0) + last > REF_TIMED_BUDGET_S:
            break
    dt = time.perf_counter() - t0
    val = done * sample_pairs / dt
    line = dict(impl='reference', metric=METRIC, value=val, unit='image-pairs/s', n_gpus=args.gpus, steps=done,
                warmup=done_w, steps_requested=args.steps, warmup_requested=args.warmup,
                ms_per_step=dt / done * 1e3, higher_is_better=True, scaling='weak', vs_baseline=None,
                dtype='f32', data='synthetic',
                config=dict(workload=f'{PAIRS_PER_GPU} synthetic 512x384 pairs per GPU per step, ViTLarge_BaseDecoder_512_dpt forward only, '
                                     f'not symmetrised (CPU arm: bounded sample of {sample_pairs} pair per step, batch 1)',
                            weights='random init (synthetic, seed 0)', device='cpu', threads=threads,
                            wall_bound_s=REF_WARMUP_BUDGET_S + REF_TIMED_BUDGET_S),
                cpu_baseline=dict(value=val, unit='image-pairs/s', cores=threads, kind='port',
                                  sample=f'{sample_pairs} pair per step x {done} steps, batch 1, oracle/forward_oracle.py'),
                e2e=dict(value=val, unit='image-pairs/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    if not args.skip_cloud_opt:
        try:
            cb = cpu_baseline_align(n_iters=3, budget_s=40.0)
            line['cloud_opt'] = dict(impl='reference', metric='cloud_opt iters/sec', value=cb['value'], unit='iters/s',
                                     cpu_baseline=cb)
        except Exception as ex:   # the forward line must be printed whatever happens to the extra leg
            line['cloud_opt'] = dict(impl='reference', unavailable=f'{type(ex).__name__}: {ex}')
    print(json.dumps(line), flush=True)


def dump_outputs(outdir, r1, r2):
    """--dump-outputs: the result of the last timed step, as packed.forward() hands it to its caller, written as
    outdir/<name>.npy (float32).  When the whole result exceeds DUMP_MAX_BYTES, every array keeps the same DUMP_SAMPLE_PX pixel
    positions, drawn with DUMP_SEED from the flat (pair, row, column) index and sorted: the sample depends only on the output
    shape, so two builds run with the same arguments write arrays that compare element for element."""
    arrays = dict(pred1_pts3d=r1['pts3d'], pred1_conf=r1['conf'], pred2_pts3d_in_other_view=r2['pts3d'], pred2_conf=r2['conf'])
    n_px = int(np.prod(r1['pts3d'].shape[:3]))
    full = sum(t.numel() * t.element_size() for t in arrays.values()) <= DUMP_MAX_BYTES - 4096     # (room for the .npy headers)
    if not full:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n_px, min(DUMP_SAMPLE_PX, n_px), replace=False))
        idx = torch.from_numpy(idx).to(r1['pts3d'].device)
    os.makedirs(outdir, exist_ok=True)
    shapes = {}
    for name, t in arrays.items():
        a = t if full else t.reshape(n_px, *t.shape[3:])[idx]
        a = a.float().cpu().numpy()
        np.save(os.path.join(outdir, name + '.npy'), a)
        shapes[name] = list(a.shape)
    return dict(dir=outdir, arrays=shapes, sample=None if full else
                f'{len(idx)} of {n_px} pixel positions, numpy default_rng({DUMP_SEED}).choice without replacement, sorted')


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernels, as recorded from `ncu --set full`
    captures in profiles/ncu_traffic.json (each entry names its capture file and the commit it was taken at).  The bench
    cannot run under ncu, so these are read from the committed record rather than measured in the timed run; an entry
    that is missing yields traffic = null."""
    path = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    try:
        return json.load(open(path))
    except (OSError, ValueError):
        return {}


def build_roofline(prof, pk, value, world):
    """`roofline` object of the JSON line: the dominant kernel class of the instrumented step (CUDA events around every
    launch) against the measured bf16 peak for a kernel timed inside a long step, plus the whole-step figure."""
    tot_ms = sum(v['ms'] for v in prof.values()) or 1.0
    name, dom = max(prof.items(), key=lambda kv: kv[1]['ms'])
    dom_tflops = dom['flops'] / dom['ms'] / 1e9 if dom['flops'] and dom['ms'] else 0.0
    alg_tflops = value * GFLOP_PER_PAIR / 1e3
    traffic = ncu_traffic().get(name)
    return dict(bound='tensor', kernel=name, achieved=dom_tflops, peak=pk['tf_sustained'], unit='TFLOP/s',
                frac=dom_tflops / pk['tf_sustained'], traffic=traffic['bytes'] if traffic else None,
                traffic_note=(f"{traffic['shape']}; algorithmic {traffic['algorithmic_bytes'] / 1e6:.1f} MB; "
                              f"{traffic['capture']} @ {traffic['commit']}") if traffic else None,
                what='dominant kernel class of the step: algorithmic FLOP of its launches / their CUDA-event time, vs the measured '
                     'cuBLAS bf16 peak sustained inside a long step (burst peak: frac_of_burst_peak)',
                peak_source=pk['source'], launches=dom['count'], share_of_step=dom['ms'] / tot_ms,
                frac_of_burst_peak=dom_tflops / pk['tf_burst'],
                whole_step=dict(achieved=alg_tflops, peak=pk['tf_sustained'] * world, unit='TFLOP/s',
                                frac=alg_tflops / (pk['tf_sustained'] * world),
                                what='pairs/s x 1856.8 GFLOP/pair (SURVEY §8d) vs measured cuBLAS bf16 sustained peak'))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--pairs', type=int, default=PAIRS_PER_GPU, help='pairs per GPU per step')
    ap.add_argument('--skip-cpu-baseline', action='store_true')
    ap.add_argument('--skip-cloud-opt', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', help='after the timed steps, write the outputs of the last one (rank 0) to '
                    'DIR/<name>.npy, float32, at most 64 MB in all (a fixed, seeded sample of pixel positions when larger)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs applies to --impl ours')
    args.warmup = max(args.warmup, 0)
    if args.impl == 'reference':
        return run_reference_arm(args)

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py (our arm) needs a CUDA B200; there is no CPU fallback')
    torch.cuda.set_device(local)
    device = torch.device('cuda', local)
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group('nccl', device_id=device)
    from dust3r_b200 import _lib
    from dust3r_b200.inference import inference
    pk = peaks()
    B = args.pairs
    net, cfg = build_model(device)
    packed = net.repack()
    g = torch.Generator(device='cpu').manual_seed(1234 + rank)
    imgs = (torch.rand((2 * B, 3, H, W), generator=g) * 2 - 1).to(device)
    idx1, idx2 = np.arange(B, dtype=np.int32), B + np.arange(B, dtype=np.int32)
    # the one collective of the path (N > 1): dust3r_b200.distributed.PairOutputGather -- the same object inference_sharded()
    # uses: this rank's {pts3d, conf} x 2 rows (6.29 MB / pair) are packed into one send buffer and ONE all_gather_into_tensor
    # rebuilds the full result on every rank.  depth=2 + async_op: the gather of step k overlaps the forward of step k+1 on
    # NVLink/NVSwitch; a slot is waited for right before it is reused and all of them at the end of the timed region.
    gather = None
    if world > 1:
        from dust3r_b200.distributed import PairOutputGather
        gather = PairOutputGather(world * B, (H, W), (H, W), True, device, depth=2)

    def step():
        r1, r2 = packed.forward(imgs, idx1, idx2, B, H, W)
        if gather is not None:
            gather.gather(r1, r2, async_op=True)
        return r1, r2

    def drain():
        if gather is not None:
            gather.wait()

    W_ = max(args.warmup, 3)
    # the last result stays referenced, in the warm-up too, so that the allocator has cached the same two output sets
    # before the timed loop starts
    for _ in range(W_):
        last = step()
    drain()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    _lib.launch_count(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        torch.cuda.synchronize()
        e0.record()
        for _ in range(args.steps):
            last = step()
        drain()
        e1.record()
        torch.cuda.synchronize()
    launches = _lib.launch_count()
    dumped = dump_outputs(args.dump_outputs, *last) if args.dump_outputs and rank == 0 else None
    del last
    ms = torch.tensor([e0.elapsed_time(e1)], device=device)
    if world > 1:
        dist.barrier()
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms[0])
    value = world * B * args.steps / ms_total * 1e3

    # ---- per-kernel-class breakdown (one extra instrumented step; not part of the timed region) ----
    _lib.prof_enable(True)
    step()
    drain()
    torch.cuda.synchronize()
    prof = _lib.prof_report()
    _lib.prof_enable(False)
    kern = {}
    tot_ms = sum(v['ms'] for v in prof.values()) or 1.0
    for k, v in sorted(prof.items(), key=lambda kv: -kv[1]['ms']):
        kern[k] = dict(launches=v['count'], ms=round(v['ms'], 3), share=round(v['ms'] / tot_ms, 4),
                       tflops=round(v['flops'] / v['ms'] / 1e9, 1) if v['flops'] and v['ms'] else None,
                       gbs=round(v['bytes'] / v['ms'] / 1e6, 1) if v['bytes'] and v['ms'] else None)

    # ---- e2e through the public API: pinned host pairs -> inference() -> CPU dict ----
    e2e = None
    if rank == 0 or world > 1:
        pairs = synth_pairs_host(B, seed=99 + rank, pin=True)
        for _ in range(2):   # warm-up: also lets the pinned-host allocator cache both result buffer sets the loop alternates between
            out = inference(pairs, net, device, batch_size=B, verbose=False)
        torch.cuda.synchronize()
        n_e2e = max(2, min(args.steps, 3))
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            out = inference(pairs, net, device, batch_size=B, verbose=False)
            _ = float(out['pred1']['conf'][0, 0, 0])
        torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t0], device=device)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        h2d = 2 * B * 3 * H * W * 4
        d2h = 2 * B * H * W * 4 * 4   # pts3d (3 f32) + conf (1 f32) for both views; the returned views are the host originals
        e2e = dict(value=world * B * n_e2e / float(dt[0]), unit='image-pairs/s', h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h,
                   api='dust3r_b200.inference.inference(pairs, model, device, batch_size=32)', host_inputs='pinned')
        # the same call with PAGEABLE host images (what the reference's load_images yields): inference() stages them through
        # pinned memory itself
        pairs_pg = synth_pairs_host(B, seed=99 + rank, pin=False)
        inference(pairs_pg, net, device, batch_size=B, verbose=False)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            out = inference(pairs_pg, net, device, batch_size=B, verbose=False)
            _ = float(out['pred1']['conf'][0, 0, 0])
        torch.cuda.synchronize()
        dtp = torch.tensor([time.perf_counter() - t0], device=device)
        if world > 1:
            dist.all_reduce(dtp, op=dist.ReduceOp.MAX)
        e2e['pageable_inputs'] = dict(value=world * B * n_e2e / float(dtp[0]), unit='image-pairs/s')

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    clocks = clk.summary()
    line = dict(metric=METRIC, value=value, unit='image-pairs/s', n_gpus=world, steps=args.steps, warmup=W_,
                ms_per_step=ms_total / args.steps, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='bf16',
                data='synthetic',
                config=dict(workload=f'{B} synthetic 512x384 pairs per GPU per step ({world * B} total), '
                                     'ViTLarge_BaseDecoder_512_dpt forward only, not symmetrised (encoder sees 2 images/pair)'
                                     + (', + the single NCCL all-gather of pointmaps of inference_sharded (PairOutputGather, async, overlapped with the next step)' if world > 1 else ''),
                            weights='random init (synthetic, seed 0)', compute='bf16 operands / fp32 accumulate / fp32 residual stream',
                            l2='activations per step (>5 GB) exceed the 126 MB L2; no explicit flush needed',
                            parallelism=f'dp{world}'),
                clocks=clocks, e2e=e2e, gpu_launches=int(launches),
                roofline=build_roofline(prof, pk, value, world),
                kernels=kern)
    if dumped:
        line['dump_outputs'] = dumped
    # GPU sections first, CPU baselines last (the GPU would otherwise idle down while the host cores run the oracle)
    if world == 1 and not args.skip_cloud_opt:
        del packed, net, imgs
        torch.cuda.empty_cache()
        line['cloud_opt'] = cloud_opt_section(device, pk)
        torch.cuda.empty_cache()
        try:
            line['cloud_opt_config5'] = cloud_opt_config5_section(device, pk)
        except torch.cuda.OutOfMemoryError as ex:      # 16 GB of observations: needs a mostly free GPU
            line['cloud_opt_config5'] = dict(unavailable=f'out of memory: {ex}')
        try:
            line['load_images'] = load_images_section(device, pk)
        except Exception as ex:                        # an extra leg must never cost the headline line
            line['load_images'] = dict(unavailable=f'{type(ex).__name__}: {ex}')
    if world == 1 and not args.skip_cpu_baseline:
        line['cpu_baseline'] = cpu_baseline_forward(1)
        if not args.skip_cloud_opt:
            line['cloud_opt']['cpu_baseline'] = cpu_baseline_align(n_iters=5, budget_s=30.0)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
