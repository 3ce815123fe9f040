#!/usr/bin/env python
"""bench.py -- optimisation steps/sec of the Aphantasia hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1]): clip_fft.py --size 1280-720 --samples 200 ViT-B/32 FFT -> S = int(200*0.95) = 190
crops (clip_fft.py:167-169), transforms_fast, macro 0.4, 'mix' loss, Adam(lr .05, betas (0,.999)). One "step" = one
train(i) body without the preview branch (clip_fft.py:235-295): synth fwd -> sample fwd -> ViT fwd -> loss -> ViT
data-gradient -> sample bwd -> [all-reduce] -> synth bwd -> Adam.

  value : steps/s with everything resident in HBM (crop tables pre-staged), C-ABI calls only, CUDA-event timed.
  e2e   : steps/s through the reference-facing Python entry points (fft_image / to_valid_rgb / slice_imgs /
          model.encode_image / sim_func + loss.backward() + torch.optim.Adam), including per step the host RNG replay,
          the pinned H2D copy of the crop table and a D2H read of the loss.
  --impl reference : the CPU oracle port of the reference path (oracle/restate.py) on the host cores.
"""
import os as _os
if _os.environ.get('NCCL_DEBUG', 'VERSION').upper() == 'VERSION':
    _os.environ['NCCL_DEBUG'] = 'WARN'          # NCCL's version banner goes to stdout: keep stdout to the one JSON line
import argparse
import ctypes as C
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

H, W, SAMPLES_FLAG, MODEL, PATCH = 720, 1280, 200, 'ViT-B/32', 32
S_TOTAL = int(SAMPLES_FLAG * 0.95)
F_VIT = {32: 8.8176e9, 16: 35.1269e9}      # forward FLOPs per image (SURVEY.md 8d)
# one workload string for BOTH arms (the driver compares config.workload of the two lines)
WORKLOAD = 'clip_fft.py --size 1280-720 --samples 200 ViT-B/32 FFT: S=190 crops/step, transforms_fast, mix loss, Adam'


def vit_gemm_shapes(S, patch=32, D=768, layers=12, out=512, res=224):
    """(M, N, K) of every tcgen05 GEMM launch of one step (forward + data-gradient)."""
    g = res // patch; T = g * g + 1; M = S * T; Mp = S * g * g; Kp = 3 * patch * patch
    fwd = [(Mp, D, Kp)] + layers * [(M, 3 * D, D), (M, D, D), (M, 4 * D, D), (M, D, 4 * D)] + [(S, out, D)]
    bwd = [(S, D, out)] + layers * [(M, 4 * D, D), (M, D, 4 * D), (M, D, D), (M, D, 3 * D)] + [(Mp, Kp, D)]
    return fwd + bwd


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index=0):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True); self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for r in self.rows if len(r) >= 7]
        if not rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples']}
        sm = sorted(float(r[0]) for r in rows)
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith('active') for r in rows)]
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': float(rows[0][1]), 'power_w_max': max(float(r[2]) for r in rows),
                'samples': len(rows), 'reasons': reasons}


# =============================================================================================== ours
class DeviceStep:
    """The whole step as direct C-ABI calls on resident buffers (no autograd, no per-step host work but launches)."""

    def __init__(self, S_local, S_total, rank, world, n_tables, seed=0):
        from aphantasia_b200 import _lib, _rng
        from aphantasia_b200.clip import VisionTransformer, synthetic_visual_state_dict
        from aphantasia_b200.image import FFTImage, _color_matrix_host
        self.L, self.lib = _lib, _lib.lib()
        self.S, self.S_total, self.world = S_local, S_total, world
        dev = torch.device('cuda')
        torch.manual_seed(seed); np.random.seed(seed)
        self.params = (0.01 * torch.randn(1, 3, H, W // 2 + 1, 2)).to(dev)
        self.gen = FFTImage(self.params, H, W, 1.5)
        self.colmat = _color_matrix_host(1.8)
        self.vis = VisionTransformer(synthetic_visual_state_dict(patch=PATCH, seed=0), max_batch=S_local)
        g = torch.Generator().manual_seed(1234)
        txt = torch.randn(1, 512, generator=g); self.txt = (10. * txt / txt.norm()).to(dev)
        lo, hi = _rng.shard_range(S_total, rank, world)
        if world == 1 and os.environ.get('APH_BENCH_SHARD_OF'):
            lo, hi = _rng.shard_range(S_total, 0, int(os.environ['APH_BENCH_SHARD_OF']))
        assert hi - lo == S_local
        tabs = []
        for _ in range(n_tables):       # every rank replays the full stream, keeps its shard (results independent of N)
            t, _f = _rng.draw_crop_table(S_total, (H, W), 224, _rng.TF_FAST, 'uniform', 0.4)
            tabs.append(torch.from_numpy(np.ascontiguousarray(t[0][lo:hi])))
        self.tables = torch.stack(tabs).to(dev)
        f32 = dict(device=dev, dtype=torch.float32)
        self.x_raw = torch.empty(3, H, W, **f32); self.rgb = torch.empty(3, H, W, **f32)
        self.stats = torch.zeros(4, device=dev, dtype=torch.float64)
        self.crops = torch.empty(S_local, 3, 224, 224, **f32); self.g_crops = torch.empty_like(self.crops)
        self.emb = torch.empty(S_local, 512, **f32); self.g_emb = torch.empty_like(self.emb)
        self.loss = torch.zeros((), **f32)
        from aphantasia_b200 import _dist
        self._dist = _dist
        g_sym = _dist.symm_empty((3, H, W)) if world > 1 else None           # symmetric memory: our own NVLS / peer all-reduce kernel
        self.g_rgb = g_sym if g_sym is not None else torch.empty(3, H, W, **f32)
        self.g_params = torch.empty_like(self.params)
        self.m = torch.zeros_like(self.params); self.v = torch.zeros_like(self.params)
        self.t = 0
        self.ev = None
        self.patch_ptr, self.patch, self.wrote = None, 0, C.c_int(0)
        if os.environ.get('APH_PATCH_FUSE', '1') != '0':
            ptr, patch, grid = C.c_void_p(), C.c_int(), C.c_int()
            self.L.check(self.lib.aph_vit_patch_operand(self.vis.handle, S_local, C.byref(ptr), C.byref(patch), C.byref(grid)), 'patch_operand')
            self.patch_ptr, self.patch = ptr, patch.value

    def _mark(self, name):
        if self.ev is not None:
            e = torch.cuda.Event(enable_timing=True); e.record(); self.ev.append((name, e))

    def step(self, i):
        lib, ck, st = self.lib, self.L.check, self.L.stream_ptr()
        tab = self.tables[i % self.tables.shape[0]]
        self._mark('start')
        ck(lib.aph_synth_fft_fwd(self.gen.plan, self.params.data_ptr(), self.gen.scale.data_ptr(), None, 0, 1.0, self.colmat, 1,
                                 self.x_raw.data_ptr(), self.stats.data_ptr(), self.rgb.data_ptr(), st), 'synth_fwd')
        self._mark('synth_fwd')
        if self.patch_ptr is not None:      # the sampler's last stage writes the encoder's bf16 patch operand (no k_patchify)
            ck(lib.aph_sample_fwd_patches(self.rgb.data_ptr(), H, W, 0, 0, tab.data_ptr(), self.S, 224, 2, self.crops.data_ptr(),
                                          self.patch_ptr, self.patch, C.byref(self.wrote), st), 'sample_fwd')
            self._mark('sample_fwd')
            ck(lib.aph_vit_fwd_prepatched(self.vis.handle, self.S, self.emb.data_ptr(), 1, st), 'vit_fwd')
        else:
            ck(lib.aph_sample_fwd(self.rgb.data_ptr(), H, W, 0, 0, tab.data_ptr(), self.S, 224, 2, self.crops.data_ptr(), st), 'sample_fwd')
            self._mark('sample_fwd')
            ck(lib.aph_vit_fwd(self.vis.handle, self.crops.data_ptr(), self.S, self.emb.data_ptr(), 1, st), 'vit_fwd')
        self._mark('vit_fwd')
        ck(lib.aph_sim_fwd(self.txt.data_ptr(), 1, self.emb.data_ptr(), self.S, 512, 1, self.loss.data_ptr(), None, self.g_emb.data_ptr(), st), 'sim')
        self.g_emb.mul_(-1.0)                       # loss = -1 * wt * sim (clip_fft.py:116,259)
        self._mark('loss')
        ck(lib.aph_vit_bwd(self.vis.handle, self.g_emb.data_ptr(), self.S, self.g_crops.data_ptr(), st), 'vit_bwd')
        self._mark('vit_bwd')
        ck(lib.aph_sample_bwd_scaled(self.g_crops.data_ptr(), H, W, 0, 0, tab.data_ptr(), self.S, 224, 2, float(self.S) / float(self.S_total),
                                     self.g_rgb.data_ptr(), st), 'sample_bwd')
        self._mark('sample_bwd')
        if self.world > 1:
            self._dist.all_reduce_sum_(self.g_rgb)
            self._mark('allreduce')
        ck(lib.aph_synth_fft_bwd(self.gen.plan, self.g_rgb.data_ptr(), self.rgb.data_ptr(), self.x_raw.data_ptr(), self.stats.data_ptr(),
                                 self.gen.scale.data_ptr(), 1.0, self.colmat, 1, self.g_params.data_ptr(), st), 'synth_bwd')
        self._mark('synth_bwd')
        self.t += 1
        ck(lib.aph_adam_step(self.params.data_ptr(), self.g_params.data_ptr(), self.m.data_ptr(), self.v.data_ptr(), self.params.numel(),
                             0.05, 0.0, 0.999, 1e-8, self.t, st), 'adam')
        self._mark('adam')


# supplementary workloads (BASELINE.json configs; effective crop counts after the script's multipliers, SURVEY.md 8)
CONFIGS = {
    'c1': dict(hw=(224, 224), S=3, patch=32, dwt=False, sim='mix', note='configs[0] shape: 224x224, --samples 4 -> S=3, ViT-B/32'),
    'c2': dict(hw=(720, 1280), S=190, patch=32, dwt=False, sim='mix', note='configs[1]: 1280x720 FFT, --samples 200 -> S=190, ViT-B/32'),
    'c3': dict(hw=(1080, 1920), S=47, patch=16, dwt=True, sim='mix', note='configs[2]: --dwt --wave db3 1920x1080, --samples 200 -> S=47, ViT-B/16'),
    'c5shard': dict(hw=(2160, 3840), S=24, patch=16, dwt=False, sim='mix', note='configs[4], one rank of 8: 3840x2160 FFT, S=190 -> 24 crops/rank, ViT-B/16 (no all-reduce)'),
}


class ApiStep:
    """The same step through the reference-facing Python entry points (what clip_fft.py's train(i) executes)."""

    def __init__(self, seed=0, cfg=None, fused_adam=False):
        from aphantasia_b200 import transforms
        from aphantasia_b200.clip import CLIP, synthetic_visual_state_dict
        from aphantasia_b200.image import dwt_image, fft_image, to_valid_rgb
        from aphantasia_b200.utils import sim_func, slice_imgs
        cfg = cfg or CONFIGS['c2']
        self.S, self.sim = cfg['S'], cfg['sim']
        h, w = cfg['hw']
        self.slice_imgs, self.sim_func, self.tf = slice_imgs, sim_func, transforms.transforms_fast
        torch.manual_seed(seed); np.random.seed(seed)
        if cfg['dwt']:
            self.params, image_f, _ = dwt_image([1, 3, h, w], 'db3', 0.3, 1.8, None)
        else:
            self.params, image_f, _ = fft_image([1, 3, h, w], 0.07, 1.5, None)
        self.image_f = to_valid_rgb(image_f, colors=1.8)
        self.model = CLIP('ViT-B/%d' % cfg['patch'], synthetic_visual_state_dict(patch=cfg['patch'], seed=0), True)
        g = torch.Generator().manual_seed(1234)
        txt = torch.randn(1, 512, generator=g); self.txt = (10. * txt / txt.norm()).cuda()
        if fused_adam:       # what APH_FUSED_ADAM=1 gives the unmodified script: Adam fused into the synthesis backward (row f2)
            from aphantasia_b200 import optim
            self.opt = optim.Adam(self.params, 0.05, betas=(.0, .999))
        else:
            self.opt = torch.optim.Adam(self.params, 0.05, betas=(.0, .999))

    def step(self, i):
        img_out = self.image_f(None)
        img_sliced = self.slice_imgs([img_out], self.S, 224, self.tf, 'uniform', 0.4)[0]
        out_enc = self.model.encode_image(img_sliced)
        loss = -1. * 1. * self.sim_func(self.txt, out_enc, self.sim)
        self.opt.zero_grad()
        loss.backward()
        self.opt.step()
        return loss.item()                          # D2H read of the step's result

    def script_step(self, i, opt_step, outdir):
        """train(i) of the unmodified script, statement for statement (clip_fft.py:235-306): incl. the per-step
        torch.cuda.empty_cache() (:285) and, every `opt_step`, the preview branch: second synthesis under no_grad, read-back,
        checkout() -> JPEG (:297-306). No loss read-back: the script never reads its loss."""
        from aphantasia_b200.utils import checkout
        img_out = self.image_f(None)
        img_sliced = self.slice_imgs([img_out], self.S, 224, self.tf, 'uniform', 0.4)[0]
        out_enc = self.model.encode_image(img_sliced)
        loss = 0
        loss += -1. * 1. * self.sim_func(self.txt, out_enc, self.sim)
        del img_out, img_sliced, out_enc; torch.cuda.empty_cache()
        self.opt.zero_grad()
        loss.backward()
        self.opt.step()
        if i % opt_step == 0:
            with torch.no_grad():
                img = self.image_f(contrast=1.1).cpu().numpy()[0]
            checkout(img, os.path.join(outdir, '%04d.jpg' % (i // opt_step)), verbose=False)


def timed(fn, steps, warmup, dist_barrier):
    for i in range(warmup):
        fn(i)
    torch.cuda.synchronize(); dist_barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn(warmup + i)
    e1.record()
    torch.cuda.synchronize(); dist_barrier()
    return e0.elapsed_time(e1) / 1e3


def usable_cpus():
    """CPUs this process may really use: affinity mask and cgroup quota, not the host's core count."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    try:
        q, per = open('/sys/fs/cgroup/cpu.max').read().split()
        if q != 'max':
            n = min(n, max(1, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return max(1, min(n, 64))      # beyond 64 threads the per-crop ops of the reference only lose to thread overhead


def _cpu_setup(threads=None):
    """Inputs of the CPU arm: same seeds / shapes as DeviceStep (so its step-0 loss is comparable). The crop table comes from the
    PYTHON specification of the RNG replay (_rng.draw_crop_table_py): nothing of libaphb200.so is loaded on this path."""
    from aphantasia_b200 import _rng
    from aphantasia_b200.clip import synthetic_visual_state_dict
    from oracle import restate as R
    cores = threads or usable_cpus()
    torch.set_num_threads(cores)
    torch.manual_seed(0); np.random.seed(0)
    params = 0.01 * torch.randn(1, 3, H, W // 2 + 1, 2)
    scale, cm = R.fft_scale(H, W, 1.5), R.color_matrix(1.8)
    vis = R.build_visual(synthetic_visual_state_dict(patch=PATCH, seed=0))
    g = torch.Generator().manual_seed(1234)
    txt = torch.randn(1, 512, generator=g); txt = 10. * txt / txt.norm()
    tabs, _ = _rng.draw_crop_table_py(S_TOTAL, (H, W), 224, _rng.TF_FAST, 'uniform', 0.4)

    def step(S):
        t0 = time.perf_counter()
        loss, _g, _e = R.reference_step(params, scale, (H, W), cm, tabs[0][:S], vis, txt, 'mix')
        return time.perf_counter() - t0, float(loss)
    return step, cores


_SAMPLE_TXT = 'oracle/restate.py reference_step (torch fp32 on the host, incl. the CLIP weight-gradients the reference also computes), 1280x720 canvas, '


def cpu_baseline_port(budget_s=30., threads=None, state=None):
    """Times the oracle port of the reference step on the host cores. A FULL 190-crop step is timed when it fits `budget_s`
    (then nothing is extrapolated); otherwise a crop sample is timed and scaled linearly in the crop count, and says so."""
    step, cores = state or _cpu_setup(threads)
    step(1)                                          # warm-up (allocator, thread pool)
    t1, _ = step(1)
    t8, _ = step(8)
    per_crop = max(t8 - t1, 1e-9) / 7.
    est_full = t1 + per_crop * (S_TOTAL - 1)
    if est_full <= budget_s:
        t_full, loss = step(S_TOTAL)
        return {'value': 1.0 / t_full, 'unit': 'steps/s', 'cores': cores, 'kind': 'port', 'extrapolated': False, 'crops_timed': S_TOTAL,
                'step0_loss': loss, 'sample': _SAMPLE_TXT + 'one full %d-crop step timed: %.2fs' % (S_TOTAL, t_full)}
    n = int(max(8, min(S_TOTAL, (budget_s - t1) / per_crop)))
    tn, _ = step(n)
    t_full = t1 + max(tn - t1, 1e-9) / max(n - 1, 1) * (S_TOTAL - 1)
    return {'value': 1.0 / t_full, 'unit': 'steps/s', 'cores': cores, 'kind': 'port', 'extrapolated': True, 'crops_timed': n, 'step0_loss': None,
            'sample': _SAMPLE_TXT + '%d of %d crops timed (%.2fs) + 1-crop step (%.2fs), extrapolated linearly in crops to %.2fs/step' % (n, S_TOTAL, tn, t1, t_full)}


def gpu_eager_baseline(steps=3):
    """Second baseline (BASELINE.md 3.5): the reference's op sequence as plain PyTorch-eager CUDA ops on THIS GPU (fp16 CLIP as
    clip.load() gives on a GPU, incl. the weight gradients the reference computes) -- tests/eager_gpu_baseline.py."""
    import importlib.util
    spec = importlib.util.spec_from_file_location('eager_gpu_baseline', os.path.join(ROOT, 'tests', 'eager_gpu_baseline.py'))
    mod = importlib.util.module_from_spec(spec); spec.loader.exec_module(mod)
    r = mod.measure(steps, ('fp16_clip_with_weight_grads',))['fp16_clip_with_weight_grads']
    return {'value': r['steps_per_s'], 'unit': 'steps/s', 'ms_per_step': r['ms_per_step'], 'steps': steps,
            'what': 'same step as PyTorch-eager CUDA ops on the same GPU (per-crop interpolate / grid_sample loop, nn.MultiheadAttention CLIP in fp16 with weight gradients)'}


def run_supplementary(args):
    """Other BASELINE configs, end to end through the Python entry points only (evidence for profiles/, not the bench line)."""
    cfg = CONFIGS[args.config]
    torch.cuda.set_device(0)
    api = ApiStep(cfg=cfg)
    t = timed(api.step, args.steps, args.warmup, lambda: None)
    flops = 2.0 * cfg['S'] * F_VIT[cfg['patch']]
    emit({'config': args.config, 'workload': cfg['note'], 'e2e_steps_per_s': args.steps / t, 'ms_per_step': 1e3 * t / args.steps,
                      'vit_tflops_of_step': flops / (t / args.steps) / 1e12, 'steps': args.steps, 'warmup': args.warmup})


def run_ours(args):
    import torch.distributed as dist
    rank = int(os.environ.get('RANK', '0')); world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl')
    barrier = (lambda: dist.barrier()) if world > 1 else (lambda: None)
    os.environ['APH_SYNC_SEED'] = '0'
    from aphantasia_b200 import _dist, _lib, _rng
    _dist.init()
    lo, hi = _rng.shard_range(S_TOTAL, rank, world)
    if world == 1 and os.environ.get('APH_BENCH_SHARD_OF'):      # profiling knob: one rank's shard of an N-GPU run on a single GPU (no all-reduce)
        lo, hi = _rng.shard_range(S_TOTAL, 0, int(os.environ['APH_BENCH_SHARD_OF']))
    K, Wm = args.steps, args.warmup

    # ---- device-resident leg (value)
    ds = DeviceStep(hi - lo, S_TOTAL, rank, world, n_tables=min(K + Wm, 32))
    loss0_dev = None
    if world == 1:          # step-0 loss (= -sim) on the initial spectrum, before anything is updated: compared with the oracle's below
        p0 = ds.params.clone()
        ds.step(0); torch.cuda.synchronize()
        loss0_dev = -float(ds.loss.item())
        ds.params.copy_(p0); ds.m.zero_(); ds.v.zero_(); ds.t = 0
    clocks = ClockSampler(local) if rank == 0 else None
    l0 = _lib.lib().aph_launch_count()
    t_dev = timed(ds.step, K, Wm, barrier)
    launches = (_lib.lib().aph_launch_count() - l0) * K // (K + Wm)
    clk = clocks.stop() if clocks else None
    if args.dump_outputs and rank == 0:       # before the stage timing below runs more steps on the same buffers
        dump_outputs(ds, args.dump_outputs)
    # per-stage split + GEMM-kernel timing, measured live right after the timed region (same process, same buffers)
    ds.ev = []
    for i in range(3):
        ds.step(i)
    torch.cuda.synchronize()
    stages = {}
    for (n0, e0), (n1, e1) in zip(ds.ev[:-1], ds.ev[1:]):
        if n1 != 'start':
            stages[n1] = stages.get(n1, 0.) + e0.elapsed_time(e1) / 3
    ds.ev = None
    gemm = time_gemms(ds, hi - lo) if os.environ.get('APH_BENCH_GEMM', '1') == '1' else {'ms': 0., 'tflops': 0., 'launches': 0}
    # the GEMM kernel inside the real step (real fused epilogues): event pair around every launch, 3 steps
    lib = _lib.lib()
    lib.aph_prof_gemm(1, None, None, None)
    for i in range(3):
        ds.step(i)
    pm, pf, pl = C.c_double(), C.c_double(), C.c_int()
    _lib.check(lib.aph_prof_gemm(0, C.byref(pm), C.byref(pf), C.byref(pl)), 'aph_prof_gemm')
    gemm_live = {'ms': pm.value / 3, 'tflops': pf.value / (pm.value * 1e-3) / 1e12 if pm.value > 0 else 0., 'launches': pl.value // 3}
    t = torch.tensor([t_dev], device='cuda', dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t_dev = float(t.item())
    del ds
    torch.cuda.empty_cache()

    if os.environ.get('APH_BENCH_LEGS', 'all') == 'device':      # profiling runs (ncu) only need the resident leg
        if rank == 0:
            emit({'value': K / t_dev, 'ms_per_step': 1e3 * t_dev / K, 'stages_ms': stages, 'gemm': gemm, 'note': 'device leg only'})
        return
    # ---- end-to-end leg through the public API (e2e)
    api = ApiStep()
    t_api = timed(api.step, K, Wm, barrier)
    t = torch.tensor([t_api], device='cuda', dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t_api = float(t.item())
    e2e_fused = None
    if world == 1 and not CONFIGS['c2']['dwt']:
        del api
        torch.cuda.empty_cache()
        api_f = ApiStep(fused_adam=True)
        t_f = timed(api_f.step, K, Wm, barrier)
        e2e_fused = {'value': K / t_f, 'unit': 'steps/s', 'ms_per_step': 1e3 * t_f / K,
                     'what': 'same as e2e with aphantasia_b200.optim.Adam (APH_FUSED_ADAM=1 for the unmodified script): the update runs inside the synthesis backward'}
        del api_f
        torch.cuda.empty_cache()
        api = ApiStep()
        for i in range(3):
            api.step(i)
    # the same loop exactly as the unmodified script runs it (empty_cache per step, preview every opt_step), wall-clock incl. the
    # asynchronous JPEG encoder's drain: what a user of clip_fft.py sees at the default --opt_step 1 and at --opt_step 50
    script = {}
    if world == 1 and os.environ.get('APH_BENCH_SCRIPT', '1') == '1':
        import shutil, tempfile
        from aphantasia_b200.utils import _drain_saves
        for ops in (1, 50):
            d = tempfile.mkdtemp(prefix='aph_bench_')
            try:
                n = max(K, 50) * (2 if ops == 50 else 1)      # opt_step 50: two previews in the window (one made the 50-step leg noisy)
                for i in range(5):
                    api.script_step(i, ops, d)
                _drain_saves(); torch.cuda.synchronize()
                t0 = time.perf_counter()
                for i in range(n):
                    api.script_step(i, ops, d)
                torch.cuda.synchronize(); _drain_saves()
                dt = time.perf_counter() - t0
                script['opt_step_%d' % ops] = {'value': n / dt, 'unit': 'steps/s', 'steps': n, 'frames_written': len(os.listdir(d))}
            finally:
                shutil.rmtree(d, ignore_errors=True)

    collective = _dist.collective_mode()
    coll_err = _dist.collective_error() if world > 1 else False
    assert not coll_err, 'a rank barrier of the symmetric all-reduce timed out'
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    peak_tf = peaks.get('bf16_tflops_sustained', 1400.0)
    peak_src = 'MEASURED_PEAKS.json bf16_tflops_sustained' if peaks else 'fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)'
    flops_vit = 2.0 * (hi - lo) * F_VIT[PATCH]
    traffic = None
    try:        # DRAM bytes per launch of the same kernel from the committed ncu capture (cannot be measured outside a profiler)
        traffic = json.load(open(os.path.join(ROOT, 'profiles', 'r2p_gemm_traffic.json')))['traffic_bytes_per_launch']
    except Exception:
        pass
    out = {
        'metric': 'optimization steps/sec @1280x720 FFT, 200 samples, ViT-B/32', 'value': K / t_dev, 'unit': 'steps/s',
        'n_gpus': world, 'steps': K, 'warmup': Wm, 'ms_per_step': 1e3 * t_dev / K, 'higher_is_better': True, 'scaling': 'strong',
        'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic (seeded spectrum, seeded synthetic ViT-B/32 weights, seeded text embedding)',
        'config': {'workload': WORKLOAD,
                   'parallelism': ('samples sharded over %d GPU(s), one all-reduce of dRGB per step (%s)' % (world, collective)) if world > 1 else 'single GPU',
                   'l2': 'working set per step (~1.9 GB of saved activations) exceeds the 126 MB L2; no explicit flush'},
        'e2e': {'value': K / t_api, 'unit': 'steps/s', 'h2d_bytes_per_step': (hi - lo) * 24 * 4, 'd2h_bytes_per_step': 4,
                'ms_per_step': 1e3 * t_api / K, 'path': 'fft_image/to_valid_rgb/slice_imgs/encode_image/sim_func + backward + torch.optim.Adam'},
        'e2e_fused_adam': e2e_fused,
        'e2e_script': script or None,
        'gpu_launches': int(launches),
        'clocks': clk,
        'roofline': {'bound': 'tensor', 'kernel': 'k_gemm_bf16_tn (tcgen05): all %d launches of one step, CUDA-event pair around each launch '
                                                  'inside the running step (real fused epilogues)' % gemm_live['launches'],
                     'achieved': gemm_live['tflops'], 'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': gemm_live['tflops'] / peak_tf, 'traffic': traffic,
                     'traffic_source': 'profiles/r2p_gemm_traffic.json (ncu --set full: dram__bytes_read+write of the 8 GEMM launches of one transformer layer inside a C2 step, per launch; algorithmic operand+output bytes of the same launches = 87 MB per launch, the difference is absorbed by the 126 MB L2 between consecutive kernels)',
                     'peak_source': peak_src, 'gemm_ms_per_step': gemm_live['ms'],
                     'isolated_plain_epilogue': {'tflops': gemm['tflops'], 'ms_per_step': gemm['ms'], 'per_shape_ms': gemm.get('per_shape_ms')},
                     'vit_step_frac': (flops_vit / (1e-3 * (stages.get('vit_fwd', 0) + stages.get('vit_bwd', 0)) + 1e-12)) / 1e12 / peak_tf},
        'stages_ms': {k: round(v, 4) for k, v in stages.items()},
    }
    out['parity'] = {'step0_loss': loss0_dev, 'what': 'loss of the first device-resident step (seed 0); the oracle value of the same step is cpu_baseline.step0_loss'}
    if world == 1:
        try:
            out['cpu_baseline'] = cpu_baseline_port()
            ol = out['cpu_baseline'].get('step0_loss')
            if ol is not None and loss0_dev is not None:
                out['parity'].update({'oracle_step0_loss': ol, 'abs_diff': abs(ol - loss0_dev), 'tolerance': 2e-3})
        except Exception as ex:      # the baseline must never take the bench line down
            out['cpu_baseline'] = {'value': None, 'unit': 'steps/s', 'cores': os.cpu_count(), 'kind': 'port', 'sample': 'failed: %r' % (ex,)}
        if os.environ.get('APH_BENCH_EAGER', '1') == '1':
            try:
                out['gpu_eager_baseline'] = gpu_eager_baseline()
            except Exception as ex:
                out['gpu_eager_baseline'] = {'value': None, 'unit': 'steps/s', 'what': 'failed: %r' % (ex,)}
    emit(out)


def dump_outputs(ds, out_dir):
    """Writes what the last timed step of the device leg handed back, one .npy per array (~34 MB at C2): the loss, the crop
    embeddings (rank 0's shard when --gpus > 1), the RGB canvas, the spectrum gradient and the spectrum after that step's Adam
    update. Inputs are seeded, so two builds run with the same arguments can be compared array for array."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {'loss': -ds.loss, 'embeddings': ds.emb, 'image': ds.rgb, 'spectrum_grad': ds.g_params, 'spectrum': ds.params}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), t.detach().float().cpu().numpy())


def time_gemms(ds, S):
    """Average duration of the step's tcgen05 GEMM launches: each shape of the step replayed on the handle's own
    operand-sized buffers with CUDA events on the launching stream (after warm-up)."""
    from aphantasia_b200 import _lib
    lib, ck = _lib.lib(), _lib.check
    shapes = vit_gemm_shapes(S, PATCH)
    uniq = sorted(set(shapes))
    st = _lib.stream_ptr()
    per = {}
    for (M, N, K) in uniq:
        a = torch.randn(M, K, device='cuda').bfloat16(); b = torch.randn(N, K, device='cuda').bfloat16()
        c = torch.empty(M, N, device='cuda')
        for _ in range(3):
            ck(lib.aph_gemm_bf16_tn(a.data_ptr(), b.data_ptr(), c.data_ptr(), M, N, K, st), 'gemm')
        reps = 10
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            ck(lib.aph_gemm_bf16_tn(a.data_ptr(), b.data_ptr(), c.data_ptr(), M, N, K, st), 'gemm')
        e1.record(); torch.cuda.synchronize()
        per[(M, N, K)] = e0.elapsed_time(e1) / reps
    ms = sum(per[s] for s in shapes)
    fl = sum(2.0 * m * n * k for (m, n, k) in shapes)
    return {'ms': ms, 'tflops': fl / (ms * 1e-3) / 1e12, 'launches': len(shapes),
            'per_shape_ms': {'%dx%dx%d' % s: round(v, 4) for s, v in per.items()}}


# =============================================================================================== reference arm
def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    K, Wm = max(args.steps, 1), args.warmup
    state = _cpu_setup()
    step, cores = state
    step(1)
    t1, _ = step(1)
    t8, _ = step(8)
    per_crop = max(t8 - t1, 1e-9) / 7.
    est_full = t1 + per_crop * (S_TOTAL - 1)
    budget = 240.0                                   # the whole --steps K --warmup W run must end within a few minutes
    n = S_TOTAL if est_full * (K + Wm) <= budget else int(max(8, min(S_TOTAL, (budget / (K + Wm) - t1) / per_crop)))
    times, loss0 = [], None
    for i in range(Wm + K):
        t, loss = step(n)
        if i == 0:
            loss0 = loss
        if i >= Wm:
            times.append(t)
    t_n = float(np.median(times))
    extrap = n < S_TOTAL
    t_full = t_n if not extrap else t1 + max(t_n - t1, 1e-9) / max(n - 1, 1) * (S_TOTAL - 1)
    v = 1.0 / t_full
    cb = {'value': v, 'unit': 'steps/s', 'cores': cores, 'kind': 'port', 'extrapolated': extrap, 'crops_timed': n, 'steps_timed': K,
          'step0_loss': loss0 if not extrap else None,
          'sample': _SAMPLE_TXT + ('%d full %d-crop steps timed, median %.2fs' % (K, S_TOTAL, t_n) if not extrap else
                                   '%d steps of %d of %d crops timed (median %.2fs), extrapolated linearly in crops to %.2fs/step' % (K, n, S_TOTAL, t_n, t_full))}
    out = {'impl': 'reference', 'metric': 'optimization steps/sec @1280x720 FFT, 200 samples, ViT-B/32', 'value': v, 'unit': 'steps/s',
           'n_gpus': args.gpus, 'steps': K, 'warmup': Wm, 'ms_per_step': 1e3 / v, 'higher_is_better': True, 'scaling': 'strong',
           'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic (same seeds / shapes as the GPU arm)',
           'config': {'workload': WORKLOAD, 'arm': 'CPU oracle port of the reference path on %d host threads' % cores},
           'extrapolated': extrap,
           'cpu_baseline': cb, 'e2e': {'value': v, 'unit': 'steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}, 'gpu_launches': 0}
    emit(out)


def main():
    # stdout carries exactly ONE line (the JSON): anything a library prints while we run (NCCL banners, torch notices) goes to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        _main()
    finally:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        if _RESULT_LINE:
            os.write(1, (_RESULT_LINE[-1] + '\n').encode())


_RESULT_LINE = []


def emit(obj):
    _RESULT_LINE.append(json.dumps(obj))


def _main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', default='c2', choices=sorted(CONFIGS), help='c2 = the bench line (default); others: supplementary e2e runs')
    ap.add_argument('--dump-outputs', metavar='DIR', help='after the timed steps, write the outputs of the last one to DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if args.dump_outputs and (args.impl != 'ours' or args.config != 'c2'):
        ap.error('--dump-outputs writes the outputs of the bench line: --impl ours --config c2')
    args.warmup = max(args.warmup, 3) if args.impl == 'ours' else args.warmup
    if args.impl == 'ours' and args.config != 'c2':
        run_supplementary(args)
    elif args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
