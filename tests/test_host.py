"""CPU-only tests of the host logic and the C-ABI surface (no compute calls: there is no GPU in the build container)."""
import os
import re
import socket
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_and_exports_every_declared_symbol():
    from aphantasia_b200 import _lib
    hdr = open(os.path.join(ROOT, 'include', 'aphb200.h')).read()
    declared = sorted(set(re.findall(r'\b(aph_[a-z0-9_]+)\s*\(', hdr)))
    assert len(declared) >= 20
    lib = _lib.lib()
    for name in declared:
        assert hasattr(lib, name), 'libaphb200.so does not export %s' % name
    assert sorted(_lib.EXPORTS) == declared, 'ctypes signature table and header disagree'
    assert lib.aph_version() == 1
    assert int(re.search(r'#define APH_CROP_PARAM_FLOATS (\d+)', hdr).group(1)) == __import__('aphantasia_b200._rng', fromlist=['x']).CROP_PARAM_FLOATS


def test_table_layout_matches_header():
    from aphantasia_b200 import _rng
    hdr = open(os.path.join(ROOT, 'include', 'aphb200.h')).read()
    get = lambda n: int(re.search(r'#define %s\s+(\d+)' % n, hdr).group(1))
    assert (get('APH_F_OFFY'), get('APH_F_OFFX'), get('APH_F_CSIZE'), get('APH_F_FLAGS')) == (_rng.F_OFFY, _rng.F_OFFX, _rng.F_CSIZE, _rng.F_FLAGS)
    assert (get('APH_F_PERSP'), get('APH_F_ER_I'), get('APH_F_ER_W'), get('APH_F_ROT'), get('APH_F_ANGLE')) == \
           (_rng.F_PERSP, _rng.F_ER_I, _rng.F_ER_W, _rng.F_ROT, _rng.F_ANGLE)
    assert (get('APH_TF_NONE'), get('APH_TF_NORMALIZE'), get('APH_TF_FAST')) == (_rng.TF_NONE, _rng.TF_NORMALIZE, _rng.TF_FAST)


@pytest.mark.parametrize('count,world', [(190, 8), (87, 4), (190, 1), (3, 2), (5, 8), (47, 3)])
def test_shard_range_is_a_balanced_partition(count, world):
    from aphantasia_b200 import _rng
    spans = [_rng.shard_range(count, r, world) for r in range(world)]
    assert spans[0][0] == 0 and spans[-1][1] == count
    assert all(a[1] == b[0] for a, b in zip(spans[:-1], spans[1:]))
    sizes = [hi - lo for lo, hi in spans]
    assert max(sizes) - min(sizes) <= 1
    if (count, world) == (190, 8): assert sizes == [24] * 6 + [23] * 2
    if (count, world) == (87, 4): assert sizes == [22, 22, 22, 21]


def test_perspective_and_rotation_helpers_match_torchvision():
    import torchvision.transforms.functional as TF
    from aphantasia_b200 import _rng
    start = [[0, 0], [223, 0], [223, 223], [0, 223]]
    end = [[11, 30], [200, 5], [190, 215], [20, 199]]
    assert _rng.perspective_coeffs(start, end) == TF._get_perspective_coeffs(start, end)
    for ang in (-30., -7., 0., 13., 29.):
        m = TF._get_inverse_affine_matrix([0., 0.], ang, [0., 0.], 1., [0., 0.])
        assert _rng.inverse_rotation_matrix(ang) == [m[0], m[1], m[3], m[4]]


@pytest.mark.skipif(torch.cuda.is_available(), reason='checks the loud failure on a GPU-less host')
def test_product_path_has_no_cpu_fallback():
    from aphantasia_b200 import transforms
    from aphantasia_b200.utils import slice_imgs
    with pytest.raises(RuntimeError, match='no CPU path'):
        slice_imgs([torch.rand(1, 3, 64, 64)], 2, 32, transforms.transforms_fast)
    with pytest.raises(NotImplementedError):
        slice_imgs([torch.rand(1, 3, 64, 64)], 2, 32, lambda x: x)


def test_dropin_module_names_resolve():
    sys.path.insert(0, os.path.join(ROOT, 'dropin'))
    try:
        for k in [k for k in sys.modules if k == 'aphantasia' or k.startswith('aphantasia.') or k in ('clip', 'imageio', 'lpips')]:
            del sys.modules[k]
        from aphantasia.image import to_valid_rgb, fft_image, dwt_image  # noqa: F401
        from aphantasia.utils import (slice_imgs, derivat, sim_func, aesthetic_model, basename, img_list, img_read, plot_text,  # noqa: F401
                                      txt_clean, checkout, old_torch)
        from aphantasia import transforms
        from aphantasia.progress_bar import ProgressBar  # noqa: F401
        import clip
        assert hasattr(transforms, 'transforms_fast') and hasattr(transforms, 'normalize') and hasattr(transforms, 'transforms_custom')
        assert clip.tokenize('red square').shape == (1, 77)
    finally:
        sys.path.remove(os.path.join(ROOT, 'dropin'))


def _free_port():
    s = socket.socket(); s.bind(('127.0.0.1', 0)); p = s.getsockname()[1]; s.close(); return p


def _worker(rank, world, port, q):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    torch.cuda.is_available = lambda: False      # the ranks act as GPU-less hosts (gloo), also where there are fewer GPUs than ranks
    sys.path.insert(0, ROOT)
    from aphantasia_b200 import _dist, _rng
    torch.manual_seed(100 + rank); np.random.seed(100 + rank)      # deliberately different before the seed sync
    st = _dist.init()
    S = 11
    tabs, _ = _rng.draw_crop_table(S, (96, 128), 32, _rng.TF_FAST, 'uniform', 0.4)
    lo, hi = _rng.shard_range(S, st['rank'], st['world'])
    # stand-in for the per-crop canvas gradients: g_s = f(table row); local mean over the shard, weighted, summed over ranks
    per_crop = torch.tensor(tabs[0][:, :3].sum(1) + tabs[0][:, 16], dtype=torch.float64)
    local = per_crop[lo:hi].mean() if hi > lo else torch.zeros((), dtype=torch.float64)
    g = (local * (hi - lo) / S).reshape(1).clone()
    _dist.all_reduce_sum_(g)
    q.put((rank, tabs[0].tobytes(), (lo, hi), float(g.item()), float(per_crop.mean().item())))
    torch.distributed.destroy_process_group()


def test_two_rank_gloo_sharding_matches_single_process():
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    q, port = ctx.Queue(), _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs: p.start()
    try:
        res = sorted(q.get(timeout=120) for _ in range(2))
    finally:
        for p in procs:
            p.join(30)
            if p.is_alive():        # its peer died: it would wait in the rendezvous and keep pytest from exiting
                p.terminate()
    (r0, t0, s0, g0, m0), (r1, t1, s1, g1, m1) = res
    assert t0 == t1, 'ranks replayed different random streams'
    assert s0 == (0, 6) and s1 == (6, 11)
    assert abs(g0 - m0) < 1e-12 and abs(g1 - m0) < 1e-12        # weighted local means, summed == the global mean


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the oracle port timed on the host cores) must print ONE JSON line with the arm's keys."""
    import json, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0'],
                         capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['unit'] == 'steps/s' and d['higher_is_better'] is True and d['value'] > 0
    assert d['metric'].startswith('optimization steps/sec') and 'workload' in d['config']
    cb = d['cpu_baseline']
    assert cb['kind'] in ('port', 'reference') and cb['cores'] >= 1 and cb['sample'] and cb['value'] == d['value']
    assert d['e2e']['value'] == d['value'] and d['e2e']['h2d_bytes_per_step'] == 0 and d['e2e']['d2h_bytes_per_step'] == 0


def test_native_replay_in_place_numpy_state_equals_copy_path():
    """The native replay advances NumPy's global MT19937 state where it lives (no get_state/set_state round trip); the result and
    the state it leaves behind must equal the copy path's, also across reseeding and interleaved draws."""
    from aphantasia_b200 import _rng

    def run(force_copy):
        torch.manual_seed(3); np.random.seed(3)
        _rng._NP_INPLACE = False if force_copy else None
        outs = []
        for i in range(5):
            tabs, _ = _rng.draw_crop_table_native(37, (360, 640), 224, _rng.TF_FAST, 'uniform', 0.4)
            outs.append(tabs[0].copy())
            outs.append(np.array([np.random.rand(), np.random.randint(0, 100), torch.rand(1).item(), np.random.randn()]))
            if i == 2:
                np.random.seed(10)
        return outs
    try:
        a, b = run(False), run(True)
    finally:
        _rng._NP_INPLACE = None
    assert _rng._numpy_state_address() is not None          # this NumPy exposes the expected mt19937_state layout
    assert all(np.array_equal(x, y) for x, y in zip(a, b))


# ---------------------------------------------------------------------------------------------- launcher (SURVEY 8b)
_LAUNCH_PROBE = '''
import sys
from aphantasia.image import to_valid_rgb, fft_image, dwt_image
from aphantasia.utils import slice_imgs, sim_func
from aphantasia import transforms
import clip, aphantasia
print("ORIGIN", aphantasia.__file__, sim_func.__module__, clip.load.__module__, sys.argv[1:])
'''


def _run_launcher(script, args, cwd):
    import subprocess
    env = dict(os.environ, APH_RUN_VERBOSE='1', PYTHONPATH=ROOT)
    return subprocess.run([sys.executable, '-m', 'aphantasia_b200.run', script] + args, capture_output=True, text=True, timeout=300, cwd=cwd, env=env)


def test_launcher_shadows_a_package_sitting_next_to_the_script(tmp_path):
    """`python script.py` puts the script's directory first on sys.path, so an `aphantasia/` package beside the script (the
    reference tree) would win over PYTHONPATH. The launcher must resolve the module names to dropin/ anyway."""
    (tmp_path / 'aphantasia').mkdir()
    (tmp_path / 'aphantasia' / '__init__.py').write_text('raise ImportError("the package next to the script was imported")\n')
    (tmp_path / 'clip.py').write_text('raise ImportError("the clip module next to the script was imported")\n')
    script = tmp_path / 'probe.py'
    script.write_text(_LAUNCH_PROBE)
    out = _run_launcher(str(script), ['--size', '224-224'], cwd=str(tmp_path))
    assert out.returncode == 0, out.stderr[-3000:]
    line = [l for l in out.stdout.splitlines() if l.startswith('ORIGIN')][0]
    assert os.path.join(ROOT, 'dropin', 'aphantasia') in line and 'aphantasia_b200.utils' in line and 'aphantasia_b200.clip' in line
    assert "['--size', '224-224']" in line
    assert 'aphantasia -> %s' % os.path.join(ROOT, 'dropin', 'aphantasia') in out.stderr


@pytest.mark.skipif(not os.path.isfile('/root/reference/clip_fft.py'), reason='the reference tree only exists in the build container')
def test_launcher_runs_the_real_clip_fft_imports():
    """The unmodified /root/reference/clip_fft.py, started from INSIDE the reference tree: all of its top-level imports
    (clip_fft.py:1-31) must resolve through the drop-in (argparse --help exits before any GPU work)."""
    out = _run_launcher('/root/reference/clip_fft.py', ['--help'], cwd='/root/reference')
    assert out.returncode == 0, out.stderr[-3000:]
    assert '--samples' in out.stdout and '--dualmod' in out.stdout
    assert 'aphantasia -> %s' % os.path.join(ROOT, 'dropin', 'aphantasia') in out.stderr
    assert 'clip -> %s' % os.path.join(ROOT, 'dropin', 'clip') in out.stderr


@pytest.mark.parametrize('wave,N', [('coif1', 1), ('coif2', 2)])
def test_tabulated_coiflets_have_their_defining_properties(wave, N):
    """coifN (length 6N): orthonormal even shifts, sum sqrt(2), 2N vanishing wavelet moments, scaling-function moments
    1..2N-1 vanishing about an integer centre. These conditions pin the filter up to reflection."""
    from aphantasia_b200._wavelets import reconstruction_filters
    rec_lo, rec_hi = reconstruction_filters(wave)
    h = np.array(rec_lo[::-1], np.float64); L = len(h)
    assert L == 6 * N and abs(h.sum() - np.sqrt(2)) < 1e-10
    for m in range(L // 2):
        assert abs(sum(h[k] * h[k + 2 * m] for k in range(L - 2 * m)) - (1. if m == 0 else 0.)) < 1e-10
    g = np.array(rec_hi, np.float64)
    for p in range(2 * N):
        assert abs(sum(g[k] * float(k) ** p for k in range(L))) < 1e-8, 'wavelet moment %d' % p
    hn = h / np.sqrt(2); c = sum(k * hn[k] for k in range(L))
    assert abs(c - round(c)) < 1e-9
    for p in range(1, 2 * N):
        assert abs(sum(hn[k] * (k - c) ** p for k in range(L))) < 1e-8, 'scaling moment %d' % p
    # PyWavelets relation between the reconstruction pair
    assert np.allclose(g, [(-1) ** k * h[k] for k in range(L)])


# ---------------------------------------------------------------------------------------------- sampler -> encoder hand-over (host logic)
def test_patchlink_stamp_and_match_rules():
    """aphantasia_b200/_patchlink.py without a GPU: which tensors may take the prepatched encoder route."""
    import gc
    import torch
    from aphantasia_b200 import _patchlink

    class Vis:                       # the attributes _patchlink reads from clip.VisionTransformer
        def __init__(self, res):
            self.input_resolution, self._patch_gen, self._handle_epoch = res, 0, 1

    saved = list(_patchlink._consumers)
    _patchlink._consumers.clear()
    try:
        assert _patchlink.target(224) is None                       # no encoder alive
        v = Vis(224)
        _patchlink.register(v)
        assert _patchlink.target(224) is v and _patchlink.target(336) is None
        os.environ['APH_PATCH_FUSE'] = '0'
        assert _patchlink.target(224) is None
        os.environ.pop('APH_PATCH_FUSE')
        x = torch.zeros(4, 3, 8, 8)
        assert not _patchlink.matches(x, v)                         # never stamped
        v._patch_gen = 7
        _patchlink.stamp(x, v, 4)
        assert _patchlink.matches(x, v)
        assert not _patchlink.matches(x * 1.0, v)                   # a derived tensor carries no stamp
        assert not _patchlink.matches(x, Vis(224))                  # another encoder
        v._patch_gen = 8                                            # the operand buffer was rewritten since
        assert not _patchlink.matches(x, v)
        v._patch_gen = 7
        v._handle_epoch = 2                                         # the handle was re-created (bigger batch)
        assert not _patchlink.matches(x, v)
        v._handle_epoch = 1
        assert _patchlink.matches(x, v)
        x.add_(1.0)                                                 # edited in place after the sampler wrote the operand
        assert not _patchlink.matches(x, v)
        w = Vis(224)
        _patchlink.register(w)
        assert _patchlink.target(224) is None                       # two live encoders (--dualmod): plain route
        del w
        gc.collect()
        assert _patchlink.target(224) is v                          # ... and back once one is gone
    finally:
        _patchlink._consumers.clear()
        for c in saved:
            _patchlink.register(c)
