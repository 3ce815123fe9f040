"""GPU parity tests: every CUDA kernel of libaphb200.so, called through the C ABI (ctypes) / the drop-in entry
points, against the CPU oracle (oracle/restate.py) and the committed reference fixtures, on identical seeds.

Tolerances (norm-wise relative error, BASELINE.json north_star): 1e-3 for the fp32 kernels (we hold them to
much tighter bounds below), 2e-2 for the bf16 tensor-core path of the ViT.
"""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import restate as R  # noqa: E402


def _rel(a, b):
    a = torch.as_tensor(np.asarray(a.detach().cpu() if torch.is_tensor(a) else a)).double()
    b = torch.as_tensor(np.asarray(b.detach().cpu() if torch.is_tensor(b) else b)).double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def _seed(s):
    torch.manual_seed(int(s)); np.random.seed(int(s))


@pytest.fixture(scope='module')
def L():
    from aphantasia_b200 import _lib
    assert torch.cuda.is_available()
    return _lib


# ---------------------------------------------------------------------------------------------- GEMM
@pytest.mark.parametrize('M,N,K', [(128, 128, 64), (256, 256, 128), (300, 384, 192), (1000, 768, 3072), (9500, 2304, 768), (190, 512, 768)])
def test_tcgen05_gemm(L, M, N, K):
    _seed(M + N + K)
    a = torch.randn(M, K, device='cuda').bfloat16()
    b = torch.randn(N, K, device='cuda').bfloat16()
    c = torch.full((M, N), float('nan'), device='cuda')
    L.check(L.lib().aph_gemm_bf16_tn(a.data_ptr(), b.data_ptr(), c.data_ptr(), M, N, K, L.stream_ptr()), 'gemm')
    torch.cuda.synchronize()
    ref = a.float() @ b.float().T
    assert torch.isfinite(c).all()
    assert _rel(c, ref) < 1e-5          # bf16 products are exact in fp32; only the accumulation order differs


# ---------------------------------------------------------------------------------------------- synth
def _run_synth(L, params, h, w, decay, colors, contrast, shift=None, cot=None):
    from aphantasia_b200.image import FFTImage, to_valid_rgb
    p = torch.tensor(params).cuda().requires_grad_(True)
    gen = FFTImage(p, h, w, decay)
    rgb_f = to_valid_rgb(gen, colors=colors)
    img = gen(None, contrast)
    rgb = rgb_f(shift, contrast) if shift is not None else rgb_f(contrast=contrast)
    grad = None
    if cot is not None:
        (rgb * torch.tensor(cot).cuda()).sum().backward()
        grad = p.grad
    return img, rgb, grad


@pytest.mark.parametrize('name', ['even', 'odd', 'sq'])
def test_synth_fft_vs_reference_golden(L, golden, name):
    h, w, decay, colors, contrast = (float(v) for v in golden['fft_%s_cfg' % name])
    h, w = int(h), int(w)
    img, rgb, grad = _run_synth(L, golden['fft_%s_params' % name], h, w, decay, colors, contrast, cot=golden['fft_%s_cot' % name])
    assert _rel(img, golden['fft_%s_img' % name]) < 2e-5
    assert _rel(rgb, golden['fft_%s_rgb' % name]) < 2e-5
    assert _rel(grad, golden['fft_%s_grad' % name]) < 1e-4
    _, rgb_s, _ = _run_synth(L, golden['fft_%s_params' % name], h, w, decay, colors, contrast, shift=torch.tensor(golden['fft_%s_shift' % name]))
    assert _rel(rgb_s, golden['fft_%s_rgb_shift' % name]) < 2e-5


@pytest.mark.parametrize('h,w', [(224, 224), (720, 1280), (135, 90), (1080, 1920)])
def test_synth_fft_vs_oracle(L, h, w):
    _seed(h * 7 + w)
    params = 0.01 * torch.randn(1, 3, h, w // 2 + 1, 2)
    cot = torch.randn(1, 3, h, w)
    img, rgb, grad = _run_synth(L, params.numpy(), h, w, 1.5, 1.8, 1.0, cot=cot.numpy())
    p = params.clone().requires_grad_(True)
    scale = R.fft_scale(h, w, 1.5)
    o_img = R.synth_fft(p, scale, h, w)
    o_rgb = R.valid_rgb(o_img, R.color_matrix(1.8))
    (o_rgb * cot).sum().backward()
    assert _rel(img, o_img) < 5e-5
    assert _rel(rgb, o_rgb) < 5e-5
    assert _rel(grad, p.grad) < 2e-4


def test_valid_rgb_standalone(L):
    from aphantasia_b200.image import to_valid_rgb
    _seed(3)
    x = torch.randn(1, 3, 40, 56)
    cot = torch.randn(1, 3, 40, 56)
    xc = x.cuda().requires_grad_(True)
    out = to_valid_rgb(lambda: xc, colors=1.8)()
    (out * cot.cuda()).sum().backward()
    xo = x.clone().requires_grad_(True)
    ref = R.valid_rgb(xo, R.color_matrix(1.8))
    (ref * cot).sum().backward()
    assert _rel(out, ref) < 1e-6 and _rel(xc.grad, xo.grad) < 1e-5


# ---------------------------------------------------------------------------------------------- sampler
@pytest.mark.parametrize('name', ['small', 'mid', 'over'])
def test_sampler_vs_reference_golden(L, golden, name):
    from aphantasia_b200 import transforms
    from aphantasia_b200.utils import slice_imgs
    H, W, cnt, size, macro, s, sub = (float(v) for v in golden['smp_%s_cfg' % name])
    H, W, cnt, size, s, sub = int(H), int(W), int(cnt), int(size), int(s), int(sub)
    align = str(golden['smp_%s_align' % name])
    _seed(golden['smp_%s_canvas_seed' % name])
    canvas = torch.rand(1, 3, H, W).half().float().cuda().requires_grad_(True)
    _seed(s)
    out = slice_imgs([canvas], cnt, size, transforms.transforms_fast, align, macro)[0]
    assert _rel(out[:, :, ::sub, ::sub], golden['smp_%s_out' % name]) < 1e-5
    _seed(int(golden['smp_%s_cot_seed' % name]))
    cot = torch.randn(out.shape)
    (out * cot.cuda()).sum().backward()
    st = max(1, sub // 2)
    assert _rel(canvas.grad[:, :, ::st, ::st], golden['smp_%s_gcanvas' % name]) < 1e-4


def test_sampler_backward_variants_agree(L, tmp_path):
    """Backward variants (each in its own process): default = three-kernel form (rotation adjoint as a gather, 3 channels per thread);
    APH_SAMPLE_BWD_OLD=1 = one-kernel form, fp32 compare-and-swap shared accumulation; APH_SAMPLE_BWD_FIXED=1 = one-kernel form, integer
    fixed-point shared accumulation; APH_SAMPLE_BWD_GATHER=1 = atomic-free tile gather. All must agree to fp32 round-off, also
    for gradients 1e-6 in magnitude (the fixed-point scale is per crop, not absolute)."""
    import os, subprocess, sys
    code = """
import torch, numpy as np, sys
sys.path.insert(0, %r)
from aphantasia_b200 import transforms
from aphantasia_b200.utils import slice_imgs
torch.manual_seed(11); np.random.seed(11)
c = torch.rand(1, 3, 360, 640).cuda().requires_grad_(True)
torch.manual_seed(5); np.random.seed(5)
out = slice_imgs([c], 24, 224, transforms.transforms_fast, 'uniform', 0.4)[0]
torch.manual_seed(6)
(out * (torch.randn(out.shape) * float(sys.argv[2])).cuda()).sum().backward()
torch.save(c.grad.cpu(), sys.argv[1])
""" % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for mag in ('1.0', '1e-6'):
        outs = []
        for k, env_add in enumerate((dict(APH_SAMPLE_BWD_FIXED='1'), dict(), dict(APH_SAMPLE_BWD_GATHER='1'), dict(APH_SAMPLE_BWD_OLD='1'))):
            path = str(tmp_path / ('variant_%d.pt' % k))
            subprocess.check_call([sys.executable, '-c', code, path, mag], env=dict(os.environ, **env_add))
            outs.append(torch.load(path))
        # the one-kernel variants share the forward's tap arithmetic; the default evaluates the rotation adjoint's weights from the
        # inverse map (|sample - pixel| hat function): same values to a few ulp of the 224-pixel coordinate
        assert _rel(outs[0], outs[3]) < 1e-5 and _rel(outs[2], outs[3]) < 1e-5 and _rel(outs[1], outs[3]) < 3e-5


def test_sampler_abi_non_rotation_matrix(L):
    """The C ABI takes any 2x2 inverse affine matrix per crop; the reference's sampler only draws rotations. Rows with a sheared /
    scaled matrix (with and without a perspective hit) must take the general scatter adjoint, rows with a rotation the gather:
    forward and backward vs the oracle on a table that mixes both."""
    from aphantasia_b200 import _rng
    from aphantasia_b200._lib import check, lib, stream_ptr
    _seed(21)
    canvas = torch.rand(1, 3, 300, 420)
    S, size = 16, 224
    _seed(9)
    tabs, frame = _rng.draw_crop_table(S, (300, 420), size, 2, 'uniform', 0.4)
    tab = tabs[0].copy()
    for k in range(0, S, 2):                                    # every other crop: not a rotation
        tab[k, _rng.F_ROT:_rng.F_ROT + 4] = [1.1, 0.25, -0.1, 0.85]
    assert (tab[:, _rng.F_FLAGS].astype(int) & 1).any(), 'table should contain perspective hits'
    co = canvas.clone().requires_grad_(True)
    ref = R.sample_crops(co, tab, size, 2)
    _seed(6)
    cot = torch.randn(ref.shape)
    (ref * cot).sum().backward()
    x = canvas.cuda().contiguous(); t = torch.tensor(tab).cuda(); out = torch.empty(S, 3, size, size, device='cuda'); g = torch.empty(1, 3, 300, 420, device='cuda')
    check(lib().aph_sample_fwd(x.data_ptr(), 300, 420, 0, 0, t.data_ptr(), S, size, 2, out.data_ptr(), stream_ptr()), 'fwd')
    cg = cot.cuda().contiguous()
    check(lib().aph_sample_bwd(cg.data_ptr(), 300, 420, 0, 0, t.data_ptr(), S, size, 2, g.data_ptr(), stream_ptr()), 'bwd')
    torch.cuda.synchronize()
    assert _rel(out, ref) < 1e-5
    assert _rel(g, co.grad) < 1e-4
    # shard weight of the multi-GPU path (S_local / S, folded into the kernels): scales the gradient, nothing else
    g2 = torch.empty_like(g)
    check(lib().aph_sample_bwd_scaled(cg.data_ptr(), 300, 420, 0, 0, t.data_ptr(), S, size, 2, 0.375, g2.data_ptr(), stream_ptr()), 'bwd_scaled')
    check(lib().aph_sample_bwd(cg.data_ptr(), 300, 420, 0, 0, t.data_ptr(), S, size, 2, g.data_ptr(), stream_ptr()), 'bwd')     # scratch must be clean again
    torch.cuda.synchronize()
    assert _rel(g2, 0.375 * co.grad) < 1e-4 and _rel(g, co.grad) < 1e-4
    # a frame whose rows are not 16-byte aligned takes the scalar-reduction drain
    Wo = 421
    canvas_o = torch.rand(1, 3, 300, Wo)
    co2 = canvas_o.clone().requires_grad_(True)
    (R.sample_crops(co2, tab, size, 2) * cot).sum().backward()
    g3 = torch.empty(1, 3, 300, Wo, device='cuda')
    check(lib().aph_sample_bwd(cg.data_ptr(), 300, Wo, 0, 0, t.data_ptr(), S, size, 2, g3.data_ptr(), stream_ptr()), 'bwd odd W')
    torch.cuda.synchronize()
    assert _rel(g3, co2.grad) < 1e-4


@pytest.mark.parametrize('kind', [0, 1, 2])
def test_sampler_vs_oracle_720p(L, kind):
    from aphantasia_b200 import _rng, transforms
    from aphantasia_b200.utils import slice_imgs
    tf = [None, transforms.normalize(), transforms.transforms_fast][kind]
    _seed(11)
    canvas = torch.rand(1, 3, 360, 640)
    S = 24
    cc = canvas.cuda().requires_grad_(True)
    _seed(5)
    out = slice_imgs([cc], S, 224, tf, 'uniform', 0.4)[0]
    _seed(5)
    tabs, frame = _rng.draw_crop_table(S, (360, 640), 224, kind, 'uniform', 0.4)
    co = canvas.clone().requires_grad_(True)
    ref = R.sample_crops(co, tabs[0], 224, kind)
    _seed(6)
    cot = torch.randn(ref.shape)
    (out * cot.cuda()).sum().backward()
    (ref * cot).sum().backward()
    assert _rel(out, ref) < 1e-5
    assert _rel(cc.grad, co.grad) < 1e-4


# ---------------------------------------------------------------------------------------------- loss / adam
@pytest.mark.parametrize('t', [None, 'mix', 'cossim'])
def test_sim_func_vs_reference_golden(L, golden, t):
    from aphantasia_b200.utils import sim_func
    v1 = torch.tensor(golden['sim_v1']).cuda(); v2 = torch.tensor(golden['sim_v2']).cuda().requires_grad_(True)
    val = sim_func(v1, v2, t)
    val.backward()
    assert _rel(val, golden['sim_%s_val' % t]) < 1e-5
    assert _rel(v2.grad, golden['sim_%s_grad' % t]) < 1e-4


def test_sim_func_pairwise_and_other_kinds(L, golden):
    from aphantasia_b200.utils import sim_func
    _seed(8)
    a = torch.randn(9, 512); b = torch.randn(9, 512)
    ac = a.cuda().requires_grad_(True); bc = b.cuda().requires_grad_(True)
    ao = a.clone().requires_grad_(True); bo = b.clone().requires_grad_(True)
    sim_func(ac, bc, 'mix').backward(); R.sim_func(ao, bo, 'mix').backward()
    assert _rel(ac.grad, ao.grad) < 1e-4 and _rel(bc.grad, bo.grad) < 1e-4
    v1 = torch.tensor(golden['sim_v1']).cuda(); v2 = torch.tensor(golden['sim_v2']).cuda()
    for t in ('ang', 'dot'):
        assert _rel(sim_func(v1, v2, t), golden['sim_%s_val' % t]) < 1e-5


def test_adam_step(L):
    _seed(2)
    p0 = torch.randn(5000); g = [torch.randn(5000) for _ in range(3)]
    p = p0.clone().requires_grad_(True)
    opt = torch.optim.Adam([p], 0.05, betas=(.0, .999))
    pc = p0.cuda(); m = torch.zeros_like(pc); v = torch.zeros_like(pc)
    for i, gi in enumerate(g):
        p.grad = gi.clone(); opt.step()
        gc = gi.cuda()
        L.check(L.lib().aph_adam_step(pc.data_ptr(), gc.data_ptr(), m.data_ptr(), v.data_ptr(), pc.numel(), 0.05, 0.0, 0.999, 1e-8, i + 1,
                                      L.stream_ptr()), 'adam')
    assert _rel(pc, p) < 1e-6


# ---------------------------------------------------------------------------------------------- ViT
def _vit_pair(patch, width, layers, heads, out, res, seed):
    from aphantasia_b200.clip import VisionTransformer
    sd = R.synthetic_visual_state_dict(patch, seed, width, layers, heads, out, res)
    return VisionTransformer(sd), R.build_visual(sd)


@pytest.mark.parametrize('cfg', [dict(patch=16, width=128, layers=2, heads=2, out=128, res=64, S=5),
                                 dict(patch=32, width=256, layers=3, heads=4, out=128, res=224, S=7),
                                 dict(patch=32, width=768, layers=12, heads=12, out=512, res=224, S=3),
                                 dict(patch=16, width=768, layers=12, heads=12, out=512, res=224, S=2)])
def test_vit_forward_backward_vs_oracle(L, cfg):
    S, res = cfg['S'], cfg['res']
    ours, ref = _vit_pair(cfg['patch'], cfg['width'], cfg['layers'], cfg['heads'], cfg['out'], res, 0)
    _seed(4)
    x = torch.randn(S, 3, res, res)
    cot = torch.randn(S, cfg['out'])
    xc = x.cuda().requires_grad_(True)
    emb = ours(xc)
    (emb * cot.cuda()).sum().backward()
    xo = x.clone().requires_grad_(True)
    eo = ref(xo)
    (eo * cot).sum().backward()
    e_emb, e_grad = _rel(emb, eo), _rel(xc.grad, xo.grad)
    print('vit %s: rel err emb %.3e grad %.3e' % (cfg, e_emb, e_grad))
    assert e_emb < 2e-2 and e_grad < 2e-2       # bf16 operands, fp32 accumulation (north_star bf16 tolerance)


# ---------------------------------------------------------------------------------------------- whole step (config 1 shape)
def test_full_step_config1_vs_oracle(L):
    """BASELINE config 1 shape (224x224 canvas, S=3, ViT-B/32): loss and d loss / d spectrum vs the CPU oracle."""
    from aphantasia_b200 import _rng, transforms
    from aphantasia_b200.clip import CLIP, synthetic_visual_state_dict
    from aphantasia_b200.image import fft_image, to_valid_rgb
    from aphantasia_b200.utils import sim_func, slice_imgs
    h = w = 224; S = 3
    sd = synthetic_visual_state_dict(patch=32, seed=0)
    model = CLIP('ViT-B/32', sd, True)
    _seed(0)
    params, image_f, _ = fft_image([1, 3, h, w], 0.07, 1.5, None)
    rgb_f = to_valid_rgb(image_f, colors=1.8)
    txt = model.encode_text(torch.zeros(1, 77, dtype=torch.long)).cuda()
    _seed(1)
    crops = slice_imgs([rgb_f()], S, 224, transforms.transforms_fast, 'uniform', 0.4)[0]
    emb = model.encode_image(crops)
    loss = -1. * sim_func(txt, emb, 'mix')
    loss.backward()
    _seed(1)
    tabs, _ = _rng.draw_crop_table(S, (h, w), 224, 2, 'uniform', 0.4)
    o_loss, o_grad, o_emb = R.reference_step(params[0].detach().cpu(), R.fft_scale(h, w, 1.5), (h, w), R.color_matrix(1.8), tabs[0],
                                             R.build_visual(sd), txt.cpu(), 'mix')
    print('config1: loss ours %.6f oracle %.6f; rel emb %.3e grad %.3e' % (loss.item(), o_loss.item(), _rel(emb, o_emb), _rel(params[0].grad, o_grad)))
    assert _rel(emb, o_emb) < 2e-2
    assert abs(loss.item() - o_loss.item()) < 2e-3
    assert _rel(params[0].grad, o_grad) < 3e-2


# ---------------------------------------------------------------------------------------------- DWT (config 3 generator)
@pytest.mark.parametrize('h,w,wave', [(64, 96, 'db3'), (135, 240, 'db3'), (100, 100, 'db2'), (270, 480, 'haar')])
def test_synth_dwt_vs_oracle(L, h, w, wave):
    """dwt_image + to_valid_rgb vs the restated pytorch_wavelets DWTInverse (parity unpinned: third-party absent)."""
    from aphantasia_b200.image import dwt_image, to_valid_rgb
    _seed(h + w)
    Ys, gen, _ = dwt_image([1, 3, h, w], wave, 0.3, 1.8, None)
    rec_lo, rec_hi = R.wavelet_filters(wave)
    assert [tuple(v) for v in R.dwt_level_shapes(h, w, len(rec_lo))] == gen.level_hw
    rgb = to_valid_rgb(gen, colors=1.8)(contrast=1.1)
    _seed(9)
    cot = torch.randn(rgb.shape)
    (rgb * cot.cuda()).sum().backward()
    Yo = [y.detach().cpu().clone().requires_grad_(True) for y in Ys]
    o_img = R.synth_dwt(Yo, rec_lo, rec_hi, 0.3, 1.1)
    o_rgb = R.valid_rgb(o_img, R.color_matrix(1.8))
    (o_rgb * cot).sum().backward()
    assert tuple(rgb.shape) == tuple(o_rgb.shape)
    assert _rel(gen(contrast=1.1), o_img) < 2e-5
    assert _rel(rgb, o_rgb) < 2e-5
    for a, b in zip(Ys, Yo):
        assert _rel(a.grad, b.grad) < 2e-4


# ---------------------------------------------------------------------------------------------- BASELINE full sizes
@pytest.mark.parametrize('h,w', [(2160, 3840)])
def test_synth_fft_4k_vs_oracle(L, h, w):
    """Config 5 canvas (3840x2160): forward values and spectrum gradient vs the CPU oracle."""
    _seed(1)
    params = 0.01 * torch.randn(1, 3, h, w // 2 + 1, 2)
    cot = torch.randn(1, 3, h, w)
    img, rgb, grad = _run_synth(L, params.numpy(), h, w, 1.5, 1.8, 1.0, cot=cot.numpy())
    p = params.clone().requires_grad_(True)
    o_rgb = R.valid_rgb(R.synth_fft(p, R.fft_scale(h, w, 1.5), h, w), R.color_matrix(1.8))
    (o_rgb * cot).sum().backward()
    assert _rel(rgb, o_rgb) < 5e-5
    assert _rel(grad, p.grad) < 3e-4


def test_synth_dwt_config3_size_vs_oracle(L):
    """Config 3 generator (db3, 1920x1080): values and wavelet-pyramid gradients vs the restated DWTInverse."""
    from aphantasia_b200.image import dwt_image, to_valid_rgb
    h, w = 1080, 1920
    _seed(3)
    Ys, gen, _ = dwt_image([1, 3, h, w], 'db3', 0.3, 1.8, None)
    assert gen.level_hw[0] == (542, 962) and gen.level_hw[-1] == (6, 6) and gen.J == 10      # SURVEY.md 8a row a4
    rgb = to_valid_rgb(gen, colors=1.8)()
    _seed(4)
    cot = torch.randn(rgb.shape)
    (rgb * cot.cuda()).sum().backward()
    rec_lo, rec_hi = R.wavelet_filters('db3')
    Yo = [y.detach().cpu().clone().requires_grad_(True) for y in Ys]
    o_rgb = R.valid_rgb(R.synth_dwt(Yo, rec_lo, rec_hi, 0.3, 1.0), R.color_matrix(1.8))
    (o_rgb * cot).sum().backward()
    assert _rel(rgb, o_rgb) < 5e-5
    for a, b in zip(Ys, Yo):
        assert _rel(a.grad, b.grad) < 3e-4


def test_sampler_config5_shape_properties(L):
    """4K canvas, ViT-B/16-sized batch shard (24 crops): size-independent properties of the fused sampler.
    (i) linearity in the canvas, (ii) <grad, delta> == d/d eps of <cot, out(c + eps delta)> (adjoint identity)."""
    from aphantasia_b200 import transforms
    from aphantasia_b200.utils import slice_imgs
    H, W, S = 2160, 3840, 24
    _seed(2)
    a = torch.rand(1, 3, H, W, device='cuda'); b = torch.rand(1, 3, H, W, device='cuda')

    def run(c):
        _seed(77)
        return slice_imgs([c], S, 224, transforms.transforms_fast, 'uniform', 0.4)[0]
    oa, ob, oab = run(a), run(b), run(2 * a - 3 * b)
    mean = torch.tensor(R.CLIP_MEAN, device='cuda').view(1, 3, 1, 1); std = torch.tensor(R.CLIP_STD, device='cuda').view(1, 3, 1, 1)
    un = lambda o: o * std + mean                   # undo the affine normalisation: what remains is linear in the canvas
    assert _rel(un(oab), 2 * un(oa) - 3 * un(ob)) < 1e-4
    c = a.clone().requires_grad_(True)
    out = run(c)
    cot = torch.randn_like(out)
    (out * cot).sum().backward()
    lhs = (c.grad * b).sum().item()
    rhs = ((un(run(b)) * cot) / std).sum().item()    # <cot, L b> with L the linear part of the sampler
    assert abs(lhs - rhs) < 1e-3 * abs(rhs)


@pytest.mark.parametrize('fix', [False, True])
def test_pixel_image_vs_oracle(L, fix):
    """Next-row generator (SURVEY.md 8f rank 3): pixel_image + to_valid_rgb vs the restatement of image.py:98-119."""
    from aphantasia_b200.image import pixel_image, to_valid_rgb
    _seed(12)
    params, image_f, _ = pixel_image([1, 3, 90, 130], None, 1.)
    rgb = to_valid_rgb(image_f, colors=2.)(None, 1.1, fix)
    cot = torch.randn(rgb.shape)
    (rgb * cot.cuda()).sum().backward()
    xo = params[0].detach().cpu().clone().requires_grad_(True)
    ref = R.valid_rgb(R.synth_pixel(xo, 1.1, fix), R.color_matrix(2.))
    (ref * cot).sum().backward()
    assert _rel(rgb, ref) < 1e-6 and _rel(params[0].grad, xo.grad) < 1e-5
    assert _rel(image_f(contrast=0.7), R.synth_pixel(xo.detach(), 0.7)) < 1e-6
