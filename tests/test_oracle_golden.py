"""Pins oracle/restate.py (and the host RNG replay) against fixtures produced by the REAL reference.
CPU only. Fixture provenance: tests/golden/make_golden.py."""
import numpy as np
import pytest
import torch

from aphantasia_b200 import _rng
from oracle import restate as R


def _seed(s):
    torch.manual_seed(int(s)); np.random.seed(int(s))


def _rel(a, b):
    a = torch.as_tensor(np.asarray(a)).double(); b = torch.as_tensor(np.asarray(b)).double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


@pytest.mark.parametrize('impl', ['py', 'native'])
@pytest.mark.parametrize('name', ['c2', 'c1', 'central', 'norm', 'overscan', 'small'])
def test_rng_replay_matches_reference(golden, name, impl):
    """Both the Python replay (executable spec) and the native C replay reproduce the parameters the REAL reference used."""
    H, W, cnt, size, kind, macro, s = golden['rng_%s_cfg' % name]
    align = str(golden['rng_%s_align' % name])
    _seed(s)
    draw = _rng.draw_crop_table_py if impl == 'py' else _rng.draw_crop_table_native
    tabs, frame = draw(int(cnt), (int(H), int(W)), int(size), int(kind), align, float(macro))
    after = np.array([torch.rand(1).item(), float(np.random.rand())])
    t, ref = tabs[0].copy(), golden['rng_%s_table' % name].copy()
    if 'over' in align:   # the capture saw wrapped canvas coordinates
        t[:, 0] = (t[:, 0] - frame[0]) % H; t[:, 1] = (t[:, 1] - frame[1]) % W
    if int(kind) != 2:
        ref[:, 3] = 0; ref[:, 16:21] = t[:, 16:21]
    if impl == 'native':      # the 8x8 float64 solve is Gaussian elimination instead of LAPACK gels: same to ~1e-15 before the fp32 cast
        assert np.abs(t[:, 4:12] - ref[:, 4:12]).max() <= 1e-6 * max(1., np.abs(ref[:, 4:12]).max())
        t[:, 4:12] = ref[:, 4:12]
    assert np.array_equal(t, ref)                       # bit-exact parameters
    assert np.array_equal(after, golden['rng_%s_after' % name])   # both generators left in the same state


@pytest.mark.parametrize('name', ['even', 'odd', 'sq'])
def test_synth_fft_oracle(golden, name):
    h, w, decay, colors, contrast = (float(v) for v in golden['fft_%s_cfg' % name])
    h, w = int(h), int(w)
    p = torch.tensor(golden['fft_%s_params' % name]).requires_grad_(True)
    scale = R.fft_scale(h, w, decay)
    img = R.synth_fft(p, scale, h, w, None, contrast)
    rgb = R.valid_rgb(img, R.color_matrix(colors))
    assert _rel(img.detach(), golden['fft_%s_img' % name]) < 1e-6
    assert _rel(rgb.detach(), golden['fft_%s_rgb' % name]) < 1e-6
    (rgb * torch.tensor(golden['fft_%s_cot' % name])).sum().backward()
    assert _rel(p.grad, golden['fft_%s_grad' % name]) < 1e-5
    shift = torch.tensor(golden['fft_%s_shift' % name])
    rgb_s = R.valid_rgb(R.synth_fft(p.detach(), scale, h, w, shift, contrast), R.color_matrix(colors))
    assert _rel(rgb_s, golden['fft_%s_rgb_shift' % name]) < 1e-6


@pytest.mark.parametrize('name', ['small', 'mid', 'over'])
def test_sampler_oracle(golden, name):
    H, W, cnt, size, macro, s, sub = (float(v) for v in golden['smp_%s_cfg' % name])
    H, W, cnt, size, s, sub = int(H), int(W), int(cnt), int(size), int(s), int(sub)
    align = str(golden['smp_%s_align' % name])
    _seed(golden['smp_%s_canvas_seed' % name])
    canvas = torch.rand(1, 3, H, W).half().float().requires_grad_(True)
    _seed(s)
    tabs, frame = _rng.draw_crop_table(cnt, (H, W), size, _rng.TF_FAST, align, macro)
    out = R.sample_crops(canvas, tabs[0], size, 2, frame)
    assert _rel(out.detach()[:, :, ::sub, ::sub], golden['smp_%s_out' % name]) < 1e-6
    _seed(int(golden['smp_%s_cot_seed' % name]))
    cot = torch.randn(out.shape)
    (out * cot).sum().backward()
    g = canvas.grad
    st = max(1, sub // 2)
    assert _rel(g[:, :, ::st, ::st], golden['smp_%s_gcanvas' % name]) < 1e-5
    gs = golden['smp_%s_gsum' % name]
    assert abs(g.double().sum().item() - gs[0]) < 1e-6 * gs[1]


@pytest.mark.parametrize('t', [None, 'mix', 'cossim', 'ang', 'dot'])
def test_sim_func_oracle(golden, t):
    v1 = torch.tensor(golden['sim_v1']); v2 = torch.tensor(golden['sim_v2']).requires_grad_(True)
    val = R.sim_func(v1, v2, t)
    val.backward()
    assert _rel(val.detach(), golden['sim_%s_val' % t]) < 1e-6
    assert _rel(v2.grad, golden['sim_%s_grad' % t]) < 1e-5
    assert _rel(R.sim_func(v1, v2.detach(), 'spher'), golden['sim_spher_val']) < 1e-6


def test_chain_oracle(golden):
    """params -> rgb -> crops -> (fixed linear encoder) -> mix loss -> d params, vs the reference's autograd."""
    h, w = 48, 64
    p = torch.tensor(golden['chain_params']).requires_grad_(True)
    rgb = R.valid_rgb(R.synth_fft(p, R.fft_scale(h, w, 1.5), h, w), R.color_matrix(1.8))
    _seed(22)
    proj = torch.randn(3 * 32 * 32, 64) / 55.
    txt = torch.randn(1, 64)
    _seed(23)
    tabs, _ = _rng.draw_crop_table(5, (h, w), 32, _rng.TF_FAST, 'uniform', 0.4)
    emb = R.sample_crops(rgb, tabs[0], 32, 2).reshape(5, -1) @ proj
    loss = -R.sim_func(txt, emb, 'mix')
    loss.backward()
    assert _rel(emb.detach(), golden['chain_emb']) < 1e-5
    assert _rel(loss.detach(), golden['chain_loss']) < 1e-5
    assert _rel(p.grad, golden['chain_grad']) < 1e-4


def test_vit_restatement_matches_hf():
    """OpenAI-layout ViT restatement vs the independent HuggingFace CLIP vision tower (tiny geometry)."""
    transformers = pytest.importorskip('transformers')
    from transformers import CLIPVisionConfig, CLIPVisionModelWithProjection
    width, layers, heads, out, patch, res = 128, 2, 2, 64, 16, 64
    sd = R.synthetic_visual_state_dict(patch, 3, width, layers, heads, out, res)
    vis = R.build_visual(sd)
    cfg = CLIPVisionConfig(hidden_size=width, intermediate_size=4 * width, num_hidden_layers=layers, num_attention_heads=heads,
                           image_size=res, patch_size=patch, projection_dim=out, hidden_act='quick_gelu', layer_norm_eps=1e-5,
                           attn_implementation='eager')
    hf = CLIPVisionModelWithProjection(cfg).eval()
    v = hf.vision_model
    g = lambda k: sd['visual.' + k]
    with torch.no_grad():
        v.embeddings.patch_embedding.weight.copy_(g('conv1.weight'))
        v.embeddings.class_embedding.copy_(g('class_embedding'))
        v.embeddings.position_embedding.weight.copy_(g('positional_embedding'))
        v.pre_layrnorm.weight.copy_(g('ln_pre.weight')); v.pre_layrnorm.bias.copy_(g('ln_pre.bias'))
        v.post_layernorm.weight.copy_(g('ln_post.weight')); v.post_layernorm.bias.copy_(g('ln_post.bias'))
        hf.visual_projection.weight.copy_(g('proj').T)
        for i, l in enumerate(v.encoder.layers):
            pre = 'transformer.resblocks.%d.' % i
            wq, wk, wv = g(pre + 'attn.in_proj_weight').chunk(3); bq, bk, bv = g(pre + 'attn.in_proj_bias').chunk(3)
            l.self_attn.q_proj.weight.copy_(wq); l.self_attn.q_proj.bias.copy_(bq)
            l.self_attn.k_proj.weight.copy_(wk); l.self_attn.k_proj.bias.copy_(bk)
            l.self_attn.v_proj.weight.copy_(wv); l.self_attn.v_proj.bias.copy_(bv)
            l.self_attn.out_proj.weight.copy_(g(pre + 'attn.out_proj.weight')); l.self_attn.out_proj.bias.copy_(g(pre + 'attn.out_proj.bias'))
            l.layer_norm1.weight.copy_(g(pre + 'ln_1.weight')); l.layer_norm1.bias.copy_(g(pre + 'ln_1.bias'))
            l.layer_norm2.weight.copy_(g(pre + 'ln_2.weight')); l.layer_norm2.bias.copy_(g(pre + 'ln_2.bias'))
            l.mlp.fc1.weight.copy_(g(pre + 'mlp.c_fc.weight')); l.mlp.fc1.bias.copy_(g(pre + 'mlp.c_fc.bias'))
            l.mlp.fc2.weight.copy_(g(pre + 'mlp.c_proj.weight')); l.mlp.fc2.bias.copy_(g(pre + 'mlp.c_proj.bias'))
    torch.manual_seed(1)
    x = torch.randn(3, 3, res, res, requires_grad=True)
    a = vis(x)
    b = hf(pixel_values=x).image_embeds
    assert _rel(a.detach(), b.detach()) < 1e-5
    ga, = torch.autograd.grad(a.sum(), x); gb, = torch.autograd.grad(b.sum(), x)
    assert _rel(ga, gb) < 1e-4


@pytest.mark.parametrize('wave', ['db3', 'coif1', 'coif2'])
def test_dwt_restatement_perfect_reconstruction_unpinned(wave):
    """PARITY UNPINNED (pytorch_wavelets / PyWavelets absent): the restated symmetric-mode analysis bank followed by the restated
    DWTInverse must give the identity; this checks self-consistency of filters and conventions, not the third party's band order."""
    rec_lo, rec_hi = R.wavelet_filters(wave)
    dec_lo, dec_hi = rec_lo[::-1], rec_hi[::-1]
    torch.manual_seed(0)
    x = torch.randn(1, 3, 40, 52, dtype=torch.float64)
    lo, hi = R.afb1d_sym(x, dec_lo, dec_hi, 3)
    ll, lh = R.afb1d_sym(lo, dec_lo, dec_hi, 2)
    hl, hh = R.afb1d_sym(hi, dec_lo, dec_hi, 2)
    y = R.dwt_inverse(ll, [torch.stack([lh, hl, hh], 2)], rec_lo, rec_hi)
    assert y.shape == x.shape and _rel(y, x) < 1e-9
