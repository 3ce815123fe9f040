"""Generates the committed golden fixtures from the REAL reference (/root/reference), build container only.

    python tests/golden/make_golden.py

Every array below is produced by executing the reference's own modules (oracle/ref_import.py loads them
in place; nothing is copied) with explicit seeds. The reference has no tests / golden vectors of its own
(SURVEY.md section 4), so these fixtures are what pins the oracle (oracle/restate.py) and the host logic
(aphantasia_b200/_rng.py). Fixtures are kept small (sub-sampled where needed).
"""
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F
import torchvision.transforms.functional as TF

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref_import  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
ref = ref_import.load()


def seed(s):
    torch.manual_seed(s); np.random.seed(s)


def capture_slice(canvas_hw, count, size, transform, align, macro, s):
    """Runs the reference slice_imgs on an index-image canvas, recording the parameters it used."""
    H, W = canvas_hw
    yy, xx = torch.meshgrid(torch.arange(H, dtype=torch.float32), torch.arange(W, dtype=torch.float32), indexing='ij')
    canvas = torch.stack([yy, xx, torch.zeros_like(yy)])[None]
    rec = []
    cur = {}
    o_interp, o_persp, o_erase, o_affine = F.interpolate, TF.perspective, TF.erase, TF.affine

    def interp(x, *a, **k):
        cur.clear()
        cur.update(offy=float(x[0, 0, 0, 0]), offx=float(x[0, 1, 0, 0]), csize=x.shape[-1], persp=None, erase=None, angle=None)
        rec.append(cur.copy())
        return o_interp(x, *a, **k)

    def persp(img, startpoints, endpoints, *a, **k):
        rec[-1]['persp'] = (startpoints, endpoints)
        return o_persp(img, startpoints, endpoints, *a, **k)

    def erase(img, i, j, h, w, v, *a, **k):
        rec[-1]['erase'] = (i, j, h, w)
        return o_erase(img, i, j, h, w, v, *a, **k)

    def affine(img, angle, *a, **k):
        rec[-1]['angle'] = angle
        return o_affine(img, angle, *a, **k)

    F.interpolate, TF.perspective, TF.erase, TF.affine = interp, persp, erase, affine
    # torchvision's transform classes look these up through the `F` alias of the functional module
    import torchvision.transforms.transforms as TT
    TT.F.perspective, TT.F.erase = persp, erase
    try:
        seed(s)
        ref.utils.slice_imgs([canvas], count, size, transform, align, macro)
        state_after = (torch.rand(1).item(), float(np.random.rand()))
    finally:
        F.interpolate, TF.perspective, TF.erase, TF.affine = o_interp, o_persp, o_erase, o_affine
        TT.F.perspective, TT.F.erase = o_persp, o_erase
    n = len(rec)
    arr = np.zeros((n, 24), np.float32)
    for c, r in enumerate(rec):
        arr[c, 0:3] = (r['offy'], r['offx'], r['csize'])
        if r['persp'] is not None:
            arr[c, 3] += 1
            arr[c, 4:12] = TF._get_perspective_coeffs(*r['persp'])
        if r['erase'] is not None and tuple(r['erase']) != (0, 0, size, size):
            arr[c, 3] += 2
            arr[c, 12:16] = r['erase']
        if r['angle'] is not None:
            arr[c, 3] += 4
            m = TF._get_inverse_affine_matrix([0., 0.], r['angle'], [0., 0.], 1., [0., 0.])
            arr[c, 16:20] = (m[0], m[1], m[3], m[4])
            arr[c, 20] = r['angle']
        else:
            arr[c, 16:20] = (1, 0, 0, 1)
    return arr, np.array(state_after, np.float64)


def main():
    g = {}
    # ---- 1. RNG / parameter replay (host logic) -------------------------------------------------
    fast, norm = ref.transforms.transforms_fast, ref.transforms.normalize()
    cases = [('c2', (720, 1280), 190, 224, fast, 'uniform', 0.4, 123),
             ('c1', (224, 224), 3, 224, fast, 'uniform', 0.4, 0),
             ('central', (300, 420), 16, 224, fast, 'central', 0.4, 7),
             ('norm', (256, 256), 9, 224, norm, 'uniform', 0., 3),
             ('overscan', (240, 320), 12, 224, fast, 'overscan', 0.4, 11),
             ('small', (64, 96), 8, 32, fast, 'uniform', 0.5, 5)]
    for name, hw, cnt, size, tf, align, macro, s in cases:
        arr, st = capture_slice(hw, cnt, size, tf, align, macro, s)
        g['rng_%s_table' % name] = arr
        g['rng_%s_after' % name] = st
        g['rng_%s_cfg' % name] = np.array([hw[0], hw[1], cnt, size, 2 if tf is fast else 1, macro, s], np.float64)
        g['rng_%s_align' % name] = np.array(align)

    # ---- 2. FFT synthesis + to_valid_rgb (forward values and gradients) --------------------------
    for name, (h, w), decay, colors, contrast, s in [('even', (24, 20), 1.5, 1.8, 1.0, 1), ('odd', (15, 21), 1.0, 1.0, 1.1, 2),
                                                      ('sq', (32, 32), 1.5, 1.8, 1.0, 3)]:
        seed(s)
        params, image_f, _ = ref.image.fft_image([1, 3, h, w], 0.07, decay, None)
        rgb_f = ref.image.to_valid_rgb(image_f, colors=colors)
        raw = image_f(contrast=contrast)
        rgb = rgb_f(contrast=contrast)
        cot = torch.randn(rgb.shape)
        (rgb * cot).sum().backward()
        g['fft_%s_params' % name] = params[0].detach().numpy()
        g['fft_%s_cfg' % name] = np.array([h, w, decay, colors, contrast], np.float64)
        g['fft_%s_img' % name] = raw.detach().numpy()
        g['fft_%s_rgb' % name] = rgb.detach().numpy()
        g['fft_%s_cot' % name] = cot.numpy()
        g['fft_%s_grad' % name] = params[0].grad.numpy().copy()
        # shift ("--noise") variant, forward only
        params[0].grad = None
        shift = torch.rand(1, 1, h, w // 2 + 1, 1) * 0.05
        g['fft_%s_shift' % name] = shift.numpy()
        g['fft_%s_rgb_shift' % name] = rgb_f(shift, contrast).detach().numpy()

    # ---- 3. sampler: values + canvas gradient on a small frame (full tensors), and a 224 case (subsampled)
    for name, hw, cnt, size, align, macro, s, sub in [('small', (64, 96), 8, 32, 'uniform', 0.5, 5, 1),
                                                       ('mid', (230, 260), 6, 224, 'uniform', 0.4, 9, 7),
                                                       ('over', (80, 120), 6, 32, 'overscan', 0.4, 13, 1)]:
        seed(100 + s)
        canvas = torch.rand(1, 3, *hw).half().float().requires_grad_(True)   # stored as its seed: the tests redraw it
        seed(s)
        out = ref.utils.slice_imgs([canvas], cnt, size, fast, align, macro)[0]
        seed(200 + s)
        cot = torch.randn(out.shape)
        (out * cot).sum().backward()
        g['smp_%s_canvas_seed' % name] = np.array(100 + s)
        g['smp_%s_cfg' % name] = np.array([hw[0], hw[1], cnt, size, macro, s, sub], np.float64)
        g['smp_%s_align' % name] = np.array(align)
        g['smp_%s_out' % name] = out.detach().numpy()[:, :, ::sub, ::sub]
        g['smp_%s_cot_seed' % name] = np.array(200 + s)
        g['smp_%s_gcanvas' % name] = canvas.grad.numpy()[:, :, ::max(1, sub // 2), ::max(1, sub // 2)]
        g['smp_%s_gsum' % name] = np.array([canvas.grad.double().sum().item(), canvas.grad.double().abs().sum().item()])

    # ---- 4. sim_func --------------------------------------------------------------------------
    seed(4)
    v1 = torch.randn(1, 512); v2 = torch.randn(7, 512, requires_grad=True)
    for t in (None, 'mix', 'cossim', 'ang', 'dot'):
        v2.grad = None
        val = ref.utils.sim_func(v1, v2, t)
        val.backward()
        g['sim_%s_val' % t] = val.detach().numpy()
        g['sim_%s_grad' % t] = v2.grad.numpy().copy()
    g['sim_spher_val'] = ref.utils.sim_func(v1, v2, 'spher').detach().numpy()
    g['sim_v1'] = v1.numpy(); g['sim_v2'] = v2.detach().numpy()

    # ---- 5. whole chain: params -> rgb -> crops -> fixed linear "encoder" -> mix loss -> d params --
    seed(21)
    h, w = 48, 64
    params, image_f, _ = ref.image.fft_image([1, 3, h, w], 0.07, 1.5, None)
    rgb_f = ref.image.to_valid_rgb(image_f, colors=1.8)
    seed(22)
    proj = torch.randn(3 * 32 * 32, 64) / 55.
    txt = torch.randn(1, 64)
    seed(23)
    crops = ref.utils.slice_imgs([rgb_f()], 5, 32, fast, 'uniform', 0.4)[0]
    emb = crops.reshape(5, -1) @ proj
    loss = -ref.utils.sim_func(txt, emb, 'mix')
    loss.backward()
    g['chain_params'] = params[0].detach().numpy()
    g['chain_loss'] = loss.detach().numpy()
    g['chain_grad'] = params[0].grad.numpy().copy()
    g['chain_emb'] = emb.detach().numpy()

    path = os.path.join(OUT, 'reference_golden.npz')
    np.savez_compressed(path, **g)
    print('wrote', path, os.path.getsize(path) // 1024, 'KiB,', len(g), 'arrays')


if __name__ == '__main__':
    main()
