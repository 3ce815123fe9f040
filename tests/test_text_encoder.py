"""CLIP text side: the BPE tokenizer, the text-tower restatement, checkpoint loading (CPU) and the CUDA text tower (GPU).

The tokenizer is checked against HuggingFace's independent CLIPTokenizer on a small merge table learned here, and on a
hand-written table with known ids. The oracle text tower is checked against HuggingFace CLIPTextModelWithProjection;
the GPU tower against the oracle. No OpenAI weights or vocabulary are involved: semantic quality is not tested here.
"""
import gzip
import importlib.util
import json
import os
import warnings
from collections import Counter, OrderedDict

import numpy as np
import pytest
import torch


def _load_text_oracle():
    spec = importlib.util.spec_from_file_location('text_oracle', os.path.join(os.path.dirname(os.path.abspath(__file__)), 'text_oracle.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


TO = _load_text_oracle()       # the CPU text-tower restatement (tests/text_oracle.py)

CORPUS = ("a red square on a blue sky. the red cat sat on the square mat; it's a photo of a cat, a photo of the sky! "
          "red red square square blue sky sky photo photo cat cat 2024 1st. the quick brown fox jumps over the lazy dog; "
          "painting of a forest at night, photograph of mountains and rivers, drawing of flowers.")


def _rel(a, b):
    a = torch.as_tensor(a.detach().cpu() if torch.is_tensor(a) else a).double()
    b = torch.as_tensor(b.detach().cpu() if torch.is_tensor(b) else b).double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def _learn_merges(corpus, n):
    """Plain BPE training on the pre-tokenized corpus: n times, merge the most frequent adjacent pair (ties: smallest pair)."""
    import regex
    from aphantasia_b200 import clip
    sym = clip.byte_symbols()
    words = Counter(regex.findall(clip._SPLIT, corpus.lower(), regex.IGNORECASE))
    seqs = {}
    for w, c in words.items():
        s = [sym[b] for b in w.encode('utf-8')]
        seqs[tuple(s[:-1] + [s[-1] + '</w>'])] = c
    merges = []
    for _ in range(n):
        pairs = Counter()
        for s, c in seqs.items():
            for p in zip(s, s[1:]):
                pairs[p] += c
        if not pairs:
            break
        best = min(pairs, key=lambda p: (-pairs[p], p))
        merges.append(best)
        out = {}
        for s, c in seqs.items():
            t, i = [], 0
            while i < len(s):
                if i + 1 < len(s) and (s[i], s[i + 1]) == best:
                    t.append(s[i] + s[i + 1]); i += 2
                else:
                    t.append(s[i]); i += 1
            out[tuple(t)] = c
        seqs = out
    return merges


def _write_bpe(tmp_path, merges):
    """The merges as OpenAI's gzip file, plus HuggingFace vocab.json / merges.txt with the same id order."""
    from aphantasia_b200 import clip
    lines = ['#version: 0.2'] + ['%s %s' % m for m in merges]
    gz = tmp_path / 'bpe.txt.gz'
    with gzip.open(gz, 'wt', encoding='utf-8') as f:
        f.write('\n'.join(lines) + '\n')
    vocab = list(clip.byte_symbols().values())
    vocab += [v + '</w>' for v in vocab]
    vocab += [a + b for a, b in merges] + ['<|startoftext|>', '<|endoftext|>']
    (tmp_path / 'vocab.json').write_text(json.dumps({v: i for i, v in enumerate(vocab)}), encoding='utf-8')
    (tmp_path / 'merges.txt').write_text('\n'.join(lines) + '\n', encoding='utf-8')
    return str(gz), len(vocab)


@pytest.fixture
def learned_bpe(tmp_path, monkeypatch):
    merges = _learn_merges(CORPUS, 30)
    assert len(merges) == 30
    gz, vocab = _write_bpe(tmp_path, merges)
    monkeypatch.setenv('APH_CLIP_BPE', gz)
    return tmp_path, gz, vocab


# ------------------------------------------------------------------------------------------------------ tokenizer (CPU)
def test_tokenizer_matches_huggingface(learned_bpe):
    pytest.importorskip('transformers')
    from transformers import CLIPTokenizer
    from aphantasia_b200 import clip
    d, _, vocab = learned_bpe
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        hf = CLIPTokenizer(str(d / 'vocab.json'), str(d / 'merges.txt'))
    for text in ['red square', "It's a photo of a CAT!", 'blue sky:0.5', '2024 was the 1st', 'red   \t square \n on  sky', '']:
        want = hf(text)['input_ids']
        got = clip.tokenize(text)[0]
        assert got[:len(want)].tolist() == want, text
        assert not got[len(want):].any(), text
    assert hf('red square')['input_ids'][0] == vocab - 2 and hf('')['input_ids'] == [vocab - 2, vocab - 1]
    long = ' '.join(['photo of the red cat'] * 20)
    with pytest.raises(RuntimeError, match='too long'):
        clip.tokenize(long)
    want = hf(long, max_length=77, truncation=True)['input_ids']
    got = clip.tokenize(long, truncate=True)[0]
    assert len(want) == 77 and got.tolist() == want and got[-1].item() == vocab - 1


def test_tokenizer_known_answer(tmp_path, monkeypatch):
    """Three merges written by hand; byte ids follow the published byte order ('!' = 0, ..., '~' = 93, U+00A1 = 94 ...)."""
    from aphantasia_b200 import clip
    gz, vocab = _write_bpe(tmp_path, [('r', 'e'), ('re', 'd</w>'), ('q', 'u')])
    monkeypatch.setenv('APH_CLIP_BPE', gz)
    assert vocab == 517
    SOT, EOT = 515, 516
    cases = {
        'red square': [SOT, 513, ord('s') - 33, 514, ord('a') - 33, ord('r') - 33, 256 + ord('e') - 33, EOT],
        'RED': [SOT, 513, EOT],
        '&amp;': [SOT, 256 + ord('&') - 33, EOT],                                  # html-unescaped to '&'
        'é': [SOT, 94 + 12 + (0xc3 - 0xae), 256 + 94 + (0xa9 - 0xa1), EOT],           # UTF-8 c3 a9
        "red's": [SOT, 513, ord("'") - 33, 256 + ord('s') - 33, EOT],
        '  ': [SOT, EOT],
    }
    for text, want in cases.items():
        got = clip.tokenize(text)[0]
        assert got[:len(want)].tolist() == want, text
        assert not got[len(want):].any(), text
    out = clip.tokenize(['red', 'qu'], context_length=5)
    assert out.dtype == torch.long and out.tolist() == [[SOT, 513, EOT, 0, 0], [SOT, ord('q') - 33, 256 + ord('u') - 33, EOT, 0]]   # 'q' 'u</w>': the merge q+u does not apply
    with pytest.raises(RuntimeError):
        clip.tokenize('square', context_length=5)          # SOT s qu a r e</w> EOT: 7 ids
    assert clip.tokenize('square', context_length=5, truncate=True)[0].tolist() == [SOT, ord('s') - 33, 514, ord('a') - 33, EOT]


def test_tokenizer_without_bpe_keeps_the_byte_stand_in(monkeypatch):
    from aphantasia_b200 import clip
    monkeypatch.delenv('APH_CLIP_BPE', raising=False)
    t = clip.tokenize('ab')[0]
    assert t[:4].tolist() == [49406, 97, 98, 49407] and not t[4:].any()


# ---------------------------------------------------------------------------------------------------- oracle (CPU)
def _token_rows(n, ctx, vocab, seed, lengths=None):
    """SOT, content ids < SOT, EOT (the largest id), zero padding. Row 0: SOT EOT; row 1: full, EOT at ctx - 1; rest random."""
    g = torch.Generator().manual_seed(seed)
    sot, eot = vocab - 2, vocab - 1
    rows = torch.zeros(n, ctx, dtype=torch.long)
    for i in range(n):
        L = lengths[i] if lengths else (0 if i == 0 else ctx - 2 if i == 1 else int(torch.randint(1, ctx - 2, (1,), generator=g)))
        rows[i, 0] = sot
        rows[i, 1:1 + L] = torch.randint(0, sot, (L,), generator=g)
        rows[i, 1 + L] = eot
    return rows


def test_text_restatement_matches_hf():
    """OpenAI-layout text tower restatement vs the independent HuggingFace CLIP text tower (tiny geometry)."""
    pytest.importorskip('transformers')
    from transformers import CLIPTextConfig, CLIPTextModelWithProjection
    width, layers, heads, ctx, vocab, out = 128, 2, 2, 20, 100, 64
    sd = TO.synthetic_text_state_dict(3, width, layers, heads, ctx, vocab, out)
    txt = TO.build_text(sd)
    cfg = CLIPTextConfig(vocab_size=vocab, hidden_size=width, intermediate_size=4 * width, num_hidden_layers=layers,
                         num_attention_heads=heads, max_position_embeddings=ctx, hidden_act='quick_gelu', layer_norm_eps=1e-5,
                         projection_dim=out, bos_token_id=vocab - 2, eos_token_id=vocab - 1, pad_token_id=0,
                         attn_implementation='eager')
    hf = CLIPTextModelWithProjection(cfg).eval()
    t = hf.text_model
    with torch.no_grad():
        t.embeddings.token_embedding.weight.copy_(sd['token_embedding.weight'])
        t.embeddings.position_embedding.weight.copy_(sd['positional_embedding'])
        t.final_layer_norm.weight.copy_(sd['ln_final.weight']); t.final_layer_norm.bias.copy_(sd['ln_final.bias'])
        hf.text_projection.weight.copy_(sd['text_projection'].T)
        for i, l in enumerate(t.encoder.layers):
            pre = 'transformer.resblocks.%d.' % i
            wq, wk, wv = sd[pre + 'attn.in_proj_weight'].chunk(3); bq, bk, bv = sd[pre + 'attn.in_proj_bias'].chunk(3)
            l.self_attn.q_proj.weight.copy_(wq); l.self_attn.q_proj.bias.copy_(bq)
            l.self_attn.k_proj.weight.copy_(wk); l.self_attn.k_proj.bias.copy_(bk)
            l.self_attn.v_proj.weight.copy_(wv); l.self_attn.v_proj.bias.copy_(bv)
            l.self_attn.out_proj.weight.copy_(sd[pre + 'attn.out_proj.weight']); l.self_attn.out_proj.bias.copy_(sd[pre + 'attn.out_proj.bias'])
            l.layer_norm1.weight.copy_(sd[pre + 'ln_1.weight']); l.layer_norm1.bias.copy_(sd[pre + 'ln_1.bias'])
            l.layer_norm2.weight.copy_(sd[pre + 'ln_2.weight']); l.layer_norm2.bias.copy_(sd[pre + 'ln_2.bias'])
            l.mlp.fc1.weight.copy_(sd[pre + 'mlp.c_fc.weight']); l.mlp.fc1.bias.copy_(sd[pre + 'mlp.c_fc.bias'])
            l.mlp.fc2.weight.copy_(sd[pre + 'mlp.c_proj.weight']); l.mlp.fc2.bias.copy_(sd[pre + 'mlp.c_proj.bias'])
    ids = _token_rows(4, ctx, vocab, 5)
    with torch.no_grad():
        a = txt(ids)
        b = hf(input_ids=ids).text_embeds
    assert a.shape == (4, out)
    assert _rel(a, b) < 1e-5


def test_oracle_text_rng_restored_and_mask_is_causal():
    g = torch.random.get_rng_state()
    TO.synthetic_text_state_dict(0, 128, 1, 2, 16, 50, 128)
    assert torch.equal(g, torch.random.get_rng_state())
    blk = TO.CausalResidualAttentionBlock(128, 2, TO.causal_mask(4))
    assert blk.attn_mask[0].tolist() == [0., float('-inf'), float('-inf'), float('-inf')] and blk.attn_mask[3].eq(0).all()
    assert not any('attn_mask' in k for k in blk.state_dict())


# --------------------------------------------------------------------------------------------- checkpoint loading (CPU)
def _full_state_dict(vocab, seed=0):
    """Tiny full OpenAI-layout checkpoint: visual (width 128, res 64, patch 32) + text (width 256, ctx 77) + logit_scale."""
    from aphantasia_b200 import clip
    sd = OrderedDict(clip.synthetic_visual_state_dict(patch=32, width=128, layers=1, heads=2, out_dim=128, res=64, seed=seed))
    sd.update(TO.synthetic_text_state_dict(seed + 1, 256, 2, 4, 77, vocab, 128))
    sd['logit_scale'] = torch.tensor(4.6052)
    return sd


def _save_archive(sd, path):
    """A TorchScript archive whose state_dict() has the given keys, like OpenAI's distributed checkpoints."""
    root = torch.nn.Module()
    for k, v in sd.items():
        *mods, leaf = k.split('.')
        m = root
        for name in mods:
            if name not in m._modules:
                m.add_module(name, torch.nn.Module())
            m = m._modules[name]
        m.register_buffer(leaf, v)
    torch.jit.save(torch.jit.script(root), str(path))


@pytest.mark.parametrize('fmt', ['torchscript', 'fp16_state_dict'])
def test_load_openai_checkpoint_formats(tmp_path, monkeypatch, fmt):
    from aphantasia_b200 import clip
    sd = _full_state_dict(600)
    half = OrderedDict((k, v.half() if v.is_floating_point() else v) for k, v in sd.items())
    path = tmp_path / 'ViT-B-32.pt'
    if fmt == 'torchscript':
        extra = OrderedDict(half)
        extra['input_resolution'] = torch.tensor(64); extra['context_length'] = torch.tensor(77); extra['vocab_size'] = torch.tensor(600)
        _save_archive(extra, path)
        with pytest.raises(RuntimeError):
            torch.load(path, map_location='cpu')          # the plain loader cannot read the archive
    else:
        torch.save(half, path)
    monkeypatch.setenv('APH_CLIP_WEIGHTS', str(path))
    monkeypatch.delenv('APH_CLIP_BPE', raising=False)
    got = clip.load_state_dict(str(path))
    assert sorted(got) == sorted(k for k in half if k != 'logit_scale')
    for k, v in got.items():
        assert v.dtype == torch.float32 and torch.equal(v, half[k].float()), k
    with pytest.warns(RuntimeWarning, match='BYTE-tokenized'):
        model, _ = clip.load('ViT-B/32')
    assert not model.synthetic and model.text is not None and model.text.handle is None      # no GPU work yet
    assert (model.text.width, model.text.layers, model.text.context_length, model.text.vocab, model.text.output_dim) == (256, 2, 77, 600, 128)
    assert model.visual.input_resolution == 64 and model.embed_dim == 128


def test_visual_only_weights_keep_the_seeded_text_stand_in(tmp_path, monkeypatch):
    from aphantasia_b200 import clip
    sd = clip.synthetic_visual_state_dict(patch=32, width=128, layers=1, heads=2, out_dim=128, res=64)
    path = tmp_path / 'visual.pt'
    torch.save(sd, path)
    monkeypatch.setenv('APH_CLIP_WEIGHTS', str(path))
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        model, _ = clip.load('ViT-B/32')
    assert model.text is None
    a = model.encode_text(torch.zeros(2, 77, dtype=torch.long))
    assert a.shape == (2, 128) and torch.allclose(a.norm(dim=-1), torch.full((2,), 10.))


# ------------------------------------------------------------------------------------------------------ GPU text tower
def _gpu_tower(sd):
    from aphantasia_b200 import clip
    return clip.TextTransformer(sd)


@pytest.mark.gpu
@pytest.mark.parametrize('geom,n', [((512, 12, 8, 77, 49408, 512), 1), ((512, 12, 8, 77, 49408, 512), 5), ((256, 2, 4, 77, 600, 128), 3)])
def test_text_tower_vs_oracle(geom, n):
    width, layers, heads, ctx, vocab, out = geom
    sd = TO.synthetic_text_state_dict(7, width, layers, heads, ctx, vocab, out)
    ids = _token_rows(n, ctx, vocab, 11 + n)
    with torch.no_grad():
        want = TO.build_text(sd)(ids)
    tower = _gpu_tower(sd)
    got = tower(ids.cuda())
    torch.cuda.synchronize()
    assert got.dtype == torch.float32 and got.shape == (n, out)
    assert _rel(got, want) < 2e-2
    got2 = tower(ids.cuda().int())                     # int32 ids are accepted too; same result
    assert torch.equal(got, got2)
    for bad in (ids.cuda()[:, :ctx - 1], ids.float().cuda(), ids):
        with pytest.raises(RuntimeError):
            tower(bad)
    oob = ids.clone(); oob[0, 3] = vocab
    with pytest.raises(RuntimeError, match='lie in'):
        tower(oob.cuda())
    tower.close()


@pytest.mark.gpu
def test_text_tower_is_causal():
    width, layers, heads, ctx, vocab, out = 256, 2, 4, 77, 600, 128
    sd = TO.synthetic_text_state_dict(9, width, layers, heads, ctx, vocab, out)
    tower = _gpu_tower(sd)
    ids = _token_rows(3, ctx, vocab, 21, lengths=[5, 30, 60])
    base = tower(ids.cuda())
    for s, L in enumerate([5, 30, 60]):
        after = ids.clone()
        after[s, L + 2:] = (after[s, L + 2:] + 17) % (vocab - 2)          # every id after this row's EOT
        assert torch.equal(tower(after.cuda()), base), s
        before = ids.clone()
        before[s, 1 + L // 2] = (before[s, 1 + L // 2] + 1) % (vocab - 2)   # one id before EOT
        changed = tower(before.cuda())
        assert not torch.equal(changed[s], base[s]), s
        others = [i for i in range(3) if i != s]
        assert torch.equal(changed[others], base[others])
    tower.close()


@pytest.mark.gpu
def test_script_prompt_path_end_to_end(tmp_path, monkeypatch, learned_bpe):
    """clip.load + the enc_text loop of clip_fft.py (split on '|', weight after ':') with real-layout weights and BPE."""
    from aphantasia_b200 import clip
    _, _, vocab = learned_bpe
    sd = _full_state_dict(vocab, seed=4)
    path = tmp_path / 'full.pt'
    torch.save(sd, path)
    monkeypatch.setenv('APH_CLIP_WEIGHTS', str(path))
    model_clip, _ = clip.load('ViT-B/32')
    assert model_clip.text is not None

    def enc_text(txt):                                   # clip_fft.py enc_text
        embs = []
        for subtxt in txt.split('|'):
            if ':' in subtxt:
                [subtxt, wt] = subtxt.split(':')
                wt = float(wt)
            else:
                wt = 1.
            emb = model_clip.encode_text(clip.tokenize(subtxt).cuda())
            embs.append([emb.detach().clone(), wt])
        return embs

    embs = enc_text('red square|blue sky:0.5')
    assert [wt for _, wt in embs] == [1., 0.5]
    try:                                                 # the prompt ids from the independent tokenizer where available
        from transformers import CLIPTokenizer
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            hf = CLIPTokenizer(str(tmp_path / 'vocab.json'), str(tmp_path / 'merges.txt'))

        def tok(t):
            ids = hf(t)['input_ids']
            out = torch.zeros(1, 77, dtype=torch.long)
            out[0, :len(ids)] = torch.tensor(ids)
            return out
    except ImportError:
        tok = clip.tokenize
    oracle = TO.build_text(sd)
    for (emb, _), sub in zip(embs, ['red square', 'blue sky']):
        ids = tok(sub)
        assert torch.equal(ids, clip.tokenize(sub))
        with torch.no_grad():
            want = oracle(ids)
        assert emb.shape == (1, 128) and _rel(emb, want) < 2e-2, sub
    # the image side still works on the same model
    img = torch.rand(2, 3, 64, 64, device='cuda')
    assert model_clip.encode_image(img).shape == (2, 128)
