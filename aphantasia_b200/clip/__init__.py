"""Drop-in for the OpenAI `clip` package as used by /root/reference/clip_fft.py (:19,119,121,133,150,216,254):
`clip.load(name, jit=False) -> (model, preprocess)`, `clip.tokenize`, `model.encode_image`, `model.encode_text`,
`model.visual.input_resolution`.

The image encoder (ViT-B/32, ViT-B/16) runs forward and data-gradient in libaphb200.so (csrc/vit.cu: tcgen05
GEMMs + fused kernels). Weights: an OpenAI state dict if `APH_CLIP_WEIGHTS=<file.pt>` is set, else seeded
synthetic weights of the same architecture (there are no CLIP weights or network in this environment).
The text encoder runs once before the optimisation loop and is not part of the hot path. With a state dict that
carries the text tower it runs in libaphb200.so (csrc/text.cu); without one, `encode_text` returns a deterministic
seeded embedding per prompt (loudly). `tokenize` is CLIP's byte-level BPE when `APH_CLIP_BPE=<bpe_simple_vocab_16e6.txt.gz>`
names the merges file, else a byte stand-in.
"""
import ctypes as C
import gzip
import hashlib
import html
import os
import re
import warnings
import zipfile
from collections import OrderedDict
from functools import lru_cache

import torch

from .. import _patchlink, _pool, _trace
from .._lib import TextConfig, VitConfig, check, lib, require_cuda, stream_ptr

_MODELS = {'ViT-B/32': dict(patch=32, width=768, layers=12, heads=12, out_dim=512, res=224),
           'ViT-B/16': dict(patch=16, width=768, layers=12, heads=12, out_dim=512, res=224)}


def available_models():
    return list(_MODELS)


def synthetic_visual_state_dict(patch=32, width=768, layers=12, heads=12, out_dim=512, res=224, seed=0):
    """Seeded synthetic weights in the OpenAI key layout, PyTorch-default-style init (private generator:
    the global RNG stream the sampler replays is left untouched)."""
    g = torch.Generator().manual_seed(seed)
    T = (res // patch) ** 2 + 1

    def uni(shape, bound):
        return (torch.rand(shape, generator=g) * 2 - 1) * bound

    def nrm(shape, std):
        return torch.randn(shape, generator=g) * std
    sd = OrderedDict()
    sd['visual.class_embedding'] = nrm((width,), width ** -0.5)
    sd['visual.positional_embedding'] = nrm((T, width), width ** -0.5)
    sd['visual.proj'] = nrm((width, out_dim), width ** -0.5)
    sd['visual.conv1.weight'] = uni((width, 3, patch, patch), (3 * patch * patch) ** -0.5)
    for n in ('ln_pre', 'ln_post'):
        sd['visual.%s.weight' % n] = torch.ones(width); sd['visual.%s.bias' % n] = torch.zeros(width)
    for i in range(layers):
        p = 'visual.transformer.resblocks.%d.' % i
        sd[p + 'attn.in_proj_weight'] = uni((3 * width, width), (6. / (4 * width)) ** 0.5)
        sd[p + 'attn.in_proj_bias'] = torch.zeros(3 * width)
        sd[p + 'attn.out_proj.weight'] = uni((width, width), width ** -0.5)
        sd[p + 'attn.out_proj.bias'] = torch.zeros(width)
        sd[p + 'ln_1.weight'] = torch.ones(width); sd[p + 'ln_1.bias'] = torch.zeros(width)
        sd[p + 'mlp.c_fc.weight'] = uni((4 * width, width), width ** -0.5)
        sd[p + 'mlp.c_fc.bias'] = uni((4 * width,), width ** -0.5)
        sd[p + 'mlp.c_proj.weight'] = uni((width, 4 * width), (4 * width) ** -0.5)
        sd[p + 'mlp.c_proj.bias'] = uni((width,), (4 * width) ** -0.5)
        sd[p + 'ln_2.weight'] = torch.ones(width); sd[p + 'ln_2.bias'] = torch.zeros(width)
    return sd


class _EncodeImage(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, vis, prepatched=False):
        require_cuda(x, 'encode_image input')
        xi = x.detach().contiguous().float()
        S = xi.shape[0]
        vis._ensure(S)
        emb = _pool.empty((S, vis.output_dim))
        need_bwd = x.requires_grad
        if prepatched:       # the sampler already wrote this batch as the conv1 operand (_patchlink): no k_patchify
            check(lib().aph_vit_fwd_prepatched(vis.handle, S, emb.data_ptr(), int(need_bwd), stream_ptr()), 'aph_vit_fwd_prepatched')
            vis.prepatched_forwards += 1
        else:
            vis._patch_gen += 1                 # k_patchify overwrites the operand buffer: outstanding stamps are void
            check(lib().aph_vit_fwd(vis.handle, xi.data_ptr(), S, emb.data_ptr(), int(need_bwd), stream_ptr()), 'aph_vit_fwd')
        _trace.encode()
        ctx.vis, ctx.S, ctx.shape = vis, S, tuple(xi.shape)
        if need_bwd:
            # The handle owns ONE activation arena: a later grad-tracked forward of the same model overwrites what this call
            # saved (clip_fft.py --enforce runs encode_image twice before loss.backward(), :254 and :276). Each saving forward
            # gets a generation stamp; a backward whose stamp is stale re-runs its forward from the saved input first
            # (deterministic kernels: identical activations), instead of silently using the other call's activations.
            vis._generation += 1
            ctx.generation = vis._generation
            ctx.handle_epoch = vis._handle_epoch
            ctx.save_for_backward(xi)
        return emb

    @staticmethod
    def backward(ctx, g):
        vis = ctx.vis
        xi, = ctx.saved_tensors
        g = g.contiguous().float()
        if ctx.generation != vis._generation or ctx.handle_epoch != vis._handle_epoch:
            vis._ensure(ctx.S)
            scratch = torch.empty(ctx.S, vis.output_dim, device=g.device, dtype=torch.float32)
            vis._patch_gen += 1
            check(lib().aph_vit_fwd(vis.handle, xi.data_ptr(), ctx.S, scratch.data_ptr(), 1, stream_ptr()), 'aph_vit_fwd (recompute)')
            vis._generation += 1            # the arena now belongs to this call; any other pending backward must recompute too
            vis.recomputes += 1
        gi = _pool.empty(ctx.shape)
        check(lib().aph_vit_bwd(vis.handle, g.data_ptr(), ctx.S, gi.data_ptr(), stream_ptr()), 'aph_vit_bwd')
        return gi, None, None


class VisionTransformer:
    """Handle-owning mirror of clip.model.VisionTransformer (forward only through the C ABI)."""

    def __init__(self, state_dict, max_batch=None):
        sd = {k[len('visual.'):]: v for k, v in state_dict.items() if k.startswith('visual.')}
        self.width = sd['conv1.weight'].shape[0]
        self.patch_size = sd['conv1.weight'].shape[-1]
        grid = round((sd['positional_embedding'].shape[0] - 1) ** 0.5)
        self.input_resolution = self.patch_size * grid
        self.layers = len([k for k in sd if k.endswith('.attn.in_proj_weight')])
        self.heads = self.width // 64
        self.output_dim = sd['proj'].shape[1]
        self._sd = {k: v.detach().float().contiguous() for k, v in sd.items()}
        self.handle, self.max_batch = None, 0
        self._generation, self.recomputes, self._handle_epoch = 0, 0, 0        # see _EncodeImage
        self._patch_gen, self._patch_written, self.prepatched_forwards = 0, False, 0      # see _patchlink
        _patchlink.register(self)
        if max_batch:
            self._ensure(max_batch)

    def _ensure(self, S):
        """(Re)creates the device handle so that its activation arena holds S samples."""
        if self.handle is not None and S <= self.max_batch:
            return
        self.close()
        cfg = VitConfig(self.patch_size, self.width, self.layers, self.heads, self.output_dim, self.input_resolution, int(S), 0)
        h = C.c_void_p()
        check(lib().aph_vit_create(C.byref(h), C.byref(cfg)), 'aph_vit_create')
        st = stream_ptr()
        for k, v in self._sd.items():
            d = v.cuda()
            check(lib().aph_vit_load_tensor(h, ('visual.' + k).encode(), d.data_ptr(), d.numel(), st), 'aph_vit_load_tensor(%s)' % k)
        torch.cuda.current_stream().synchronize()      # staging copies `d` die with this scope
        check(lib().aph_vit_finalize(h), 'aph_vit_finalize')
        self.handle, self.max_batch = h, int(S)
        self._handle_epoch += 1

    def close(self):
        if self.handle is not None:
            lib().aph_vit_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __call__(self, x):
        return _EncodeImage.apply(x, self, _patchlink.matches(x, self))


_TEXT_KEYS = ('token_embedding.', 'positional_embedding', 'transformer.', 'ln_final.', 'text_projection')


def has_text_tower(state_dict):
    return 'token_embedding.weight' in state_dict and 'text_projection' in state_dict


class TextTransformer:
    """Handle-owning text tower of clip.model.CLIP (forward only through the C ABI); geometry from the state-dict shapes."""

    def __init__(self, state_dict):
        sd = {k: v for k, v in state_dict.items() if k.startswith(_TEXT_KEYS)}
        self.vocab, self.width = sd['token_embedding.weight'].shape
        self.context_length = sd['positional_embedding'].shape[0]
        self.layers = len([k for k in sd if k.endswith('.attn.in_proj_weight')])
        self.heads = self.width // 64
        self.output_dim = sd['text_projection'].shape[1]
        self._sd = {k: v.detach().float().contiguous() for k, v in sd.items()}
        self.handle, self.max_batch = None, 0

    def _ensure(self, n):
        """(Re)creates the device handle so that its activation buffers hold n prompts."""
        if self.handle is not None and n <= self.max_batch:
            return
        self.close()
        cfg = TextConfig(self.width, self.layers, self.heads, self.context_length, self.vocab, self.output_dim, int(n))
        h = C.c_void_p()
        check(lib().aph_text_create(C.byref(h), C.byref(cfg)), 'aph_text_create')
        self.handle = h           # destroyed by close() if a load below fails
        st = stream_ptr()
        for k, v in self._sd.items():
            d = v.cuda()
            check(lib().aph_text_load_tensor(h, k.encode(), d.data_ptr(), d.numel(), st), 'aph_text_load_tensor(%s)' % k)
        torch.cuda.current_stream().synchronize()      # staging copies `d` die with this scope
        check(lib().aph_text_finalize(h), 'aph_text_finalize')
        self.max_batch = int(n)

    def close(self):
        if self.handle is not None:
            lib().aph_text_destroy(self.handle)
            self.handle, self.max_batch = None, 0

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __call__(self, tokens):
        if not (isinstance(tokens, torch.Tensor) and tokens.is_cuda and not tokens.is_floating_point() and not tokens.is_complex()
                and tokens.dtype != torch.bool):
            raise RuntimeError('aphantasia_b200: encode_text needs a CUDA integer tensor (clip.tokenize(...).cuda()); '
                               'this implementation has no CPU path')
        if tokens.dim() != 2 or tokens.shape[1] != self.context_length or tokens.shape[0] == 0:
            raise RuntimeError('aphantasia_b200: encode_text tokens must be [n, %d], got %s' % (self.context_length, tuple(tokens.shape)))
        ids = tokens.detach().to(torch.int64).contiguous()
        if bool(((ids < 0) | (ids >= self.vocab)).any()):
            raise RuntimeError('aphantasia_b200: encode_text token ids must lie in [0, %d)' % self.vocab)
        n = ids.shape[0]
        self._ensure(n)
        emb = torch.empty(n, self.output_dim, device=ids.device, dtype=torch.float32)
        check(lib().aph_text_fwd(self.handle, ids.data_ptr(), n, emb.data_ptr(), stream_ptr()), 'aph_text_fwd')
        return emb


class CLIP:
    """What clip_fft.py needs from clip.model.CLIP."""

    def __init__(self, name, state_dict, synthetic):
        self.name, self.synthetic = name, synthetic
        self.visual = VisionTransformer(state_dict)
        self.embed_dim = self.visual.output_dim
        self.text = TextTransformer(state_dict) if has_text_tower(state_dict) else None

    def encode_image(self, image):
        return self.visual(image)

    def encode_text(self, tokens):
        """The text tower on the GPU when the state dict carries it: tokens int [n, ctx] on CUDA -> fp32 [n, out].
        Otherwise a deterministic seeded stand-in per token row, unit norm x 10."""
        if self.text is not None:
            return self.text(tokens)
        dev = tokens.device
        digest = hashlib.sha256(tokens.detach().cpu().numpy().tobytes() + self.name.encode()).digest()
        g = torch.Generator().manual_seed(int.from_bytes(digest[:7], 'little'))
        emb = torch.randn(tokens.shape[0], self.embed_dim, generator=g)
        emb = 10. * emb / emb.norm(dim=-1, keepdim=True)
        return emb.to(dev)

    def eval(self):
        return self

    def cuda(self):
        return self

    def float(self):
        return self


def byte_symbols():
    """The 256 byte symbols of CLIP's byte-level BPE, in vocabulary order: bytes whose code point is a printable
    Latin-1 character ('!'..'~', '\xa1'..'\xac', '\xae'..'\xff') stand for themselves; the remaining 68 bytes, in
    increasing order, are shifted to U+0100 onwards so no symbol is whitespace or a control character.
    Returns {byte value: symbol} in that order."""
    direct = [b for b in range(256) if 0x21 <= b <= 0x7e or 0xa1 <= b <= 0xac or 0xae <= b <= 0xff]
    table = {b: chr(b) for b in direct}
    shifted = [b for b in range(256) if b not in table]
    table.update((b, chr(256 + i)) for i, b in enumerate(shifted))
    return table


# CLIP's pre-tokenizer: the two special tokens, English contractions, runs of letters, single digits, runs of other symbols
_SPLIT = r"""<\|startoftext\|>|<\|endoftext\|>|'s|'t|'re|'ve|'m|'ll|'d|[\p{L}]+|[\p{N}]|[^\s\p{L}\p{N}]+"""
_SOT, _EOT = '<|startoftext|>', '<|endoftext|>'
_MAX_MERGES = 49152 - 256 - 2        # the ViT-B vocabulary (49408 ids) uses the first 48894 merges of the file


class BPETokenizer:
    """CLIP's byte-level BPE, written from the published algorithm:
    html-unescape (twice) -> collapse whitespace -> lower-case -> split with CLIP's pattern -> map each word's UTF-8
    bytes to byte symbols (byte_symbols) -> merge adjacent symbol pairs by rank, the last symbol carrying '</w>'.
    Vocabulary ids: the 256 byte symbols, the same 256 with '</w>', one id per merge, then <|startoftext|>, <|endoftext|>.
    OpenAI's tokenizer also runs ftfy.fix_text first; ftfy is not a dependency here, so mojibake is not repaired."""

    def __init__(self, bpe_path):
        import regex
        with gzip.open(bpe_path, 'rt', encoding='utf-8') as f:
            lines = f.read().split('\n')[1:]                      # first line: header
        merges = [tuple(l.split()) for l in lines if l.strip()][:_MAX_MERGES]
        bad = [m for m in merges if len(m) != 2]
        if bad:
            raise RuntimeError('aphantasia_b200.clip: %s: malformed merge line %r' % (bpe_path, ' '.join(bad[0])))
        self.byte_sym = byte_symbols()
        vocab = list(self.byte_sym.values())
        vocab += [v + '</w>' for v in vocab]
        vocab += [a + b for a, b in merges]
        vocab += [_SOT, _EOT]
        self.encoder = {v: i for i, v in enumerate(vocab)}
        self.ranks = {m: i for i, m in enumerate(merges)}
        self.sot, self.eot = self.encoder[_SOT], self.encoder[_EOT]
        self.pattern = regex.compile(_SPLIT, regex.IGNORECASE)
        self.cache = {_SOT: (_SOT,), _EOT: (_EOT,)}

    def bpe(self, word):
        if word in self.cache:
            return self.cache[word]
        syms = list(word[:-1]) + [word[-1] + '</w>']
        while len(syms) > 1:
            pairs = [(self.ranks.get((a, b), len(self.ranks)), i) for i, (a, b) in enumerate(zip(syms, syms[1:]))]
            rank = min(pairs)[0]
            if rank == len(self.ranks):
                break
            first, second = next((syms[i], syms[i + 1]) for r, i in pairs if r == rank)
            out, i = [], 0
            while i < len(syms):                    # every non-overlapping occurrence, left to right
                if i + 1 < len(syms) and syms[i] == first and syms[i + 1] == second:
                    out.append(first + second); i += 2
                else:
                    out.append(syms[i]); i += 1
            syms = out
        self.cache[word] = tuple(syms)
        return self.cache[word]

    def encode(self, text):
        text = html.unescape(html.unescape(text)).strip()
        text = re.sub(r'\s+', ' ', text).strip().lower()
        ids = []
        for word in self.pattern.findall(text):
            word = ''.join(self.byte_sym[b] for b in word.encode('utf-8'))
            ids.extend(self.encoder[s] for s in self.bpe(word))
        return ids


@lru_cache(maxsize=4)
def _bpe_tokenizer(path):
    return BPETokenizer(path)


def bpe_path():
    """The merges file named by APH_CLIP_BPE, or None."""
    path = os.environ.get('APH_CLIP_BPE')
    if path and not os.path.isfile(path):
        raise RuntimeError('aphantasia_b200.clip: APH_CLIP_BPE=%s is not a file' % path)
    return path or None


def tokenize(texts, context_length=77, truncate=False):
    """clip.tokenize: LongTensor [n, context_length] = <|startoftext|>, BPE ids, <|endoftext|>, zero padding.
    A prompt longer than the context raises RuntimeError; with truncate=True it is cut and its last id is <|endoftext|>.
    Without APH_CLIP_BPE: a byte-level stand-in (start 49406, UTF-8 bytes, end 49407, zero padded, silently cut)."""
    if isinstance(texts, str):
        texts = [texts]
    out = torch.zeros(len(texts), context_length, dtype=torch.long)
    path = bpe_path()
    if path is None:
        for i, t in enumerate(texts):
            b = list(t.encode('utf-8'))[:context_length - 2]
            toks = [49406] + b + [49407]
            out[i, :len(toks)] = torch.tensor(toks)
        return out
    tok = _bpe_tokenizer(path)
    for i, t in enumerate(texts):
        toks = [tok.sot] + tok.encode(t) + [tok.eot]
        if len(toks) > context_length:
            if not truncate:
                raise RuntimeError('Input %s is too long for context length %d' % (t, context_length))
            toks = toks[:context_length]
            toks[-1] = tok.eot
        out[i, :len(toks)] = torch.tensor(toks)
    return out


_ARCHIVE_EXTRAS = ('input_resolution', 'context_length', 'vocab_size', 'logit_scale')


def load_state_dict(path):
    """An OpenAI CLIP checkpoint as a host fp32 state dict: either a plain state dict (torch.save) or the TorchScript
    archive OpenAI distributes (ViT-B-32.pt). The archive's input_resolution / context_length / vocab_size and logit_scale
    entries are dropped; fp16 tensors become fp32."""
    scripted = False
    if zipfile.is_zipfile(path):
        with zipfile.ZipFile(path) as z:
            scripted = any(n.endswith('/constants.pkl') or n == 'constants.pkl' for n in z.namelist())
    if scripted:
        with warnings.catch_warnings():
            warnings.simplefilter('ignore', DeprecationWarning)       # torch.jit.load is the only reader of this format
            sd = torch.jit.load(path, map_location='cpu').state_dict()
    else:
        sd = torch.load(path, map_location='cpu')
        if hasattr(sd, 'state_dict'):
            sd = sd.state_dict()
    return OrderedDict((k, v.float() if v.is_floating_point() else v) for k, v in sd.items() if k not in _ARCHIVE_EXTRAS)


def load(name, device=None, jit=False, download_root=None):
    """clip.load: returns (model, preprocess). `preprocess` is unused by the scripts (None)."""
    if name not in _MODELS:
        raise RuntimeError('aphantasia_b200.clip: model %s not available (B200 hot path covers %s)' % (name, available_models()))
    path = os.environ.get('APH_CLIP_WEIGHTS_' + name.replace('/', '').replace('-', '').upper(), os.environ.get('APH_CLIP_WEIGHTS'))
    if path and os.path.isfile(path):
        sd = load_state_dict(path)
        synthetic = False
        bpe = bpe_path()
        print(' [aphantasia_b200.clip] %s: weights real (%s); text tower %s; tokenizer %s'
              % (name, path, 'real' if has_text_tower(sd) else 'absent (seeded text embeddings)',
                 'BPE (%s)' % bpe if bpe else 'byte stand-in'))
        if not bpe:
            warnings.warn('aphantasia_b200.clip: real CLIP weights but APH_CLIP_BPE is not set: prompts are BYTE-tokenized, '
                          'so text embeddings do not mean what the prompt says. Point APH_CLIP_BPE at bpe_simple_vocab_16e6.txt.gz.',
                          RuntimeWarning, stacklevel=2)
    else:
        sd = synthetic_visual_state_dict(seed=int(os.environ.get('APH_CLIP_SEED', '0')), **_MODELS[name])
        synthetic = True
        print(' [aphantasia_b200.clip] no CLIP weights available: using seeded synthetic %s weights and seeded text embeddings' % name)
    return CLIP(name, sd, synthetic), None
