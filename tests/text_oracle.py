"""CPU restatement of the CLIP text encoder -- TEST INFRASTRUCTURE ONLY (never imported by the product).

Restates OpenAI clip/model.py (third-party `clip` 1.0, not in the reference tree; cited by function): CLIP.__init__ (the
text-tower modules), CLIP.initialize_parameters, CLIP.build_attention_mask (-inf strictly above the diagonal) and
CLIP.encode_text. Built from the image-encoder restatement's blocks in oracle/restate.py (LayerNorm, QuickGELU MLP,
nn.MultiheadAttention), with the causal mask added by a subclass. Parity: cross-checked at test time against the independent
HuggingFace CLIPTextModelWithProjection (tests/test_text_encoder.py) -> pinned w.r.t. HF, unpinned w.r.t. OpenAI weights.
"""
from collections import OrderedDict

import torch
import torch.nn as nn

from oracle import restate as R

TEXT_KEYS = ('token_embedding.', 'positional_embedding', 'transformer.', 'ln_final.', 'text_projection')


def causal_mask(ctx):
    """CLIP.build_attention_mask: additive [ctx, ctx] mask, -inf where key j > query i."""
    return torch.empty(ctx, ctx).fill_(float('-inf')).triu_(1)


class CausalResidualAttentionBlock(R.ResidualAttentionBlock):
    """The image encoder's block with an attention mask (a plain attribute, not part of the state dict)."""

    def __init__(self, d_model, n_head, attn_mask):
        super().__init__(d_model, n_head)
        self.attn_mask = attn_mask

    def forward(self, x):
        y = self.ln_1(x)
        x = x + self.attn(y, y, y, need_weights=False, attn_mask=self.attn_mask)[0]
        return x + self.mlp(self.ln_2(x))


class CausalTransformer(nn.Module):
    def __init__(self, width, layers, heads, attn_mask):
        super().__init__()
        self.resblocks = nn.Sequential(*[CausalResidualAttentionBlock(width, heads, attn_mask) for _ in range(layers)])

    def forward(self, x):
        return self.resblocks(x)


class TextTransformer(nn.Module):
    def __init__(self, width=512, layers=12, heads=8, context_length=77, vocab_size=49408, output_dim=512):
        super().__init__()
        self.context_length = context_length
        self.transformer = CausalTransformer(width, layers, heads, causal_mask(context_length))
        self.token_embedding = nn.Embedding(vocab_size, width)
        self.positional_embedding = nn.Parameter(torch.empty(context_length, width))
        self.ln_final = R.LayerNorm(width)
        self.text_projection = nn.Parameter(torch.empty(width, output_dim))
        nn.init.normal_(self.token_embedding.weight, std=0.02)                          # initialize_parameters
        nn.init.normal_(self.positional_embedding, std=0.01)
        proj_std = (width ** -0.5) * ((2 * layers) ** -0.5)
        attn_std, fc_std = width ** -0.5, (2 * width) ** -0.5
        for b in self.transformer.resblocks:
            nn.init.normal_(b.attn.in_proj_weight, std=attn_std)
            nn.init.normal_(b.attn.out_proj.weight, std=proj_std)
            nn.init.normal_(b.mlp.c_fc.weight, std=fc_std)
            nn.init.normal_(b.mlp.c_proj.weight, std=proj_std)
        nn.init.normal_(self.text_projection, std=width ** -0.5)

    def forward(self, text):
        x = self.token_embedding(text) + self.positional_embedding                          # encode_text
        x = self.transformer(x.permute(1, 0, 2)).permute(1, 0, 2)
        x = self.ln_final(x)
        return x[torch.arange(x.shape[0]), text.argmax(dim=-1)] @ self.text_projection       # EOT token = the largest id


def synthetic_text_state_dict(seed=0, width=512, layers=12, heads=8, ctx=77, vocab=49408, out=512):
    """Seeded synthetic text-tower weights in the OpenAI key layout (no prefix), fp32; the global RNG is restored
    (seeded like oracle.restate.synthetic_visual_state_dict)."""
    g = torch.random.get_rng_state()
    torch.manual_seed(seed)
    m = TextTransformer(width, layers, heads, ctx, vocab, out)
    torch.random.set_rng_state(g)
    return OrderedDict((k, v.detach().clone()) for k, v in m.state_dict().items())


def build_text(state_dict):
    """The text tower of an OpenAI-layout state dict (visual.* and the other top-level entries are ignored)."""
    sd = {k: v for k, v in state_dict.items() if k.startswith(TEXT_KEYS)}
    width = sd['token_embedding.weight'].shape[1]
    layers = len([k for k in sd if k.endswith('.attn.in_proj_weight')])
    m = TextTransformer(width, layers, width // 64, sd['positional_embedding'].shape[0], sd['token_embedding.weight'].shape[0],
                        sd['text_projection'].shape[1])
    m.load_state_dict({k: v.float() for k, v in sd.items()})
    return m.float().eval()
