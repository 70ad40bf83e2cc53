"""Test-only helpers for the attention end point (cnn_fm_attention) other than Mixed_4f.

`encoder_forward` is tests/torch_ref.py's differentiable InceptionV1 restatement (fp64 torch, the gradient reference of
cnn_finetune) returning the feature map at any end point; `train_case` is the seeded teacher-forcing case of
tests/test_oracle_known_answers.py with the feature map and attention-dropout masks sized from the config's end point.
Nothing here is imported by the product.
"""
import numpy as np
import torch

from _common import make_weights, fake_features
import torch_ref as TR


def encoder_forward(P, images, endpoint):
    """images [B,224,224,3] NHWC -> (im_embed [B,1024], fm [B,S*S,C] at `endpoint`) differentiable in P."""
    from comic_b200 import weights as wts
    x = torch.as_tensor(np.asarray(images), dtype=next(iter(P.values())).dtype).permute(0, 3, 1, 2)
    x = TR._cbr(P, x, 'Conv2d_1a_7x7', 2)
    x = TR._maxpool(x, 3, 2)
    x = TR._cbr(P, x, 'Conv2d_2b_1x1')
    x = TR._cbr(P, x, 'Conv2d_2c_3x3')
    x = TR._maxpool(x, 3, 2)
    fm = None
    for b in wts.BLOCKS:
        if len(b) == 3:
            x = TR._maxpool(x, b[1], b[2])
        else:
            sc = wts.block_conv_scopes(b[0])
            b0 = TR._cbr(P, x, sc[0])
            b1 = TR._cbr(P, TR._cbr(P, x, sc[1]), sc[2])
            b2 = TR._cbr(P, TR._cbr(P, x, sc[3]), sc[4])
            b3 = TR._cbr(P, TR._maxpool(x, 3, 1), sc[5])
            x = torch.cat([b0, b1, b2, b3], 1)
        if b[0] == endpoint:
            fm = x.permute(0, 2, 3, 1).reshape(x.shape[0], x.shape[2] * x.shape[3], x.shape[1])
    return x.mean(dim=(2, 3)), fm


def train_case(c, B=3, L=7, seed=0, dropout=True):
    """-> (W, im_embed, fm, captions, masks, keeps) with fm [B, M, C] of the config's end point."""
    from comic_b200 import weights as wts
    d = wts.Dims(c)
    rng = np.random.default_rng(seed)
    W = make_weights(c, include_cnn=False)
    im, fm = fake_features(B, C=d.C, M=d.M, seed=seed + 1)
    V = 258 if c.token_type == 'radix' else len(c.itow)
    go, eos = (256, 257) if c.token_type == 'radix' else (c.wtoi['<GO>'], c.wtoi['<EOS>'])
    caps = np.full((B, L), -1, np.int32)
    lens = rng.integers(2, L - 1, size=B)
    lens[0] = L - 2
    for b in range(B):
        n = int(lens[b])
        caps[b, 0] = go
        caps[b, 1:1 + n] = rng.integers(0, V - 2, size=n)
        caps[b, 1 + n] = eos
    T = L - 1
    masks, keeps = None, (1.0, 1.0, 1.0)
    if dropout:
        keeps = (0.65, 0.65, 0.9)
        masks = dict(init_in=(rng.uniform(size=(B, d.W + d.A)) < keeps[0]).astype(np.float32),
                     inp=(rng.uniform(size=(T, B, d.W + d.A)) < keeps[0]).astype(np.float32),
                     out=(rng.uniform(size=(T, B, d.R)) < keeps[1]).astype(np.float32),
                     att=(rng.uniform(size=(T, B, d.H, d.M)) < keeps[2]).astype(np.float32))
    return W, im, fm, caps, masks, keeps
