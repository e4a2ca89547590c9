"""Determinism and batch invariance of the encoders' stem gather and statistics passes at a ragged size.

150x300 input: the stem output row (150 pixels) is not a multiple of the gather's 128-pixel segment, and no layer's
pixel count (11250, 2850, 722) is a multiple of the statistics pass's 64 splits, so the last segment, the last
split and the empty tail lanes are all exercised.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
H, W = 150, 300


def _encoder(variant, norm):
    from tf_raft_b200.layers.extractor import BasicEncoder, SmallEncoder
    cls = BasicEncoder if variant == 'raft' else SmallEncoder
    return cls(output_dim=128, norm_type=norm, seed=7, backend='native')


def _images(n):
    return torch.from_numpy(np.random.default_rng(11).uniform(0, 255, (n, H, W, 3)).astype(np.float32)).cuda()


@pytest.mark.parametrize('variant', ['raft', 'small'])
@pytest.mark.parametrize('norm,training', [('instance', False), ('batch', True)])
def test_encoder_repeatable(variant, norm, training):
    """Two calls of the same encoder on the same input give bitwise equal outputs."""
    enc, x = _encoder(variant, norm), _images(3)
    a = enc(x, training=training, raw_image=True).clone()
    b = enc(x, training=training, raw_image=True)
    assert torch.equal(a, b)


@pytest.mark.parametrize('variant', ['raft', 'small'])
@pytest.mark.parametrize('raw_image', [True, False])
def test_instance_norm_encoder_batch_invariant(variant, raw_image):
    """InstanceNorm statistics are per image: image 0 of a batch of 3 equals image 0 run alone."""
    enc, x = _encoder(variant, 'instance'), _images(3)
    if not raw_image:
        x = 2 * (x / 255.0) - 1.0
    batch = enc(x, training=False, raw_image=raw_image)[:1].clone()
    alone = enc(x[:1].contiguous(), training=False, raw_image=raw_image)
    assert torch.equal(batch, alone)
