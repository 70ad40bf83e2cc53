"""Host side of `--cnn_fm_attention` (no GPU): the model dimensions, decoder variable shapes and parameter counts at every
built end point against the oracle's InceptionV1 end points, the refusal of the end points that are not built, a
checkpoint round trip and the train.py flag."""
import numpy as np
import pytest

from _common import comic_config, make_weights, images
import comic_b200  # noqa: F401
from comic_b200 import checkpoint as ck
from comic_b200 import cli
from comic_b200 import weights as wts
import inception_v1_oracle as I

BUILT = ['MaxPool_4a_3x3', 'Mixed_4b', 'Mixed_4c', 'Mixed_4d', 'Mixed_4e', 'Mixed_4f', 'MaxPool_5a_2x2', 'Mixed_5b',
         'Mixed_5c']
REFUSED = ['Conv2d_1a_7x7', 'MaxPool_2a_3x3', 'Conv2d_2b_1x1', 'Conv2d_2c_3x3', 'MaxPool_3a_3x3', 'Mixed_3b', 'Mixed_3c',
           'AvgPool_0a_7x7']


@pytest.fixture(scope='module')
def oracle_endpoints():
    c = comic_config()
    _, ep = I.inception_v1(images(1), make_weights(c))
    return ep


def test_built_end_points_are_the_library_ids():
    """FM_ENDPOINTS is in network order; its index is COMIC_FM_* (include/comic_b200.h)."""
    assert list(wts.FM_ENDPOINTS) == BUILT


@pytest.mark.parametrize('proj', ['tied', 'independent', None])
@pytest.mark.parametrize('endpoint', BUILT)
def test_dims_follow_the_end_point(oracle_endpoints, endpoint, proj):
    c = comic_config(cnn_fm_attention=endpoint, cnn_fm_projection=proj)
    d = wts.Dims(c)
    _, S, S2, C = oracle_endpoints[endpoint].shape
    assert (d.M, d.C) == (S * S2, C)
    assert d.A == (C if proj is None else d.R)
    assert d.VAL == (C if proj is None else d.R)


@pytest.mark.parametrize('endpoint', BUILT)
def test_decoder_parameter_count_follows_memory_layer(endpoint):
    """Only memory_layer [C, R] (and value_layer [C, R] when independent) depend on C for projected models."""
    base_t = wts.count_params(wts.decoder_shapes(comic_config()))
    base_i = wts.count_params(wts.decoder_shapes(comic_config(cnn_fm_projection='independent')))
    C = wts.Dims(comic_config(cnn_fm_attention=endpoint)).C
    sh = wts.decoder_shapes(comic_config(cnn_fm_attention=endpoint))
    assert sh[wts.DEC + 'memory_layer/kernel'] == (C, 512)
    assert wts.count_params(sh) == base_t + (C - 832) * 512
    sh = wts.decoder_shapes(comic_config(cnn_fm_attention=endpoint, cnn_fm_projection='independent'))
    assert sh[wts.DEC + 'value_layer/kernel'] == (C, 512)
    assert wts.count_params(sh) == base_i + 2 * (C - 832) * 512


@pytest.mark.parametrize('endpoint', REFUSED)
def test_end_points_not_built_are_refused_on_the_host(endpoint):
    """Refused by Dims (which every Engine, Trainer and weight initialiser builds first) before a device is touched; the
    message names the end points that are built."""
    c = comic_config(cnn_fm_attention=endpoint)
    with pytest.raises(NotImplementedError, match='Mixed_4b, Mixed_4c') as e:
        wts.Dims(c)
    assert endpoint in str(e.value)
    with pytest.raises(NotImplementedError):
        wts.init_weights(c, include_cnn=False)


def test_checkpoint_round_trip_at_a_non_default_end_point(tmp_path):
    c = comic_config(cnn_fm_attention='Mixed_5c', cnn_fm_projection='independent')
    W = wts.init_weights(c, seed=5, include_cnn=False)
    prefix = str(tmp_path / 'run' / 'model_compact-3')
    rng = np.random.default_rng(0)
    trained = {k: (np.asarray(v) + rng.standard_normal(np.shape(v)).astype(np.float32) * 0.01).astype(np.float32)
               for k, v in W.items()}
    ck.write_v2(prefix, trained, with_data_crc=False)
    shapes = ck.variable_shapes(prefix)
    assert shapes[wts.DEC + 'memory_layer/kernel'] == [1024, 512]
    assert shapes[wts.DEC + 'value_layer/kernel'] == [1024, 512]
    c.checkpoint_path, c.resume_training, c.checkpoint_exclude_scopes = str(tmp_path / 'run'), True, ''
    got, info = ck.restore_weights(c, W)
    assert info['mode'] == 'resume'
    for k in W:
        np.testing.assert_array_equal(got[k], trained[k])


def test_cli_parses_a_7x7_end_point():
    args = cli.create_train_parser().parse_args(['--cnn_fm_attention', 'Mixed_5b'])
    c = cli.config_from_train_args(args)
    assert c.cnn_fm_attention == 'Mixed_5b'
    d = wts.Dims(c)
    assert (d.M, d.C) == (49, 832)


@pytest.mark.parametrize('endpoint', ['Mixed_4c', 'MaxPool_4a_3x3', 'Mixed_5b', 'Mixed_5c'])
def test_torch_encoder_restatement_matches_oracle_end_point(endpoint):
    """The fp64 gradient reference of cnn_finetune (tests/fm_endpoint_ref.py) computes the oracle's feature map."""
    import fm_endpoint_ref as FR
    import torch_ref as TR
    c = comic_config(cnn_fm_attention=endpoint)
    W = make_weights(c, seed=11)
    img = images(1, seed=5)
    emb, fm = FR.encoder_forward(TR.cnn_params(W), img, endpoint)
    o_emb, o_fm, _ = I.encoder(img.astype(np.float64), W, c)
    np.testing.assert_allclose(fm.detach().numpy(), o_fm, rtol=0, atol=1e-9 * np.abs(o_fm).max())
    np.testing.assert_allclose(emb.detach().numpy(), o_emb, rtol=0, atol=1e-9 * np.abs(o_emb).max())
