"""keras_compat: model code written in the Keras functional style (the style of deephar/models/*.py) records the same
graph, weight list and kernel plan as the function-style mirror of deephar/layers.py; unsupported Keras features are
rejected when the model is built."""
import gzip
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from deephar_b200 import keras_compat as K
from deephar_b200 import layers as L
from deephar_b200.graph import Graph
from deephar_b200.model import Model
from oracle import ops_torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
sys.path.insert(0, GOLDEN)
sys.path.insert(0, os.path.dirname(GOLDEN))


def _keras_style(inp):
    """A stem + separable residual unit + hourglass step, as one would write it for Keras."""
    x = K.Conv2D(32, (3, 3), strides=(2, 2), padding='same', use_bias=False, name='conv1')(inp)
    x = K.BatchNormalization(scale=False, name='bn1')(x)
    x = K.Activation('relu', name='act1')(x)
    a = K.SeparableConv2D(64, (5, 5), padding='same', use_bias=False, name='sep1')(K.Activation('relu')(x))
    a = K.BatchNormalization(name='bn2')(a)
    s = K.Conv2D(64, (1, 1), padding='same', use_bias=False, name='short')(x)
    x = K.add([s, a])
    low = K.MaxPooling2D((2, 2), strides=(2, 2), padding='same')(x)
    low = K.TimeDistributed(K.SeparableConv2D(64, (3, 3), padding='same', use_bias=False), name='td_low')(low)
    x = K.add([x, K.UpSampling2D((2, 2))(low)])
    h = K.Conv2D(8, (1, 1), use_bias=False, name='heat')(K.Activation('relu')(x))
    hm = K.channel_softmax_2d(h)
    return [K.softargmax2d(hm), K.keypoint_confidence(hm), K.concatenate([x, h])]


def _function_style(inp):
    x = L.conv2d(inp, 32, (3, 3), strides=(2, 2), name='conv1')
    x = L.relu(L.BatchNormalization(x, scale=False, name='bn1'), name='act1')
    a = L.BatchNormalization(L.sepconv2d(L.relu(x), 64, (5, 5), name='sep1'), name='bn2')
    s = L.conv2d(x, 64, (1, 1), name='short')
    x = L.add([s, a])
    low = L.sepconv2d(L.maxpooling2d(x), 64, (3, 3), name='td_low')
    x = L.add([x, L.UpSampling2D(low)])
    h = L.conv2d(L.relu(x), 8, (1, 1), padding='valid', name='heat')
    hm = L.channel_softmax_2d(h)
    return [L.softargmax2d(hm), L.keypoint_confidence(hm), L.concatenate([x, h])]


def _models():
    inp = K.Input(shape=(32, 32, 3))
    mk = K.Model(inputs=inp, outputs=_keras_style(inp), name='toy')
    g = Graph('toy')
    g.outputs = _function_style(g.input((32, 32, 3)))
    return mk, Model(g)


def test_keras_style_records_the_same_model():
    mk, mf = _models()
    assert mk.weight_specs == mf.weight_specs
    assert ('td_low/depthwise_kernel', (3, 3, 64, 1)) in mk.weight_specs
    assert [k.kind for k in mk.plan.kops] == [k.kind for k in mf.plan.kops]
    assert mk.output_shape == mf.output_shape == [(None, 8, 2), (None, 8, 1), (None, 16, 16, 72)]
    assert mk.name == 'toy' and mk.input_shape == (None, 32, 32, 3)


def test_clip_input_folds_time():
    inp = K.Input(shape=(4, 16, 16, 3))
    assert inp.g.frames_per_clip == 4 and inp.shape == (16, 16, 3)


def test_unsupported_keras_features_fail_at_build_time():
    inp = K.Input(shape=(16, 16, 3))
    with pytest.raises(NotImplementedError):
        K.Conv2D(8, (3, 3))                                   # Keras default use_bias=True
    with pytest.raises(NotImplementedError):
        K.Conv2D(8, (3, 3), use_bias=False, activation='relu')
    with pytest.raises(NotImplementedError):
        K.SeparableConv2D(8, (3, 3), use_bias=False, depth_multiplier=2)
    with pytest.raises(NotImplementedError):
        K.Activation('tanh')
    with pytest.raises(NotImplementedError):
        K.BatchNormalization(epsilon=1e-5)
    with pytest.raises(TypeError):
        K.UpSampling2D(interpolation='bilinear')
    shared = K.Conv2D(3, (1, 1), use_bias=False)
    y = shared(inp)
    with pytest.raises(NotImplementedError):
        shared(y)
    other = K.Input(shape=(16, 16, 3))
    with pytest.raises(ValueError):
        K.Model(inputs=other, outputs=[y])


@pytest.mark.gpu
def test_keras_style_model_runs_and_matches_oracle(cuda):
    mk, _ = _models()
    mk.init_synthetic_weights(7)
    x = np.random.default_rng(0).uniform(-1, 1, (3, 32, 32, 3)).astype(np.float32)
    outs = mk.predict(x)
    refs = _oracle_forward(mk.get_weights(), x)
    for o, r in zip(outs, refs):
        assert o.shape == r.shape and np.abs(o - r).max() <= 1e-4


def _oracle_forward(w, x):
    o = ops_torch
    w = {k: o.from_numpy(v) for k, v in w.items()}

    def bn(t, name, scale=True):
        return o.batchnorm(t, w[name + '/gamma'] if scale else None, w[name + '/beta'], w[name + '/moving_mean'],
                           w[name + '/moving_variance'])

    t = o.conv2d(o.from_numpy(x), w['conv1/kernel'], (2, 2), 'same')
    t = o.relu(bn(t, 'bn1', scale=False))
    a = bn(o.separable_conv2d(o.relu(t), w['sep1/depthwise_kernel'], w['sep1/pointwise_kernel']), 'bn2')
    t = o.conv2d(t, w['short/kernel']) + a
    low = o.maxpool2d(t, (2, 2), (2, 2), 'same')
    low = o.separable_conv2d(low, w['td_low/depthwise_kernel'], w['td_low/pointwise_kernel'])
    t = t + o.upsample2d(low)
    h = o.conv2d(o.relu(t), w['heat/kernel'], (1, 1), 'valid')
    hm = o.channel_softmax_2d(h)
    pose = o.to_numpy(o.softargmax2d(hm)).reshape(-1, 8, 2)
    vis = o.to_numpy(o.keypoint_confidence(hm)).reshape(-1, 8, 1)
    return [pose, vis, o.to_numpy(o.concat([t, h]))]


def _function_style_backbone(blocks, ksize=(5, 5), heatmaps=48):
    from deephar_b200 import reception as R
    g = Graph('backbone')
    x = R._stem(g.input((256, 256, 3)))
    width, outs = x.channels, []
    for b in range(1, blocks + 1):
        x = R.build_reception_block(x, name='rBlock%d' % b, ksize=ksize)
        ident = x
        x = R.build_sconv_block(x, name='SepConv%d' % b, ksize=ksize)
        h = R.build_regmap_block(x, heatmaps, name='RegMap%d' % b)
        outs.append(h)
        if b < blocks:
            x = L.add([ident, x, R.build_fremap_block(h, width, name='fReMap%d' % b)])
    g.outputs = outs
    return Model(g)


def test_nested_models_and_session_counters():
    """`Model(xi, x, name=...)(inp)` re-records the block under its scope; auto-names count per session."""
    K.clear_session()
    xi = K.Input(shape=(16, 16, 8))
    y = K.BatchNormalization()(K.Conv2D(8, (3, 3), padding='same', use_bias=False)(xi))
    blk = K.Model(inputs=xi, outputs=y, name='Blk')
    inp = K.Input(shape=(16, 16, 8))
    z = K.Conv2D(4, (1, 1), use_bias=False)(K.Activation('relu')(blk(inp)))
    m = K.Model(inputs=inp, outputs=z)
    assert [n for n, _ in m.weight_specs] == [
        'Blk/conv2d_1/kernel', 'Blk/batch_normalization_1/gamma', 'Blk/batch_normalization_1/beta',
        'Blk/batch_normalization_1/moving_mean', 'Blk/batch_normalization_1/moving_variance', 'conv2d_2/kernel']
    assert m.optional_weights == [] and [k.kind for k in m.plan.kops] == ['conv', 'conv']
    with pytest.raises(NotImplementedError):
        blk(inp)                                               # a nested model is applied once
    with pytest.raises(NotImplementedError):
        blk.predict(np.zeros((1, 16, 16, 8), np.float32))      # ... and then belongs to the outer model


def test_reference_backbone_builders_record_the_same_model():
    """The REFERENCE'S OWN code -- deephar/layers.py and models/reception.py::_stem / build_reception_block /
    build_sconv_block / build_regmap_block / build_fremap_block, unmodified -- imported on a `keras` that is
    keras_compat (tests/reference_dropin) records the weight list, auto-names and kernel plan of deephar_b200's builders."""
    got = _recorded('3')
    want = _function_style_backbone(3)
    assert [(n, tuple(s)) for n, s in got['weight_specs']] == want.weight_specs
    assert len(want.weight_specs) > 200
    assert got['plan'] == [[k.kind, [list(t.shape) for t in k.outs]] for k in want.plan.kops]
    assert [tuple(s) for s in got['output_shape']] == [tuple(s) for s in want.output_shape]


def test_reference_spnet_skeleton_records_the_same_model():
    """Same for deephar/models/spnet.py::entry_flow and models/common.py::residual_unit / downscaling_unit /
    upscaling_unit (the reference's code and its own ModelConfig / pose layout, on the recording keras)."""
    from deephar_b200 import common, spnet
    from deephar_b200.config import ModelConfig, pa16j2d
    got = _recorded('spnet')
    cfg = ModelConfig((256, 256, 3), pa16j2d, num_pyramids=2, num_levels=4, num_pose_features=160, num_visual_features=160)
    g = Graph('spnet_skeleton')
    x = spnet.entry_flow(g.input((256, 256, 3)), cfg)
    d = common.downscaling_unit(x, cfg, out_size=x.channels + cfg.growth, name='dn1')
    d = common.residual_unit(d, cfg.kernel_size, name='mid1')
    u = common.upscaling_unit(d, cfg, out_size=x.channels, name='up1')
    g.outputs = [L.add([x, u]), d]
    want = Model(g)
    assert [(n, tuple(s)) for n, s in got['weight_specs']] == want.weight_specs and len(want.weight_specs) > 60
    assert got['plan'] == [[k.kind, [list(t.shape) for t in k.outs]] for k in want.plan.kops]
    assert [tuple(s) for s in got['output_shape']] == [tuple(s) for s in want.output_shape]


@pytest.mark.parametrize('concat', [0, 1])
def test_reference_full_reception_build_records_the_headline_model(concat):
    """The reference's COMPLETE `reception.build()` (reception.py:225-321) -- unmodified file, Lambda channel slices
    and head-model calls included -- on the recording keras, with `deephar.models.blocks`' four parameter-free head
    builders taken from keras_compat: the recorded model IS deephar_b200.reception.build's (BASELINE configs[0]/[1]:
    weight list, auto-names, kernel plan, output order and shapes)."""
    from deephar_b200 import reception
    got = _recorded('full2d %d' % concat)
    want = reception.build((256, 256, 3), 16, dim=2, num_context_per_joint=2, num_blocks=8, ksize=(5, 5),
                           concat_pose_confidence=bool(concat), export_heatmaps=bool(concat))
    assert [(n, tuple(s)) for n, s in got['weight_specs']] == want.weight_specs
    assert got['plan'] == [[k.kind, [list(t.shape) for t in k.outs]] for k in want.plan.kops]
    assert [tuple(s) for s in got['output_shape']] == [tuple(s) for s in want.output_shape]
    assert len(got['output_shape']) == 16        # 8 x (pose, visible), or 8 x (pose|visible, heat-maps)


def _recorded_lines(case):
    """The JSON lines tests/reference_dropin/run_reference_backbone.py printed for `case` (its arguments) when it ran the
    reference's own builder code on the recording keras; stored by tests/golden/make_dropin_golden.py."""
    with gzip.open(os.path.join(GOLDEN, 'ref_dropin_models.json.gz')) as f:
        return json.load(f)[case]


def _recorded(case):
    """The recorded model of `case`, with the lines that follow it (split_model's) merged in."""
    lines = _recorded_lines(case)
    got = next(d for d in lines if 'weight_specs' in d)
    for d in lines:
        if 'weight_specs' not in d:
            got.update(d)
    return got


def _same_model(got, want, same_launch_order=True):
    plan = [[k.kind, [list(t.shape) for t in k.outs]] for k in want.plan.kops]
    assert [(n, tuple(s)) for n, s in got['weight_specs']] == want.weight_specs
    assert got['optional_weights'] == list(want.optional_weights)
    assert [tuple(s) for s in got['output_shape']] == [tuple(s) for s in want.output_shape]
    # every output is the same expression of the same weights (op, attributes, names, operands -- recursively) ...
    assert got['signatures'] == want.graph.signatures()
    # ... compiled into the same kernel launches
    assert sorted(map(str, got['plan'])) == sorted(map(str, plan))
    if same_launch_order:
        assert got['plan'] == plan
    # ... whose buffer plan was replayed by compiler.verify_plan in the recorded launch order
    assert got['plan_checked'] > 2 * len(plan)


def test_reference_reception_3d_build_records_the_c3_model():
    """reception.build(dim=3) of the reference, unmodified: the 3-D head is Lambda / keras.backend arithmetic there
    (reshape to (H, W, D, joints), two means, global max poolings, sigmoid -- reception.py:193-222); recorded as backend
    ops and rewritten into the fused pose_regression_3d op, the model is deephar_b200.reception.build's (BASELINE
    configs[2]), launch for launch."""
    from deephar_b200 import reception
    got = _recorded('full3d')
    want = reception.build((256, 256, 3), 17, dim=3, num_blocks=8, ksize=(5, 5), concat_pose_confidence=False)
    _same_model(got, want)
    assert len(got['plan']) == 134 and len(got['output_shape']) == 16


@pytest.mark.parametrize('which', ['penn', 'ntu'])
def test_reference_full_spnet_build_records_the_c4_c5_models(which):
    """The reference's COMPLETE `spnet.build(cfg)` -- spnet.py, common.py, layers.py, activations.py, config.py, all
    unmodified -- on the recording keras: the channel soft-max body, the frozen SeparableConv2D soft-argmax (its grid
    values are checked), the Lambda joint confidence, kronecker product, confidence mask, depth expectation and
    max+min poolings are traced as backend ops and rewritten into deephar_b200's fused ops.  The result is the SAME
    function of the SAME weights as deephar_b200.spnet.build(cfg) (BASELINE configs[3] / configs[4]) and compiles to the
    same 345 / 237 launches; only the position of the per-block pose-output copies in the launch sequence differs
    (the reference concatenates (pose, confidence) after the re-injection add, spnet.py:239-240)."""
    from deephar_b200 import spnet
    from deephar_b200.config import ModelConfig, pa16j2d, pa17j3d
    if which == 'penn':
        cfg = ModelConfig((16, 256, 256, 3), pa16j2d, num_actions=[15], num_pyramids=6, action_pyramids=[5, 6],
                          num_levels=4, pose_replica=True, num_pose_features=160, num_visual_features=160)
    else:
        cfg = ModelConfig((16, 256, 256, 3), pa17j3d, num_actions=[60], num_pyramids=2, action_pyramids=[1, 2],
                          num_levels=4, pose_replica=False, num_pose_features=192, num_visual_features=192)
    got = _recorded('spnet_full ' + which)
    want = spnet.build(cfg)
    _same_model(got, want, same_launch_order=False)
    assert len(got['plan']) == {'penn': 345, 'ntu': 237}[which]
    assert len(got['output_shape']) == {'penn': 24, 'ntu': 12}[which]
    # the reference's split_model (spnet.py:417-448) on the recorded model: pose outputs / action outputs
    n_pose = spnet.get_num_predictions(cfg.num_pyramids, cfg.num_levels)
    (pname, pn, pshapes, pshared), (aname, an, ashapes, ashared) = got['split']
    assert (pname, pn, aname, an) == ('Pose', n_pose, 'Action', len(got['output_shape']) - n_pose)
    assert pshapes == got['output_shape'][:n_pose] and ashapes == got['output_shape'][n_pose:]
    assert pshared and ashared              # views of the full model's network: the weights loaded into it are theirs


@pytest.mark.parametrize('pose_dim', [2, 3, 'v2'])
def test_reference_merge_model_build_records_the_clip_models(pose_dim):
    """deephar/models/action.py::build_merge_model, unmodified, on the recording keras (SURVEY 8 a16 / f2): get_layer()
    of the pose network's sub-models re-applied under TimeDistributed, the nested `PoseReg` model, the two-Input PoseAR
    model, TimeDistributed head models, sjProb(4 * hs), soft-max -> kronecker product, the 3-D head with its doubled
    visibility logit (action.py:291-292) and the set_weights()-initialised 1x1 merge convolutions: the recorded model is
    deephar_b200.action.build_merge_model's -- weights, expressions, launches and their order."""
    from deephar_b200 import action, reception
    version = 'v1'
    if pose_dim == 'v2':                    # the wider PoseAR net (action.py:63-72), 2-D poses
        pose_dim, version = 2, 'v2'
    got = _recorded('merge %d' % pose_dim + (' v2' if version == 'v2' else ''))
    if pose_dim == 2:
        pe = reception.build((256, 256, 3), 16, dim=2, num_blocks=4, num_context_per_joint=2, ksize=(5, 5))
        want = action.build_merge_model(pe, 15, (256, 256, 3), 16, 16, 4, pose_dim=2, pose_net_version=version)
    else:
        pe = reception.build((256, 256, 3), 20, dim=3, num_blocks=4, depth_maps=8, ksize=(5, 5))
        want = action.build_merge_model(pe, 60, (256, 256, 3), 16, 20, 4, pose_dim=3, depth_maps=8, output_poses=True)
    _same_model(got, want)
    assert len(got['weight_specs']) == 421 and len(got['output_shape']) == (9 if pose_dim == 2 else 11)


def test_builder_options_off_the_baseline_configs_match_the_reference_builders():
    """reception.build / spnet.build arguments the BASELINE configs do not exercise (context maps 0 / 1, alpha, heat-map and
    feature export, depth_maps, 3 levels, growth, kernel 3x3, predict_rootz, several action sets, sam_alpha, image_div,
    other action pyramids, pa20j3d): the reference's builder, recorded, and the product's builder give the same model;
    what one refuses the other refuses."""
    from ref_cases import RECORDED_SWEEP_RECEPTION, RECORDED_SWEEP_SPNET, SWEEP_SPNET_BASE
    from deephar_b200 import config as pconfig
    from deephar_b200 import reception, spnet
    rows = _recorded_lines('sweep')
    assert len(rows) == len(RECORDED_SWEEP_RECEPTION) + len(RECORDED_SWEEP_SPNET) == 13
    builders = []
    for kw in RECORDED_SWEEP_RECEPTION:
        nj = 17 if kw.get('dim') == 3 else 16
        builders.append(('reception %r' % (kw,), lambda kw=kw, nj=nj: reception.build((128, 128, 3), nj, **kw)))
    for shape, layout, extra in RECORDED_SWEEP_SPNET:
        kw = dict(SWEEP_SPNET_BASE)
        kw.update(extra)
        builders.append(('spnet %r %s %r' % (shape, layout, extra),
                         lambda shape=shape, layout=layout, kw=kw: spnet.build(pconfig.ModelConfig(shape, getattr(pconfig, layout), **kw))))
    refused = 0
    for ref, (tag, build) in zip(rows, builders):
        assert ref['tag'] == tag
        K.clear_session()
        try:
            prod = build()
        except Exception as e:                                  # noqa: BLE001
            assert ref.get('ref_error') == type(e).__name__, (tag, type(e).__name__)    # never one side only
            refused += 1
            continue
        assert 'ref_error' not in ref, tag
        assert [(n, tuple(s)) for n, s in ref['weight_specs']] == [(n, tuple(s)) for n, s in prod.weight_specs], tag
        assert ref['signatures'] == prod.graph.signatures(), tag
        assert [tuple(s) for s in ref['output_shape']] == [tuple(s) for s in prod.output_shape], tag
        assert ref['kinds'] == sorted(k.kind for k in prod.plan.kops), tag
    assert refused == 3 and [r['ref_error'] for r in rows if r['tag'].startswith("reception {'dim': 4")] == ['ValueError']


def test_head_models_and_lambda_slices():
    K.clear_session()
    inp = K.Input(shape=(32, 32, 8))
    h = K.Conv2D(48, (1, 1), use_bias=False, name='RegMap')(inp)
    hs = K.Lambda(lambda x: x[:, :, :, :16])(h)
    hc = K.Lambda(lambda x: x[:, :, :, 16:])(h)
    pose = K.build_context_aggregation(16, 2, 0.8, name='Agg')(
        [K.build_softargmax_2d((32, 32, 16), name='sSAM')(hs), K.build_softargmax_2d((32, 32, 32), name='cSAM')(hc),
         K.build_joints_probability((32, 32, 32), name='cjProb')(hc)])
    vis = K.build_joints_probability((32, 32, 16), name='sjProb')(hs)
    m = K.Model(inputs=inp, outputs=[pose, vis, hs])
    assert [k.kind for k in m.plan.kops] == ['conv', 'pose_regression_2d_context']
    assert m.output_shape == [(None, 16, 2), (None, 16, 1), (None, 32, 32, 16)]
    # indexing other than a channel slice fails in the Lambda; backend arithmetic that is not one of the reference's
    # constructions, and a head call outside the recordable patterns, fail when the model is built -- naming the ops
    with pytest.raises(NotImplementedError):
        K.Lambda(lambda x: x[:, 1:, :, :])(h)
    with pytest.raises(NotImplementedError):
        K.Lambda(lambda x: x + 1)(h)
    odd = K.Model(inputs=inp, outputs=[K.Lambda(lambda x: 4 * x)(h)])
    with pytest.raises(NotImplementedError, match='k_scale'):
        odd.plan
    lone = K.Model(inputs=inp, outputs=[K.build_softargmax_2d((32, 32, 48))(h)])
    with pytest.raises(NotImplementedError):
        lone.plan


# ---------------------------------------------------------------------------------------------------------------------
# backend-op tracing (keras_trace.py), without the reference tree: a small multitask clip model written the way one
# writes it for Keras -- soft-max / soft-argmax / confidence / feature pooling as backend arithmetic -- against the
# same model written with the fused helpers of deephar_b200.layers
# ---------------------------------------------------------------------------------------------------------------------
def _grid_expectation(prob, along, name, values=None):
    """E[coordinate] of every map as a frozen depthwise convolution over the whole map with a coordinate-grid kernel."""
    KB = K.backend
    _, _, rows, cols, ch = KB.int_shape(prob)
    conv = K.SeparableConv2D(ch, (rows, cols), use_bias=False, name=name)
    out = K.TimeDistributed(conv, name=name)(prob)
    w = conv.get_weights()
    w[0][:] = 0
    w[1][:] = 0
    ramp = np.linspace(0., 1., cols if along == 'x' else rows) if values is None else values
    for c in range(ch):
        w[0][:, :, c, 0] = ramp[None, :] if along == 'x' else ramp[:, None]
        w[1][0, 0, c, c] = 1
    conv.set_weights(w)
    conv.trainable = False
    out = K.Lambda(lambda t: KB.squeeze(t, axis=-2))(out)
    out = K.Lambda(lambda t: KB.squeeze(t, axis=-2))(out)
    return K.Lambda(lambda t: KB.expand_dims(t, axis=-1))(out)


def _keras_style_multitask(inp, n_maps=6, n_act=5, sharpness=2.0, bad_grid=False):
    KB = K.backend

    def spatial_softmax(t):
        t = sharpness * t
        e = KB.exp(t - KB.max(t, axis=(-3, -2), keepdims=True))
        return e / KB.clip(KB.sum(e, axis=(-3, -2), keepdims=True), KB.epsilon(), None)

    def confidence(t):
        return KB.expand_dims(K.GlobalMaxPooling2D()(4 * K.AveragePooling2D((2, 2), strides=(1, 1))(t)), axis=-1)

    def pooled_features(ts):
        hm, f = ts
        hm = KB.tile(KB.expand_dims(hm, axis=-1), [1, 1, 1, 1, 1, KB.int_shape(f)[-1]])
        f = KB.tile(KB.expand_dims(f, axis=-2), [1, 1, 1, 1, KB.int_shape(hm)[-2], 1])
        return KB.sum(hm * f, axis=(2, 3))

    def max_plus_min(t):
        return K.MaxPooling2D((2, 2), padding='same')(t) - K.MaxPooling2D((2, 2), padding='same')(-t)

    def global_max_plus_min(t):
        return K.GlobalMaxPooling2D()(t) - K.GlobalMaxPooling2D()(-t)

    feat = K.TimeDistributed(K.Conv2D(16, (3, 3), strides=(2, 2), padding='same', use_bias=False), name='feat')(inp)
    feat = K.TimeDistributed(K.Activation('relu'))(feat)
    maps = K.TimeDistributed(K.Conv2D(n_maps, (1, 1), use_bias=False), name='maps')(feat)
    depth = K.TimeDistributed(K.Conv2D(n_maps, (1, 1), use_bias=False), name='depth')(feat)
    prob = K.TimeDistributed(K.Activation(spatial_softmax), name='prob')(maps)
    xy = K.concatenate([_grid_expectation(prob, 'x', 'xy_x', np.linspace(0., 2., 16) if bad_grid else None),
                        _grid_expectation(prob, 'y', 'xy_y')], name='xy')
    vis = K.TimeDistributed(K.Lambda(confidence), name='vis')(prob)
    z = K.multiply([K.Activation('sigmoid')(depth), prob])
    z = K.Lambda(lambda t: KB.expand_dims(KB.sum(t, axis=(-2, -3)), axis=-1))(z)
    xyz = K.concatenate([xy, z], name='xyz')
    pose = K.concatenate([xyz, vis], name='pose')

    masked = K.Lambda(lambda ts: ts[0] * ts[1])([xyz, K.Lambda(lambda t: KB.tile(t, (1, 1, 1, 3)))(vis)])
    a = K.Conv2D(8, (3, 3), padding='same', use_bias=False, name='pose_conv')(masked)
    b = K.Conv2D(8, (1, 1), padding='same', use_bias=False, name='vis_conv')(K.Lambda(pooled_features, name='kron')([prob, feat]))
    x = K.concatenate([a, b])
    x = K.Lambda(max_plus_min)(K.Conv2D(12, (3, 3), padding='same', use_bias=False, name='mix')(x))
    x = K.Activation('relu')(K.BatchNormalization(name='bn')(x))
    logits = K.Conv2D(n_act, (3, 3), padding='same', use_bias=False, name='cls')(x)
    act = K.Activation('softmax', name='action')(K.Lambda(global_max_plus_min)(logits))
    return [pose, act]


def _function_style_multitask(inp, n_maps=6, n_act=5, sharpness=2.0):
    feat = L.relu(L.conv2d(inp, 16, (3, 3), strides=(2, 2), name='feat'))
    maps = L.conv2d(feat, n_maps, (1, 1), padding='valid', name='maps')
    depth = L.conv2d(feat, n_maps, (1, 1), padding='valid', name='depth')
    prob = L.channel_softmax_2d(maps, alpha=sharpness, name='prob')
    xy = L.softargmax2d(prob, name='xy')
    vis = L.keypoint_confidence(prob, name='vis')
    xyz = L.concatenate([xy, L.depth_expectation(depth, prob)], name='xyz')
    pose = L.concatenate([xyz, vis], name='pose')
    masked = L.mask_multiply(L.frames_to_clip(xyz), L.frames_to_clip(vis))
    a = L.conv2d(masked, 8, (3, 3), name='pose_conv')
    b = L.conv2d(L.frames_to_clip(L.kronecker_prod(prob, feat, name='kron')), 8, (1, 1), name='vis_conv')
    x = L.max_min_pooling(L.conv2d(L.concatenate([a, b]), 12, (3, 3), name='mix'), (2, 2))
    x = L.relu(L.BatchNormalization(x, name='bn'))
    logits = L.conv2d(x, n_act, (3, 3), name='cls')
    return [pose, L.softmax_lastaxis(L.global_max_min_pooling(logits), name='action')]


def test_backend_arithmetic_is_rewritten_into_the_fused_ops():
    K.clear_session()
    inp = K.Input(shape=(4, 32, 32, 3))
    mk = K.Model(inputs=inp, outputs=_keras_style_multitask(inp), name='toy_multitask')
    g = Graph('toy_multitask')
    g.frames_per_clip = 4
    g.outputs = _function_style_multitask(g.input((32, 32, 3)))
    mf = Model(g)
    assert mk.weight_specs == mf.weight_specs                      # the frozen grid kernels are not weights
    assert [n for n, _ in mk.weight_specs if n.startswith('xy')] == []
    assert mk.graph.signatures() == mf.graph.signatures()
    assert [(k.kind, [t.shape for t in k.outs]) for k in mk.plan.kops] == \
           [(k.kind, [t.shape for t in k.outs]) for k in mf.plan.kops]
    assert 'sam2d' in [k.kind for k in mk.plan.kops] and mk.output_shape == [(None, 4, 6, 4), (None, 5)]


def test_backend_arithmetic_that_is_not_a_known_construction_is_rejected():
    KB = K.backend
    # a frozen grid that is not the reference's [0, 1] ramp
    K.clear_session()
    inp = K.Input(shape=(4, 32, 32, 3))
    m = K.Model(inputs=inp, outputs=_keras_style_multitask(inp, bad_grid=True))
    with pytest.raises(NotImplementedError, match='soft-argmax grid'):
        m.plan
    # heat-map x feature pooling without the time axis: the reference's axis=(2, 3) would sum columns and joints
    K.clear_session()
    inp = K.Input(shape=(32, 32, 3))
    f = K.Conv2D(8, (3, 3), padding='same', use_bias=False)(inp)
    h = K.Conv2D(4, (1, 1), use_bias=False)(f)

    def pooled(ts):
        hm = KB.tile(KB.expand_dims(ts[0], axis=-1), [1, 1, 1, 1, 8])
        ft = KB.tile(KB.expand_dims(ts[1], axis=-2), [1, 1, 1, 4, 1])
        return KB.sum(hm * ft, axis=(2, 3))
    m = K.Model(inputs=inp, outputs=[K.Lambda(pooled)([h, f])])
    with pytest.raises(NotImplementedError, match='clip tensors'):
        m.plan
    # shape rules of the backend functions themselves
    assert KB.int_shape(h) == (None, 32, 32, 4) and KB.ndim(h) == 4
    assert KB.int_shape(KB.mean(KB.reshape(KB.expand_dims(h), (-1, 32, 32, 2, 2)), axis=3)) == (None, 32, 32, 2)
    with pytest.raises(NotImplementedError):
        KB.sum(h, axis=0)                                          # the batch axis
    with pytest.raises(ValueError):
        KB.squeeze(h, axis=-1)


def test_dropin_registers_a_recording_keras():
    """deephar_b200.dropin.install(): `import keras` / `import tensorflow` resolve to the recording front end; what the
    forward path never calls exists but fails, by name, when it is called."""
    code = r'''
import sys
import deephar_b200.dropin as d
k = d.install()
assert d.install() is k
import keras, tensorflow as tf
import keras.backend as K
from keras.layers import Input, Conv2D, Dense, LSTM, Lambda, TimeDistributed
from keras.models import Model
from keras.optimizers import SGD, RMSprop
from keras.callbacks import Callback, LearningRateScheduler
from keras.utils import Sequence
from keras.utils.data_utils import get_file
from keras.regularizers import l1
from deephar_b200 import keras_compat
assert keras.__version__ == '2.1.4' and Model is keras_compat.Model and K.epsilon() == 1e-7
SGD(lr=0.1); LearningRateScheduler(lambda e: 0.1)
class Loader(Sequence):
    pass
for bad in (lambda: Dense(10), lambda: LSTM(4), lambda: tf.divide(1, 2), lambda: K.sqrt(1)):
    try:
        bad()
    except NotImplementedError as e:
        continue
    raise AssertionError('stub did not fail')
try:
    get_file('no-such-file-in-the-keras-cache', 'http://x')      # a cache look-up: nothing is downloaded
except IOError:
    pass
else:
    raise AssertionError('get_file invented a file')
inp = Input(shape=(16, 16, 3))
m = Model(inputs=inp, outputs=Conv2D(4, (3, 3), padding='same', use_bias=False, name='c')(inp), name='tiny')
assert m.weight_specs == [('c/kernel', (3, 3, 3, 4))] and [k_.kind for k_ in m.plan.kops] == ['conv']
B = sys.modules['deephar.models.blocks']   # what `from .blocks import *` in the reference's model files will find
assert B.build_softargmax_2d is keras_compat.build_softargmax_2d
d.uninstall()
assert 'keras' not in sys.modules and 'deephar.models.blocks' not in sys.modules
print('ok')
'''
    out = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, timeout=300,
                         cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    assert out.returncode == 0 and out.stdout.strip().endswith('ok'), out.stderr[-2000:]


def test_models_as_layers_of_other_models():
    """What deephar/models/action.py does with Keras models, on small ones: a two-Input model used as a layer, sub-models
    fetched with get_layer() and applied again in another model (same weight names there), a model nesting nested models
    (one scope per weight), set_weights() that does NOT freeze while the layer stays trainable."""
    KB = K.backend
    K.clear_session()
    # a "pose network" with two named blocks
    inp = K.Input(shape=(16, 16, 3))
    xi = K.Input(shape=(16, 16, 3))
    stem = K.Model(xi, K.Conv2D(8, (3, 3), padding='same', use_bias=False)(xi), name='Stem')
    x = stem(inp)
    xi = K.Input(shape=KB.int_shape(x)[1:])
    head = K.Model(xi, K.Conv2D(4, (1, 1), use_bias=False)(K.Activation('relu')(xi)), name='Head')
    pe = K.Model(inputs=inp, outputs=head(x))
    assert pe.get_layer('Stem') is stem and pe.get_layer('Head').name == 'Head'
    with pytest.raises(ValueError):
        pe.get_layer('nope')
    assert [n for n, _ in pe.weight_specs] == ['Stem/conv2d_1/kernel', 'Head/conv2d_2/kernel']

    pe.set_weights({n: np.full(sh, 0.25, np.float32) for n, sh in pe.weight_specs})     # "pre-trained" pose network

    # a clip model re-using them: Stem under TimeDistributed, Head nested once more inside 'Wrap'
    clips = K.Input(shape=(4, 16, 16, 3))
    f = K.TimeDistributed(pe.get_layer('Stem'), name='td_Stem')(clips)
    wi = K.Input(shape=KB.int_shape(f)[2:])
    wrap = K.Model(wi, pe.get_layer('Head')(wi), name='Wrap')
    maps = K.TimeDistributed(wrap, name='td_Wrap')(f)
    assert KB.int_shape(wrap.output) == (None, 16, 16, 4) and KB.int_shape(maps) == (None, 4, 16, 16, 4)

    # a two-Input sub-model on (T, joints, c) tensors, applied to per-frame results
    a, b = K.Input(shape=(4, 4, 2)), K.Input(shape=(4, 4, 1))
    masked = K.Lambda(lambda ts: ts[0] * ts[1])([a, K.Lambda(lambda t: KB.tile(t, [1, 1, 1, 2]))(b)])
    two = K.Model(inputs=[a, b], outputs=K.Conv2D(6, (3, 3), padding='same', use_bias=False)(masked), name='Two')
    assert a.g is b.g and len(a.g.inputs) == 2                       # the two Inputs became one graph
    with pytest.raises(NotImplementedError):
        two.plan                                                     # several Inputs: only inside another model

    def softmax(t):
        e = KB.exp(t - KB.max(t, axis=(-3, -2), keepdims=True))
        return e / KB.clip(KB.sum(e, axis=(-3, -2), keepdims=True), KB.epsilon(), None)
    prob = K.TimeDistributed(K.Activation(softmax), name='prob')(maps)
    xy = K.concatenate([_grid_expectation(prob, 'x', 'xy_x'), _grid_expectation(prob, 'y', 'xy_y')], name='xy')
    vis = K.TimeDistributed(K.Lambda(lambda t: KB.expand_dims(K.GlobalMaxPooling2D()(
        4 * K.AveragePooling2D((2, 2), strides=(1, 1))(t)), axis=-1)), name='vis')(prob)
    y = two([xy, vis])
    # merge weights initialised by hand but left trainable: they stay weights of the model
    conv = K.SeparableConv2D(6, (1, 1), use_bias=False)
    z = conv(y)
    w = conv.get_weights()
    w[0].fill(1.)
    conv.set_weights(w)
    m = K.Model(clips, [z, xy])
    assert [n for n, _ in m.weight_specs] == ['Stem/conv2d_1/kernel', 'Head/conv2d_2/kernel', 'Two/conv2d_3/kernel',
                                              'separable_conv2d_1/depthwise_kernel', 'separable_conv2d_1/pointwise_kernel']
    kinds = [k.kind for k in m.plan.kops]
    assert kinds.count('conv') == 3 and 'sam2d' in kinds and 'mask_mul' in kinds and kinds[-1] == 'sepconv'
    assert m.output_shape == [(None, 4, 4, 6), (None, 4, 4, 2)]
    m.init_synthetic_weights(3)                                      # the layers shared with `pe` keep pe's weights
    got = m.get_weights()
    assert got['Stem/conv2d_1/kernel'].min() == got['Head/conv2d_2/kernel'].max() == 0.25
    assert np.unique(got['Two/conv2d_3/kernel']).size > 10
    with pytest.raises(NotImplementedError):
        stem.plan                                                    # applied as a layer: compile the outer model
    with pytest.raises(NotImplementedError):
        pe.get_layer('Stem')(f)                                      # once per model


def test_a_model_of_some_outputs_shares_the_compiled_network():
    """Model(full.input, full.outputs[:n]) after the full model exists (spnet.py:443-446): a view, not a second network."""
    K.clear_session()
    inp = K.Input(shape=(16, 16, 3))
    a = K.Conv2D(4, (3, 3), padding='same', use_bias=False, name='a')(inp)
    b = K.Conv2D(2, (1, 1), use_bias=False, name='b')(K.Activation('relu')(a))
    full = K.Model(inputs=inp, outputs=[a, b], name='full')
    table = {n: np.full(s, 0.5, np.float32) for n, s in full.weight_specs}
    full.set_weights(table)
    part = K.Model(full.input, full.outputs[1:], name='part')
    assert part.name == 'part' and part.output_shape == [(None, 16, 16, 2)] and part.input_shape == (None, 16, 16, 3)
    assert part._compiled().full is full._compiled()
    assert part._compiled().full.get_weights()['b/kernel'].max() == 0.5
    other = K.Model(full.input, K.Conv2D(2, (1, 1), use_bias=False, name='c')(a))       # not a subset: its own network
    assert [n for n, _ in other.weight_specs] == ['a/kernel', 'b/kernel', 'c/kernel'] and other.optional_weights == ['b/kernel']


@pytest.mark.parametrize('which', ['mpii', 'h36m', 'penn_multitask', 'ntu_multitask', 'mpii+predict', 'h36m+predict'])
def test_reference_entry_scripts_run_unmodified(which):
    """The reference's entry scripts of every BASELINE config, executed AS THEY ARE (runpy) after dropin.install()
    (tests/reference_dropin/run_reference_script.py): exp/mpii/eval_mpii_singleperson.py (configs[0]/[1], the headline
    model), exp/h36m/eval_h36m.py (configs[2]), exp/pennaction/eval_penn_multitask.py (configs[3]) and
    exp/ntu/eval_ntu_multitask.py (configs[4]) -- reception.build / spnet.build, load_weights, the scripts' own re-wiring
    (Model(model.input, [concatenate([pose, vis]) ...]), split_model) and the reference's own evaluators calling
    predict().  What those runs ended up with is stored in tests/golden/ref_entry_scripts.json.gz
    (make_entry_script_golden.py, which also checks there that the evaluators raised nothing): the scores the evaluators
    returned and the recording of the re-wired model.  Here, without the reference, the same re-wiring is rebuilt with
    keras_compat on deephar_b200's builders (tests/reference_dropin/standins.py): it records the same model (weights,
    output expressions, launches, split views), holds the loaded weights, replays memory-safe and, executed on the CPU,
    computes the oracle's outputs; and the scores recomputed from the oracle's outputs on the same stand-in datasets
    equal the evaluators'.  The '+predict' variants recompute them from the product's OWN Model.predict / _bind / launch
    sequence of the re-wired model, with only the device stood in for (tests/fake_cuda.py --arithmetic: numpy behind the
    C entry points)."""
    here = os.path.dirname(os.path.abspath(__file__))
    with gzip.open(os.path.join(GOLDEN, 'ref_entry_scripts.json.gz')) as f:
        rec = json.load(f)
    own_predict = which.endswith('+predict')
    which = which.split('+')[0]
    rec = rec[which]
    cmd = [sys.executable, os.path.join(here, 'reference_dropin', 'standins.py'), which]
    if own_predict:
        cmd = [sys.executable, os.path.join(here, 'fake_cuda.py'), '--arithmetic'] + cmd[1:] + ['predict']
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    got = json.loads([l for l in out.stdout.splitlines() if l.startswith('{')][-1])
    expected_calls = {'mpii': ['eval_singleperson_pckh'], 'h36m': ['eval_human36m_sc_error'],
                      'penn_multitask': ['eval_multiclip_dataset', 'eval_singleclip_generator', 'eval_singleperson_pckh'],
                      'ntu_multitask': ['eval_multiclip_dataset']}[which]
    assert sorted(rec['returned']) == sorted(got['returned']) == expected_calls
    for fn in expected_calls:
        assert len(rec['returned'][fn]) == 1
        # fp32 buffers under the product's own predict vs the fp32 torch oracle: continuous scores agree to ~1e-6
        assert rec['returned'][fn][0] == pytest.approx(got['returned'][fn], rel=1e-4 if own_predict else 1e-9, abs=1e-12), fn
    model = got['model']
    for key in ('weight_specs', 'signatures', 'optional_weights', 'output_shape'):
        assert model[key] == rec['model'][key], key
    # the same launches; in the same order except for SPNet's per-block pose-output copies (as in
    # test_reference_full_spnet_build_records_the_c4_c5_models)
    assert sorted(map(str, model['plan'])) == sorted(map(str, rec['model']['plan']))
    if which in ('mpii', 'h36m'):
        assert model['plan'] == rec['model']['plan']
    assert got['split'] == rec['split']
    assert model['weights_are_the_files']            # loaded BEFORE the re-wiring, shared with it as Keras shares layers
    assert model['plan_checked'] > model['launches']   # the re-wired model's buffer plan replays memory-safe
    assert model['plan_emulation_max_err'] < 5e-4    # ... and, executed on the CPU, computes the oracle's outputs (fp32 oracle)
    if which in ('mpii', 'h36m'):
        assert rec['output_shape'] == [[None, 16 if which == 'mpii' else 17, 3 if which == 'mpii' else 4]] * 8
    else:
        assert rec['output_shape'] == [[None, 15 if which == 'penn_multitask' else 60]] * 6      # the 'Action' split
        assert [s[3] for s in rec['split']] == [True, True]          # views of the loaded full network
        assert max(rec['returned']['eval_multiclip_dataset'][0]) == 50.0        # labels: one right, one wrong by design


def test_get_file_is_a_cache_lookup(tmp_path, monkeypatch):
    from deephar_b200 import dropin
    monkeypatch.setenv('KERAS_HOME', str(tmp_path))
    with pytest.raises(IOError) as e:
        dropin.get_file('w.h5', 'https://example.invalid/w.h5', cache_subdir='models')
    assert str(tmp_path / 'models' / 'w.h5') in str(e.value) and 'example.invalid' in str(e.value)
    (tmp_path / 'models').mkdir()
    (tmp_path / 'models' / 'w.h5').write_bytes(b'abc')
    assert dropin.get_file('w.h5', 'x', cache_subdir='models', md5_hash='900150983cd24fb0d6963f7d28e17f72') == \
        str(tmp_path / 'models' / 'w.h5')
    with pytest.warns(UserWarning):
        assert dropin.get_file('w.h5', 'x', cache_subdir='models', md5_hash='0' * 32).endswith('w.h5')
    absolute = tmp_path / 'annotations.mat'
    absolute.write_bytes(b'')
    assert dropin.get_file(str(absolute), 'x') == str(absolute)     # datasets/annothelper.py passes absolute paths


def test_predict_takes_its_input_in_a_list_as_keras_does():
    from deephar_b200 import reception
    m = reception.build((64, 64, 3), num_joints=16, dim=2, num_context_per_joint=2, num_blocks=1, ksize=(3, 3))
    x = np.zeros((2, 64, 64, 3), np.float64)
    assert m._host_input([x]).shape == (2, 64, 64, 3) and m._host_input([x]).dtype == np.float32   # mpii_tools.py:80-86
    with pytest.raises(ValueError):
        m.predict([x, x])
    with pytest.raises(ValueError):
        m.predict([x[:, :32]])
    for bad in (0, -1, 2.5):
        with pytest.raises(ValueError):
            m.predict(x, batch_size=bad)
