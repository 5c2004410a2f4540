"""Executes the reference's own model builders after deephar_b200.dropin.install() and prints the recorded model's
weight list, kernel plan, output shapes and expression digests as JSON.  Runs where the reference tree exists
(DEEPHAR_REFERENCE); tests/golden/make_dropin_golden.py stores what it prints for tests/test_keras_compat.py.

    DEEPHAR_REFERENCE=<reference checkout> python run_reference_backbone.py <case>"""
import json
import os
import sys
import warnings

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
if not os.path.isdir(os.environ.get('DEEPHAR_REFERENCE', '')):
    raise SystemExit('set DEEPHAR_REFERENCE to the reference checkout')
sys.path[:0] = [os.environ['DEEPHAR_REFERENCE'], ROOT]
warnings.filterwarnings('ignore')
import deephar_b200.dropin  # noqa: E402
deephar_b200.dropin.install()                                 # `keras` / `tensorflow` -> the recording front end
_stderr, sys.stderr = sys.stderr, open(os.devnull, 'w')       # the reference prints a banner on import
import deephar  # noqa: E402,F401
from deephar.models import reception as R  # noqa: E402
sys.stderr = _stderr

from keras.layers import Input, add  # noqa: E402   (= deephar_b200.keras_compat)
from keras.models import Model  # noqa: E402
from deephar_b200 import keras_compat  # noqa: E402
from deephar_b200.compiler import verify_plan  # noqa: E402


def spnet_case():
    """spnet.py:317-352 entry_flow + common.py:25-108 residual / downscaling / upscaling units (the conv skeleton of a
    pyramid level), driven by the reference's own ModelConfig."""
    from deephar.config import ModelConfig
    from deephar.models import spnet as S
    from deephar.models.common import downscaling_unit, residual_unit, upscaling_unit
    from deephar.utils.pose import pa16j2d
    cfg = ModelConfig((256, 256, 3), pa16j2d, num_pyramids=2, num_levels=4, num_pose_features=160, num_visual_features=160)
    keras_compat.clear_session()
    inp = Input(shape=(256, 256, 3))
    x = S.entry_flow(inp, cfg)
    d = downscaling_unit(x, cfg, out_size=x.shape[-1] + cfg.growth, name='dn1')
    d = residual_unit(d, cfg.kernel_size, name='mid1')
    u = upscaling_unit(d, cfg, out_size=x.shape[-1], name='up1')
    y = add([x, u])
    m = Model(inputs=inp, outputs=[y, d], name='spnet_skeleton')
    print(json.dumps({'weight_specs': [[n, list(s)] for n, s in m.weight_specs],
                      'plan': [[k.kind, [list(t.shape) for t in k.outs]] for k in m.plan.kops],
                      'output_shape': [list(s) for s in m.output_shape]}))


def _dump(m):
    print(json.dumps({'weight_specs': [[n, list(s)] for n, s in m.weight_specs],
                      'plan': [[k.kind, [list(t.shape) for t in k.outs]] for k in m.plan.kops],
                      'output_shape': [list(s) for s in m.output_shape],
                      'optional_weights': list(m.optional_weights),
                      'signatures': m.graph.signatures(),
                      'plan_checked': verify_plan(m.plan, m.graph)}))       # memory-safe in ITS launch order


def full_model_case(concat):
    """The reference's COMPLETE reception.build() (reception.py:225-321), heads included: BASELINE configs[0]/[1]."""
    keras_compat.clear_session()
    _dump(R.build((256, 256, 3), 16, dim=2, num_context_per_joint=2, num_blocks=8, ksize=(5, 5),
                  concat_pose_confidence=bool(concat), export_heatmaps=bool(concat)))


def full_3d_case():
    """reception.build(dim=3) with its Lambda / keras.backend 3-D head (reception.py:193-222): BASELINE configs[2]."""
    keras_compat.clear_session()
    _dump(R.build((256, 256, 3), 17, dim=3, num_blocks=8, ksize=(5, 5), concat_pose_confidence=False))


def full_spnet_case(which):
    """The reference's COMPLETE spnet.build(cfg) (spnet.py:355-410) on its own layers.py / activations.py / common.py /
    config.py: prediction blocks with the frozen-SeparableConv2D soft-argmax, Lambda confidence, kronecker product,
    depth expectation and the whole action head.  BASELINE configs[3] (PennAction) and configs[4] (NTU, 3-D)."""
    from deephar.config import ModelConfig
    from deephar.models import spnet as S
    from deephar.utils.pose import pa16j2d, pa17j3d
    keras_compat.clear_session()
    if which == 'penn':
        cfg = ModelConfig((16, 256, 256, 3), pa16j2d, num_actions=[15], num_pyramids=6, action_pyramids=[5, 6],
                          num_levels=4, pose_replica=True, num_pose_features=160, num_visual_features=160)
    else:
        cfg = ModelConfig((16, 256, 256, 3), pa17j3d, num_actions=[60], num_pyramids=2, action_pyramids=[1, 2],
                          num_levels=4, pose_replica=False, num_pose_features=192, num_visual_features=192)
    full = S.build(cfg)
    _dump(full)
    # spnet.py:417-448 on the recorded model: Model(full.input, full.outputs[:n]) / [n:]
    pose, act = S.split_model(full, cfg, interlaced=False, model_names=['Pose', 'Action'])
    print(json.dumps({'split': [[pose.name, len(pose.outputs), [list(s) for s in pose.output_shape],
                                 pose._compiled().full is full._compiled()],
                                [act.name, len(act.outputs), [list(s) for s in act.output_shape],
                                 act._compiled().full is full._compiled()]]}))


def merge_model_case(pose_dim, version='v1'):
    """deephar/models/action.py::build_merge_model (the CVPR'18 clip model, action.py:319-400), unmodified: the
    sub-models of the pose network are fetched with get_layer() and re-applied under TimeDistributed, `PoseReg` nests
    them again, PoseAR is a two-Input model, the heads are TimeDistributed head models, sjProb(4 * hs), the soft-max of
    the heat-maps feeds the kronecker product, 1x1 SeparableConv2D merge weights set with set_weights()."""
    from deephar.models import action as A
    keras_compat.clear_session()
    if pose_dim == 2:
        pe = R.build((256, 256, 3), 16, dim=2, num_blocks=4, num_context_per_joint=2, ksize=(5, 5))
        m = A.build_merge_model(pe, 15, (256, 256, 3), 16, 16, 4, pose_dim=2, pose_net_version=version, full_trainable=False)
    else:
        pe = R.build((256, 256, 3), 20, dim=3, num_blocks=4, depth_maps=8, ksize=(5, 5))
        m = A.build_merge_model(pe, 60, (256, 256, 3), 16, 20, 4, pose_dim=3, depth_maps=8, output_poses=True)
    _dump(m)


def option_sweep_case():
    """Builder options off the BASELINE configs (ref_cases.RECORDED_SWEEP_*): the reference's reception.build /
    spnet.build (unmodified, recorded), one JSON line per configuration -- the recorded weight list, output expressions,
    output shapes and launch kinds, or the exception the builder raised.  tests/test_keras_compat.py builds the product
    model for the same arguments and compares.  (spnet.py:210-214 keeps a module-level action-block counter across builds
    in one process -- a second model is named act7_..., which breaks by_name loading in the reference itself; reset here
    per build.)"""
    from deephar.config import ModelConfig as RefConfig
    from deephar.models import spnet as S
    from deephar.utils import pose as ref_pose
    sys.path.insert(0, os.path.join(ROOT, 'tests', 'golden'))
    from ref_cases import RECORDED_SWEEP_RECEPTION, RECORDED_SWEEP_SPNET, SWEEP_SPNET_BASE

    def record(tag, ref_fn):
        keras_compat.clear_session()
        S.__dict__.pop('act_cnt', None)
        res = {'tag': tag}
        try:
            ref = ref_fn()
            res.update(weight_specs=[[n, list(s)] for n, s in ref.weight_specs], signatures=ref.graph.signatures(),
                       output_shape=[list(s) for s in ref.output_shape], kinds=sorted(k.kind for k in ref.plan.kops))
        except Exception as e:                                  # noqa: BLE001
            res = {'tag': tag, 'ref_error': type(e).__name__}
        print(json.dumps(res))

    for kw in RECORDED_SWEEP_RECEPTION:
        nj = 17 if kw.get('dim') == 3 else 16
        record('reception %r' % (kw,), lambda: R.build((128, 128, 3), nj, **kw))
    for shape, layout, extra in RECORDED_SWEEP_SPNET:
        kw = dict(SWEEP_SPNET_BASE)
        kw.update(extra)
        record('spnet %r %s %r' % (shape, layout, extra), lambda: S.build(RefConfig(shape, getattr(ref_pose, layout), **kw)))


def main():
    if sys.argv[1] == 'sweep':
        return option_sweep_case()
    if sys.argv[1] == 'merge':
        return merge_model_case(int(sys.argv[2]), *sys.argv[3:4])
    if sys.argv[1] == 'spnet':
        return spnet_case()
    if sys.argv[1] == 'full3d':
        return full_3d_case()
    if sys.argv[1] == 'spnet_full':
        return full_spnet_case(sys.argv[2])
    if sys.argv[1] == 'full2d':
        return full_model_case(int(sys.argv[2]))
    blocks, ksize, heatmaps = int(sys.argv[1]), (5, 5), 48
    keras_compat.clear_session()
    inp = Input(shape=(256, 256, 3))
    x = R._stem(inp)
    width = x.shape[-1]
    outs = []
    for b in range(1, blocks + 1):
        x = R.build_reception_block(x, name='rBlock%d' % b, ksize=ksize)
        ident = x
        x = R.build_sconv_block(x, name='SepConv%d' % b, ksize=ksize)
        h = R.build_regmap_block(x, heatmaps, name='RegMap%d' % b)
        outs.append(h)
        if b < blocks:
            x = add([ident, x, R.build_fremap_block(h, width, name='fReMap%d' % b)])
    m = Model(inputs=inp, outputs=outs, name='backbone')
    print(json.dumps({'weight_specs': [[n, list(s)] for n, s in m.weight_specs],
                      'plan': [[k.kind, [list(t.shape) for t in k.outs]] for k in m.plan.kops],
                      'output_shape': [list(s) for s in m.output_shape]}))


if __name__ == '__main__':
    main()
