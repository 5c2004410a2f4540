"""Parity against the REFERENCE'S OWN builder code.

tests/golden/ref_*.npz were written by tests/golden/make_reference_golden.py, which imports
deephar/models/{reception,spnet,action,blocks,common}.py, layers.py and activations.py UNMODIFIED from
the reference checkout and executes them on tests/golden/keras_shim (an eager float64 stand-in for the Keras 2.1.4
API; keras/tensorflow themselves are not installable here).  Each fixture holds the weight list of the
reference model as Keras would save it, and the outputs of the reference graph for seeded inputs and the
product's synthetic weights (assigned by name).

  * weight lists: the product's `weight_specs` must be exactly the reference's learned weights (names with
    Keras auto-name counters, and shapes); the only allowed extras are `optional_weights` (layers the
    reference builds but keras.Model prunes because they feed no output);
  * oracle (numpy fp64) vs reference outputs: <= 1e-9 (1e-6 for the merge model) -- pins the oracle's
    restatement of the graph wiring;
  * independent torch-CPU fp32 op set vs reference outputs: <= 2e-4;
  * the product's compiled plan, executed on the CPU (tests/plan_emulator.py) vs reference outputs: <= 2e-6;
  * product (GPU) vs reference outputs: north-star tolerance 1e-3 (-m gpu).
"""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, 'golden'))
from ref_cases import MERGE3D_CASE, MERGE_CASE, positive_last_regmap, RECEPTION_CASES, SPNET_CASES, SPNET_FULL_CASES  # noqa: E402

from deephar_b200 import action, reception, spnet  # noqa: E402
from deephar_b200.config import ModelConfig, pa16j2d, pa17j3d  # noqa: E402
from oracle import action as oracle_action  # noqa: E402
from oracle import ops_np, ops_torch  # noqa: E402
from oracle import reception as oracle_reception  # noqa: E402
from oracle import spnet as oracle_spnet  # noqa: E402

ALL_CASES = list(RECEPTION_CASES) + list(SPNET_CASES) + list(SPNET_FULL_CASES) + ['merge_model', 'merge3d_model']
SPNET_ALL = dict(SPNET_CASES)
SPNET_ALL.update({k: v[:5] for k, v in SPNET_FULL_CASES.items()})
LAYOUTS = {'pa16j2d': (pa16j2d, oracle_spnet.pa16j2d), 'pa17j3d': (pa17j3d, oracle_spnet.pa17j3d)}


def _fixture(case):
    z = np.load(os.path.join(HERE, 'golden', 'ref_%s.npz' % case))
    outs = [z['out%d' % i] for i in range(len([k for k in z.files if k.startswith('out')]))]
    return z, outs


def _input(case, z):
    """Frames of the fixture: stored, or (full-size cases) regenerated from the recorded recipe and checked
    against the recorded CRC."""
    if 'x' in z.files:
        return z['x']
    import zlib
    from oracle import synth
    if case in RECEPTION_CASES:
        shape, _, _, xs, frames = RECEPTION_CASES[case]
        x = synth.synth_frames(frames, shape[0], shape[1], seed=xs)
    else:
        shape, _, _, _, batch, xs = SPNET_FULL_CASES[case]
        x = np.random.default_rng(xs).uniform(-1.0, 1.0, (batch,) + shape)
    x = np.ascontiguousarray(x, dtype=np.float32)
    assert zlib.crc32(x.tobytes()) == int(z['x_crc32']), 'regenerated input differs from the one the fixture was made with'
    return x


def _product(case):
    if case in RECEPTION_CASES:
        shape, kw, seed = RECEPTION_CASES[case][:3]
        return reception.build(shape, **kw), seed
    if case in SPNET_ALL:
        shape, layout, kw, seed, _ = SPNET_ALL[case]
        return spnet.build(ModelConfig(shape, LAYOUTS[layout][0], **kw)), seed
    if case == 'merge3d_model':
        mc = MERGE3D_CASE
        pe = reception.build(mc['input_shape'], **mc['reception'])
        return action.build_merge_model(pe, mc['num_actions'], mc['input_shape'], mc['num_frames'], mc['num_joints'],
                                        mc['num_blocks'], pose_dim=3, depth_maps=mc['depth_maps'], output_poses=True), mc['seed']
    mc = MERGE_CASE
    pe = reception.build(mc['input_shape'], **mc['reception'])
    return action.build_merge_model(pe, mc['num_actions'], mc['input_shape'], mc['num_frames'], mc['num_joints'],
                                    mc['num_blocks'], pose_dim=2), mc['seed']


def _init_weights(case, m, seed):
    """The weights the fixture was made with: the product's synthetic weights (+ the case's weight hook)."""
    m.init_synthetic_weights(seed)
    if case == 'merge_model':
        m.set_weights(positive_last_regmap(m.get_weights(), MERGE_CASE['num_blocks']))
    return m


def _oracle(case, ops, table, x):
    if case in RECEPTION_CASES:
        return oracle_reception.forward(ops, table, x, **RECEPTION_CASES[case][1])
    if case in SPNET_ALL:
        shape, layout, kw, _, _ = SPNET_ALL[case]
        return oracle_spnet.forward(ops, table, x, oracle_spnet.ModelConfig(shape, LAYOUTS[layout][1], **kw))
    if case == 'merge3d_model':
        mc = MERGE3D_CASE
        return oracle_action.forward(ops, table, x, mc['num_actions'], mc['num_joints'], mc['num_blocks'],
                                     ksize=mc['reception']['ksize'], output_poses=True, pose_dim=3,
                                     depth_maps=mc['depth_maps'])
    mc = MERGE_CASE
    return oracle_action.forward(ops, table, x, mc['num_actions'], mc['num_joints'], mc['num_blocks'],
                                 mc['reception']['num_context_per_joint'], mc['reception']['ksize'])


@pytest.mark.parametrize('case', ALL_CASES)
def test_weight_list_is_the_references(case):
    z, _ = _fixture(case)
    m, _ = _product(case)
    ref = dict(zip([str(n) for n in z['weight_names']], [str(s) for s in z['weight_shapes']]))
    optional = set(m.optional_weights)
    assert optional == set(str(n) for n in z['optional_in_product'])
    mine = {n: repr(tuple(s)) for n, s in m.weight_specs if n not in optional}
    assert mine == ref
    # nothing the reference freezes as a constant may be expected from a checkpoint
    assert not (set(str(n) for n in z['fixed_names']) & set(n for n, _ in m.weight_specs))


@pytest.mark.parametrize('case', ALL_CASES)
def test_oracle_matches_reference_graph(case):
    z, ref_outs = _fixture(case)
    m, seed = _product(case)
    assert seed == int(z['seed'])
    table = _init_weights(case, m, seed).get_weights()          # host-side only: no device is touched
    x = _input(case, z).astype(np.float64)
    big = case.startswith('spnet') or case.endswith(('fullsize', 'c1_heatmaps'))
    # numpy fp64 oracle on the small graphs, the torch-CPU fp32 op set on the 128x128 SPNets and the full-size
    # ReceptionNet (CPU-suite time)
    outs = _oracle(case, ops_torch if big else ops_np, table, x)
    assert len(outs) == len(ref_outs)
    # the merge model feeds the ill-conditioned context division (see below) into a second network: fp64
    # rounding differences between the two implementations are amplified to ~3e-8 there
    tol = 2e-4 if big else (1e-6 if case.startswith('merge') else 1e-9)
    for o, r in zip(outs, ref_outs):
        assert o.shape == r.shape
        assert np.abs(np.asarray(o, np.float64) - r).max() <= tol * max(1.0, np.abs(r).max())


@pytest.mark.parametrize('case', ALL_CASES)
def test_compiled_plan_matches_reference_graph(case):
    """No oracle in between: the product's COMPILED PLAN for the case (fused launches, planned and aliased buffers),
    executed on the CPU in float64 by tests/plan_emulator.py -- one numpy op per kernel contract of
    include/deephar_b200.h -- reproduces the outputs of the reference's own builder code, at every BASELINE config's
    full size (C1 / C3 one frame, C4 / C5 one 16-frame clip).  What the GPU run adds is the kernels' arithmetic."""
    from plan_emulator import PlanEmulator
    z, ref_outs = _fixture(case)
    m, seed = _product(case)
    _init_weights(case, m, seed)
    x = _input(case, z).astype(np.float64)
    with np.errstate(over='ignore'):
        outs = PlanEmulator(m).run(x)
    assert len(outs) == len(ref_outs)
    for i, (o, r) in enumerate(zip(outs, ref_outs)):
        assert o.shape == r.shape and np.isfinite(o).all(), (case, i)
        # fixtures stored in float32 bound the agreement at ~1e-7; the float64 ones agree to 1e-14
        assert np.abs(o - r).max() <= 2e-6 * max(1.0, np.abs(r).max()), (case, i, float(np.abs(o - r).max()))


@pytest.mark.gpu
@pytest.mark.parametrize('case', ALL_CASES)
def test_product_matches_reference_graph(cuda, case):
    z, ref_outs = _fixture(case)
    m, seed = _product(case)
    _init_weights(case, m, seed)
    x = _input(case, z)
    outs = m.predict(x)
    if not isinstance(outs, (list, tuple)):
        outs = [outs]
    assert len(outs) == len(ref_outs)
    # context-aggregated 2-D poses divide by a sum of raw signed confidences (reception.py:175-180): joints where
    # that sum cancels are ill-conditioned in ANY precision -- bound them by the oracle's condition number and
    # exclude cond > 100 (must be < 2 % of joints), exactly as tests/test_gpu_reception.py does
    cond = None
    if case in RECEPTION_CASES and RECEPTION_CASES[case][1].get('num_context_per_joint') and \
            not RECEPTION_CASES[case][1].get('concat_pose_confidence', True):
        dbg = {}
        oracle_reception.forward(ops_torch if case.endswith(('fullsize', 'c1_heatmaps')) else ops_np, m.get_weights(),
                                 x.astype(np.float64), debug=dbg, **RECEPTION_CASES[case][1])
        cond = [np.asarray(c, dtype=np.float64) for c in dbg['ctx_cond']]
    skipped = total = ties = maps = 0
    per_block = 3 if (case in RECEPTION_CASES and RECEPTION_CASES[case][1].get('export_heatmaps') and
                      not RECEPTION_CASES[case][1].get('concat_pose_confidence', True)) else 2
    for i, (o, r) in enumerate(zip(outs, ref_outs)):
        assert o.shape == r.shape
        scale = np.maximum(np.abs(r), 1.0)
        err = np.abs(o.astype(np.float64) - r) / scale
        lim = 1e-3
        if per_block == 3 and i % per_block == 2:
            # exported heat-maps: north-star "bit-exact for argmax joint indices" -- the arg-max pixel of every
            # joint map must be the reference's, unless the reference's two best pixels are closer than the
            # value tolerance (a tie no fp32 implementation can order)
            n_, h_, w_, c_ = r.shape
            fo, fr = o.reshape(n_, h_ * w_, c_).astype(np.float64), r.reshape(n_, h_ * w_, c_).astype(np.float64)
            top2 = np.sort(fr, axis=1)[:, -2:, :]
            tie = (top2[:, 1] - top2[:, 0]) <= 2e-3 * np.maximum(1.0, np.abs(top2[:, 1]))
            same = fo.argmax(axis=1) == fr.argmax(axis=1)
            assert np.all(same | tie), '%s output %d: arg-max pixel differs on %d maps' % (case, i, int((~(same | tie)).sum()))
            ties += int(tie.sum())
            maps += tie.size
            err = np.abs(o.astype(np.float64) - r) / max(1.0, float(np.abs(r).max()))
        # (the merge-model fixtures use heat-maps that keep the context division well conditioned for every joint
        # -- ref_cases.positive_last_regmap -- so all of p1..p4, v1..v4, m are held to the 1e-3 bar)
        if cond is not None and i % per_block == 0:
            k = cond[i // per_block]
            bad = k > 100.0
            skipped += int(bad.sum())
            total += bad.size
            err = np.where(bad[..., None], 0.0, err)
            lim = np.maximum(1e-3, 0.2 * 1e-3 * k)[..., None]
        assert np.all(err <= lim), '%s output %d: max err %g' % (case, i, float(err.max()))
    if total:
        assert skipped <= max(1, total // 50)
    if maps:
        assert ties <= max(1, maps // 20), '%d of %d heat-maps have an unresolvable top-2 tie' % (ties, maps)


def test_options_off_the_baseline_configs_numerically():
    """For builder arguments the BASELINE configs do not use (no / one context map, alpha, heat-map and feature export,
    depth_maps, 3 pyramid levels, growth, 3x3 kernels, predict_rootz, two action sets, sam_alpha, image_div, pa20j3d,
    other action pyramids): the product's compiled plan, executed by tests/plan_emulator.py, reproduces the outputs of the
    reference's own builder code executed on the eager float64 Keras shim (tests/golden/ref_option_sweep.npz, written by
    make_option_sweep_golden.py) for the same seeded inputs and synthetic weights."""
    import zlib
    from plan_emulator import PlanEmulator
    from ref_cases import option_sweep_inputs, option_sweep_sample_index
    from deephar_b200 import config as pconfig
    z = np.load(os.path.join(HERE, 'golden', 'ref_option_sweep.npz'))
    cases = option_sweep_inputs()
    assert len(cases) == 10
    for i, (kind, spec, x) in enumerate(cases):
        if kind == 'reception':
            m = reception.build((64, 64, 3), 17 if spec['dim'] == 3 else 16, **spec)
        else:
            shape, layout, kw = spec
            m = spnet.build(pconfig.ModelConfig(shape, getattr(pconfig, layout), **kw))
        assert zlib.crc32(np.ascontiguousarray(x, dtype=np.float32).tobytes()) == int(z['x_crc32_%d' % i]), \
            'regenerated input differs from the one the fixture was made with'
        optional = set(m.optional_weights)
        assert sorted(n for n, _ in m.weight_specs if n not in optional) == [str(n) for n in z['names%d' % i]], (i, spec)
        m.init_synthetic_weights(1234)
        with np.errstate(over='ignore'):
            outs = PlanEmulator(m).run(x)
        assert len(outs) == len({f.split('_')[1] for f in z.files if f.startswith('out%d_' % i)}), (i, spec)
        for k, o in enumerate(outs):
            key = 'out%d_%d' % (i, k)
            if key in z.files:
                r = z[key]
                assert o.shape == r.shape, (i, spec, k)
            else:                   # a large output: its shape and the values at fixed positions
                assert o.shape == tuple(z[key + '_shape']), (i, spec, k)
                o, r = o.ravel()[option_sweep_sample_index(o.size)], z[key + '_sample']
            assert np.abs(o - r).max() <= 1e-9 * max(1.0, np.abs(r).max()), (i, spec, k, float(np.abs(o - r).max()))
