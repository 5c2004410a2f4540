"""The stand-ins the reference's entry scripts run on (tests/reference_dropin/run_reference_script.py), and the scores
their evaluators must return, recomputed without the reference: seeded datasets, the case models with their seeded
weights, and the PCKh / MPJPE / action accuracies from a forward's outputs (the oracle's, or the product's own
Model.predict).

    python standins.py <case> [predict]

prints one JSON line: {'returned': {evaluator: [scores]}} from the oracle's outputs (or from Model.predict of the model the
script evaluates), and 'model' / 'split': the script's final model rebuilt with keras_compat (script_models).
"""
import gzip
import hashlib
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

from deephar_b200 import reception as product_reception  # noqa: E402
from deephar_b200 import spnet as product_spnet  # noqa: E402
from deephar_b200.config import ModelConfig as ProductConfig  # noqa: E402
from deephar_b200.config import pa16j2d as product_pa16j2d  # noqa: E402
from deephar_b200.config import pa17j3d as product_pa17j3d  # noqa: E402
from oracle import ops_torch, synth  # noqa: E402
from oracle import postprocess as oracle_post  # noqa: E402
from oracle import reception as oracle_reception  # noqa: E402
from oracle import spnet as oracle_spnet  # noqa: E402

T = 8                                   # num_frames of both multitask scripts
N_FRAMES = 3                            # frames in the MPII / Human3.6M stand-in datasets

PENN_KW = dict(num_actions=[15], num_pyramids=6, action_pyramids=[5, 6], num_levels=4, pose_replica=True,
               num_pose_features=160, num_visual_features=160)
NTU_KW = dict(num_actions=[60], num_pyramids=2, action_pyramids=[1, 2], num_levels=4, pose_replica=False,
              num_pose_features=192, num_visual_features=192)
CASES = {
    'mpii': dict(script='exp/mpii/eval_mpii_singleperson.py', cache='weights_PE_MPII_cvpr18_19-09-2017.h5',
                 reception=dict(num_joints=16, dim=2, num_blocks=8, num_context_per_joint=2, ksize=(5, 5),
                                concat_pose_confidence=False)),
    'h36m': dict(script='exp/h36m/eval_h36m.py', cache='weights_3DPE_H36M_cvpr18_Nov-2017.h5',
                 reception=dict(num_joints=17, dim=3, num_blocks=8, ksize=(5, 5), concat_pose_confidence=False)),
    'penn_multitask': dict(script='exp/pennaction/eval_penn_multitask.py', local='weights/weights_mpii+penn_ar_028.hdf5',
                           spnet=(PENN_KW, product_pa16j2d, oracle_spnet.pa16j2d), action=('pennaction', 15),
                           split=('2DPose', '2DAction')),
    'ntu_multitask': dict(script='exp/ntu/eval_ntu_multitask.py',
                          local='output/ntu_spnet_trial-03-ft_replica_0ae2bf7/weights_3dp+ntu_ar_062.hdf5',
                          spnet=(NTU_KW, product_pa17j3d, oracle_spnet.pa17j3d), action=('ntuaction', 60),
                          split=('3DPose', '3DAction')),
}


class Oracle(object):
    """The CPU oracle's forward of the case's model: all outputs of the FULL model, as float32 arrays."""

    def __init__(self, case):
        self.case = case
        if 'reception' in case:
            self.model = product_reception.build((256, 256, 3), **case['reception'])
        else:
            kw, layout, olayout = case['spnet']
            self.model = product_spnet.build(ProductConfig((T, 256, 256, 3), layout, **kw))
            self.ocfg = oracle_spnet.ModelConfig((T, 256, 256, 3), olayout, **kw)
        self.model.init_synthetic_weights(77)
        self.table = self.model.get_weights()
        self.memo = {}

    def __call__(self, table, x):
        key = (x.shape, hashlib.sha1(np.ascontiguousarray(x).tobytes()).hexdigest())
        if key not in self.memo:
            if 'reception' in self.case:
                outs = oracle_reception.forward(ops_torch, table, x, **self.case['reception'])
            else:
                outs = oracle_spnet.forward(ops_torch, table, x, self.ocfg)
            self.memo[key] = [np.asarray(o, np.float32) for o in outs]
        return self.memo[key]


class PredictForward(object):
    """The same call on the product's own Model.predict of the model a pose script evaluates (script_models: one
    concatenate([pose, visibility]) output per block), its outputs split back into (pose, visibility) pairs."""

    def __init__(self, oracle, model):
        self.table, self.model = oracle.table, model

    def __call__(self, table, x):
        assert table is self.table
        outs = self.model.predict(x)
        outs = outs if isinstance(outs, list) else [outs]
        return [np.asarray(p, np.float32) for o in outs for p in (o[..., :-1], o[..., -1:])]


def script_models(name, oracle):
    """The models the case's entry script ends up with, rebuilt with keras_compat on the product's builder: the full
    model with the case's weights loaded (load_weights), then -- made AFTER that, on its tensors -- one
    concatenate([pose, visibility], name='blk<b>') output per block (eval_mpii_singleperson.py:56-61, eval_h36m.py:55-60),
    or split_model's pose and action models (spnet.py:417-448, interlaced=False).  -> (full, [the models the script
    keeps])"""
    from deephar_b200 import keras_compat as K
    case = CASES[name]
    g = oracle.model.graph
    full = K.Model(g.inputs[0], list(g.outputs), name=oracle.model.name)
    full.set_weights(oracle.table)
    if 'reception' in case:
        outs = [K.concatenate([full.outputs[2 * b], full.outputs[2 * b + 1]], name='blk%d' % (b + 1))
                for b in range(len(full.outputs) // 2)]
        return full, [K.Model(full.input, outs, name=full.name)]
    kw = case['spnet'][0]
    n_pose = product_spnet.get_num_predictions(kw['num_pyramids'], kw['num_levels'])
    return full, [K.Model(full.input, full.outputs[:n_pose], name=case['split'][0]),
                  K.Model(full.input, full.outputs[n_pose:], name=case['split'][1])]


def describe_script_model(name, oracle, full, kept):
    """What the script ended up with: the recording of the model whose plan runs (the re-wired model of a pose script,
    the full model of a multitask one -- its split models are views of it): weight list, output expressions, launches;
    whether it holds the loaded weights; the launches compiler.verify_plan replays memory-safe; and how far its plan,
    executed on the CPU (tests/plan_emulator.py), is from the oracle's outputs for one item.  `split`: name, number of
    outputs, output shapes and whether it is a view of the full network, per model the script keeps."""
    from deephar_b200.compiler import verify_plan
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    from plan_emulator import PlanEmulator
    impl = (kept[0] if 'reception' in CASES[name] else full)._compiled()
    if 'reception' in CASES[name]:
        x1 = (mpii_batches(N_FRAMES)[0][0] if name == 'mpii' else h36m_frames(N_FRAMES)[0])[:1]
        ref1 = oracle(oracle.table, x1)
        ref1 = [np.concatenate([ref1[2 * b], ref1[2 * b + 1]], axis=-1) for b in range(len(ref1) // 2)]
    else:
        x1 = ClipDataset(None, None).clip(0, 0, 0)[None]
        ref1 = oracle(oracle.table, x1)
    with np.errstate(over='ignore'):
        emu = PlanEmulator(impl).run(x1)
    assert len(emu) == len(ref1) and all(o.shape == r.shape for o, r in zip(emu, ref1))
    held = impl.get_weights()
    model = {
        'weight_specs': [[n, list(s)] for n, s in impl.weight_specs], 'signatures': impl.graph.signatures(),
        'plan': [[k.kind, [list(t.shape) for t in k.outs]] for k in impl.plan.kops],
        'optional_weights': list(impl.optional_weights), 'output_shape': [list(s) for s in impl.output_shape],
        'weights_are_the_files': set(held) == set(oracle.table) and all(np.array_equal(held[k], oracle.table[k])
                                                                       for k in oracle.table),
        'launches': len(impl.plan.kops), 'plan_checked': verify_plan(impl.plan, impl.graph),
        'plan_emulation_max_err': max(float(np.abs(o - r).max()) for o, r in zip(emu, ref1))}
    split = [[m.name, len(m.outputs), [list(s) for s in m.output_shape], m._compiled().full is full._compiled()]
             for m in kept] if 'spnet' in CASES[name] else []
    return model, split


# ---- stand-ins for the datasets -------------------------------------------------------------------------------------
def mpii_batches(n):
    rng = np.random.default_rng(11)
    x = synth.synth_frames(n, 256, 256, seed=21)
    pose = np.concatenate([rng.uniform(0.2, 0.8, (n, 16, 2)), np.ones((n, 16, 1))], axis=-1)
    afmat = np.tile(np.array([[1 / 300.0, 0, 0.05], [0, 1 / 300.0, 0.1], [0, 0, 1]]), (n, 1, 1))
    head = rng.uniform(40, 60, (n, 1))
    return [x], [pose, afmat, head]


def h36m_frames(n):
    """The frames and crop maps of the Human3.6M stand-in (its cameras and poses: h36m_batches of run_reference_script.py)."""
    afmat = np.zeros((n, 3, 3))
    afmat[:, 0, 0] = afmat[:, 1, 1] = 1 / 500.0
    afmat[:, 0, 2], afmat[:, 1, 2], afmat[:, 2, 2] = -0.3, -0.2, 1.0
    return synth.synth_frames(n, 256, 256, seed=22), afmat


class ClipDataset(object):
    """PennAction / Ntu with topology='sequences': two test sequences of two clips each; the loader honours
    `dataconf.fixed_hflip` as the real one does (deephar/data/pennaction.py:135-160)."""
    key, n_actions, labels = 'pennaction', 15, (0, 0)

    def __init__(self, path, dataconf, *args, **kwargs):
        self.dataconf = dataconf
        self.use_gt_bbox = kwargs.get('use_gt_bbox', True)

    def get_length(self, mode):
        return 2

    def get_shape(self, key):
        assert key == self.key
        return (self.n_actions,)

    def get_clip_index(self, i, mode, subsamples=[1]):
        return [list(range(T)), list(range(3, 3 + T))]

    def clip(self, i, start, hflip):
        x = synth.synth_frames(T, 256, 256, seed=100 + 10 * i + start)
        return x[:, :, ::-1].copy() if hflip else x

    def get_data(self, i, mode, frame_list=None, bbox=None):
        onehot = np.zeros(self.n_actions)
        onehot[self.labels[i]] = 1
        return {'frame': self.clip(i, frame_list[0], self.dataconf.fixed_hflip), self.key: onehot}


def set_clip_labels(forward, case):
    """Ground truth of the clip stand-in: sequence 0 is labelled with what the last prediction block says about it
    (multi-clip product), sequence 1 with another class -- so that the accuracies are neither all 0 nor all 100."""
    ClipDataset.key, ClipDataset.n_actions = case['action']
    probe = ClipDataset(None, None)
    last = []
    for i in range(2):
        prod = np.ones(ClipDataset.n_actions)
        for fl in probe.get_clip_index(i, None):
            for hflip in (0, 1):
                prod = prod * forward(forward.table, probe.clip(i, fl[0], hflip)[None])[-1][0]
        last.append(int(np.argmax(prod)))
    ClipDataset.labels = (last[0], (last[1] + 1) % ClipDataset.n_actions)


# ---- the scores from a forward's outputs alone ----------------------------------------------------------------------
def expected_pckh(forward, x, pose, afmat, head, n_pose_outputs, clip):
    xin = x.reshape((-1, T) + x.shape[1:]) if clip else x
    ref = forward(forward.table, xin)
    y_true = oracle_post.transform_pose_sequence(afmat, pose[:, :, 0:2], inverse=True)
    out = []
    for b in range(n_pose_outputs):
        p = ref[b if clip else 2 * b]
        p = p.reshape((-1,) + p.shape[-2:])[:, :, 0:2]
        out.append(oracle_post.pckh(y_true, oracle_post.transform_pose_sequence(afmat, p, inverse=True), head, 0.5))
    return out


def expected_action_scores(forward, ds, first_action_output):
    """exp/common/penn_tools.py:42-82 (single clip, accuracy as a fraction) and :85-150 / ntu_tools.py:53-140 (product
    over clips x h-flip, accuracy in %)."""
    n = ds.get_length(None)
    single = [forward(forward.table, ds.clip(i, 0, 0)[None])[first_action_output:] for i in range(n)]
    nb = len(single[0])
    sc_single = [float(np.mean([np.argmax(single[i][b][0]) == ds.labels[i] for i in range(n)])) for b in range(nb)]
    prod = np.ones((nb, n, ds.n_actions))
    for i in range(n):
        for fl in ds.get_clip_index(i, None):
            for hflip in (0, 1):
                pred = forward(forward.table, ds.clip(i, fl[0], hflip)[None])[first_action_output:]
                for b in range(nb):
                    prod[b, i] *= pred[b][0]
    sc_multi = [float(100.0 * np.sum(np.argmax(prod[b], axis=-1) == np.array(ds.labels)) / n) for b in range(nb)]
    return sc_single, sc_multi


def expected_scores(name, forward, h36m=None):
    """{evaluator: [scores]} the case's script must get back from its evaluators on the stand-ins, computed from
    `forward`'s outputs.  h36m: {pose_w, uvd, scam} of the Human3.6M stand-in."""
    case = CASES[name]
    if name == 'mpii':
        (x,), (pose, afmat, head) = mpii_batches(N_FRAMES)
        n_pose = len(forward(forward.table, x)) // 2
        return {'eval_singleperson_pckh': expected_pckh(forward, x, pose, afmat, head, n_pose, clip=False)}
    if name == 'h36m':
        x, afmat = h36m_frames(N_FRAMES)
        ref = forward(forward.table, x)
        return {'eval_human36m_sc_error': list(oracle_post.human36m_mpjpe(
            [ref[2 * b] for b in range(len(ref) // 2)], afmat, np.asarray(h36m['uvd'])[:, 0, 2], np.asarray(h36m['scam']),
            np.asarray(h36m['pose_w'])))}
    set_clip_labels(forward, case)
    ds = ClipDataset(None, None)
    n_pose = product_spnet.get_num_predictions(case['spnet'][0]['num_pyramids'], case['spnet'][0]['num_levels'])
    single, multi = expected_action_scores(forward, ds, n_pose)
    if name == 'ntu_multitask':
        return {'eval_multiclip_dataset': multi}
    (x,), (pose, afmat, head) = mpii_batches(T)
    return {'eval_singleclip_generator': single, 'eval_multiclip_dataset': multi,
            'eval_singleperson_pckh': expected_pckh(forward, x, pose, afmat, head, n_pose, clip=True)}


def main():
    name = sys.argv[1]
    oracle = Oracle(CASES[name])
    full, kept = script_models(name, oracle)
    forward = PredictForward(oracle, kept[0]) if sys.argv[2:] == ['predict'] else oracle
    h36m = None
    if name == 'h36m':
        with gzip.open(os.path.join(ROOT, 'tests', 'golden', 'ref_entry_scripts.json.gz')) as f:
            h36m = json.load(f)['h36m']['standin']
    scores = expected_scores(name, forward, h36m)
    model, split = describe_script_model(name, oracle, full, kept)
    print(json.dumps({'returned': {k: [float(s) for s in v] for k, v in scores.items()}, 'model': model, 'split': split}))


if __name__ == '__main__':
    main()
