"""Runs one of the reference's ENTRY SCRIPTS, unmodified (runpy), on deephar_b200 after dropin.install():

    mpii           : exp/mpii/eval_mpii_singleperson.py       (BASELINE configs[0]/[1]: the headline model's evaluator)
    h36m           : exp/h36m/eval_h36m.py                    (BASELINE configs[2])
    penn_multitask : exp/pennaction/eval_penn_multitask.py    (BASELINE configs[3], 8-frame clips as the script has them)
    ntu_multitask  : exp/ntu/eval_ntu_multitask.py            (BASELINE configs[4], 8-frame clips)

    python run_reference_script.py <case> <empty working directory>

Everything model-side of the script is the product's: `reception.build` / `spnet.build` record the deephar_b200 model,
`get_file` finds the weight file in the Keras cache, `load_weights(path[, by_name=True])` reads the Keras HDF5 file, the
scripts' own re-wiring -- `Model(model.input, [concatenate([pose_b, vis_b]) ...])` made AFTER load_weights, `split_model`
-- compiles on the same layers and keeps their weights, and the reference's own evaluators (exp/common/*_tools.py) drive
`model.predict`.  What is NOT the product's, because it does not exist in the container: the datasets (seeded stand-ins for
`deephar.data.*` returning what the scripts unpack), the released checkpoints (seeded weights in the same Keras HDF5
layout, written by deephar_b200.keras_h5.save where each script looks for its file) and -- on CPU only -- the forward
itself: without a GPU `Model.predict` is the oracle's forward behind the product's own input checks (TEST
INFRASTRUCTURE; set DEEPHAR_B200_SCRIPT_ON_GPU=1 on a B200 to run the real one).  One stale name is aliased:
eval_penn_multitask.py imports `eval_singleclip_generator`, which exp/common/penn_tools.py has since renamed to
`eval_singleclip_gt_bbox_generator` (the script fails with ImportError on the reference's own stack too).

Prints one JSON line: every score an evaluator returned to the script, the same scores recomputed from the oracle's outputs
alone (standins.py), what the compiled model looks like and, for h36m, the cameras and poses of the stand-in dataset.
tests/golden/make_entry_script_golden.py stores it for tests/test_keras_compat.py.

    DEEPHAR_REFERENCE=<reference checkout> python run_reference_script.py <case> <empty working directory>
"""
import contextlib
import io
import json
import os
import runpy
import sys
import types
import warnings

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get('DEEPHAR_REFERENCE', '')
if not os.path.isdir(REF):
    raise SystemExit('set DEEPHAR_REFERENCE to the reference checkout')
sys.path[:0] = [REF, ROOT]
warnings.filterwarnings('ignore')
import numpy as np  # noqa: E402

import deephar_b200.dropin  # noqa: E402
deephar_b200.dropin.install()
_stderr, sys.stderr = sys.stderr, open(os.devnull, 'w')       # the reference prints a banner on import
import deephar  # noqa: E402,F401
import deephar.data  # noqa: E402
sys.stderr = _stderr

from deephar_b200 import keras_h5  # noqa: E402
from deephar_b200 import model as product_model  # noqa: E402
from oracle import postprocess as oracle_post  # noqa: E402
sys.path.insert(0, HERE)
from standins import (CASES, ClipDataset, N_FRAMES, Oracle, T, describe_script_model,  # noqa: E402
                      expected_action_scores, expected_pckh, h36m_frames, mpii_batches, set_clip_labels)

ON_GPU = os.environ.get('DEEPHAR_B200_SCRIPT_ON_GPU') == '1'


def install_oracle_predict(oracle):
    """CPU stand-in for the device forward: the product's own input handling, then the oracle (see the module docstring)."""
    def predict(self, x, batch_size=32, verbose=0):
        x = self._host_input(x)
        outs = oracle(self.get_weights(), x)
        if len(self.graph.outputs) == len(outs) // 2:           # the script's re-wrapped model: [pose_b | vis_b] per block
            outs = [np.concatenate([outs[2 * b], outs[2 * b + 1]], axis=-1) for b in range(len(outs) // 2)]
        assert [tuple(o.shape[1:]) for o in outs] == [tuple(s[1:]) for s in self.output_shape]
        return outs[0] if len(outs) == 1 else outs
    product_model.Model.predict = predict


# ---- stand-ins for the datasets (the rest: standins.py) ---------------------------------------------------------
def h36m_batches(n):
    from deephar.utils.camera import Camera
    rng = np.random.default_rng(36)
    x, afmat = h36m_frames(n)
    nj = 17
    scam, pose_w, uvd = [], np.zeros((n, nj, 3)), np.zeros((n, nj, 3))
    for i in range(n):
        q, _ = np.linalg.qr(rng.normal(size=(3, 3)))
        if np.linalg.det(q) < 0:
            q[:, 0] = -q[:, 0]
        cam = Camera(q, rng.normal(0, 500, 3), rng.uniform(1100, 1200, 2), rng.uniform(480, 540, 2),
                     rng.normal(0, 1e-3, 2), rng.normal(0, 5e-3, 3))
        scam.append(cam.serialize())
        pts = np.concatenate([rng.normal(0, 400, (nj, 2)), rng.uniform(4000, 6000, (nj, 1))], axis=1)
        pose_w[i] = (np.matmul(cam.R_inv, pts.T) + cam.t).T
        uvd[i] = cam.project(pose_w[i])
    import deephar.data.human36m as h36m_data
    h36m_data.ACTION_LABELS = ['action%02d' % i for i in range(15)]      # set by the loader when it reads the annotations
    return [x], [pose_w, uvd, afmat, np.array(scam), rng.integers(0, 15, (n, 1))]


class FrameDataset(object):
    """MpiiSinglePerson / Human36M with topology='frames': only its length is asked for."""
    n = N_FRAMES

    def __init__(self, *args, **kwargs):
        pass

    def get_length(self, mode):
        return self.n


def make_loader(frame_batches):
    class Loader(object):
        """BatchLoader(dataset, x_keys, y_keys, mode, batch_size=..., shuffle=False)"""

        def __init__(self, dataset, *args, **kwargs):
            self.dataset = dataset

        def __len__(self):
            return self.dataset.get_length(None)

        def __getitem__(self, i):
            if isinstance(self.dataset, FrameDataset):
                return frame_batches
            d = self.dataset.get_data(i, None, frame_list=[0])
            return [d['frame'][None]], [d[self.dataset.key][None]]
    return Loader


def main():
    name, workdir = sys.argv[1], os.path.abspath(sys.argv[2])
    case = CASES[name]
    oracle = Oracle(case)

    # working directory laid out as the scripts expect to find the reference checkout (it is read-only, and they write)
    os.makedirs(os.path.join(workdir, 'datasets', 'PennAction'), exist_ok=True)
    os.symlink(os.path.join(REF, 'exp'), os.path.join(workdir, 'exp'))
    with open(os.path.join(workdir, 'datasets', 'PennAction', 'penn_pred_bboxes_multitask.json'), 'w') as f:
        f.write('{}')
    # the "released checkpoint": seeded weights in the Keras HDF5 layout, where the script looks for its file
    if 'cache' in case:
        path = os.path.join(os.path.expanduser(os.environ.get('KERAS_HOME') or os.path.join('~', '.keras')), 'models',
                            case['cache'])
    else:
        path = os.path.join(workdir, case['local'])
    os.makedirs(os.path.dirname(path), exist_ok=True)
    keras_h5.save(path, oracle.model.weight_specs, oracle.table)

    # datasets
    if name == 'penn_multitask':
        FrameDataset.n = T                                      # the pose model of a clip network takes T frames at a time
    frames = h36m_batches(FrameDataset.n) if name == 'h36m' else mpii_batches(FrameDataset.n)
    if 'action' in case:
        set_clip_labels(oracle, case)
    for cls in ('MpiiSinglePerson', 'Human36M'):
        setattr(deephar.data, cls, FrameDataset)
    for cls in ('PennAction', 'Ntu'):
        setattr(deephar.data, cls, ClipDataset)
    deephar.data.BatchLoader = make_loader(frames)
    sys.modules['annothelper'] = types.ModuleType('annothelper')
    for fn in ('check_mpii_dataset', 'check_h36m_dataset', 'check_pennaction_dataset', 'check_ntu_dataset'):
        setattr(sys.modules['annothelper'], fn, lambda: None)
    np.float = float                                            # the reference predates numpy 1.24

    # the evaluators the script imports, wrapped to keep what they return (the scripts only print it)
    sys.path.append(os.path.join(REF, 'exp', 'common'))
    returned = {}
    import mpii_tools, h36m_tools, penn_tools, ntu_tools        # noqa: E401
    penn_tools.eval_singleclip_generator = penn_tools.eval_singleclip_gt_bbox_generator       # stale name, see docstring

    class OldNumpy(types.ModuleType):
        """numpy as the reference knew it (1.14): `np.float`, and `np.equal(a, b, dtype=np.float)` (penn_tools.py:69)"""

        def __getattr__(self, attr):
            return getattr(np, attr)
    old = OldNumpy('numpy')
    old.equal = lambda a, b, dtype=None: np.equal(a, b) if dtype is None else np.equal(a, b).astype(dtype)
    penn_tools.np = ntu_tools.np = old

    def recording(mod, fn):
        inner = getattr(mod, fn)

        def wrapper(*args, **kwargs):
            out = inner(*args, **kwargs)
            returned.setdefault(fn, []).append([float(s) for s in out])
            return out
        setattr(mod, fn, wrapper)
    recording(mpii_tools, 'eval_singleperson_pckh')
    recording(h36m_tools, 'eval_human36m_sc_error')
    recording(penn_tools, 'eval_singleclip_generator')
    recording(penn_tools, 'eval_multiclip_dataset')
    recording(ntu_tools, 'eval_multiclip_dataset')

    if not ON_GPU:
        install_oracle_predict(oracle)

    os.chdir(workdir)
    sys.argv = [os.path.join(REF, case['script'])]
    printed = io.StringIO()
    with contextlib.redirect_stdout(printed):
        g = runpy.run_path(sys.argv[0], run_name='__main__')

    # ---- what the script ended up with ----
    want = {}
    if name in ('mpii', 'h36m'):
        model = g['model']
        x = frames[0][0]
        ref = oracle(oracle.table, x)
        if name == 'mpii':
            want['eval_singleperson_pckh'] = [expected_pckh(oracle, x, g['p_val'], g['afmat_val'], g['head_val'],
                                                            len(ref) // 2, clip=False)]
        else:
            want['eval_human36m_sc_error'] = [oracle_post.human36m_mpjpe(
                [ref[2 * b] for b in range(len(ref) // 2)], g['afmat_val'], g['puvd_val'][:, 0, 2], g['scam_val'], g['pw_val'])]
        full = model
    else:
        full = g['full_model']
        pose_model, action_model = g['models']
        n_pose = len(pose_model.outputs)
        ds = g['penn_seq'] if name == 'penn_multitask' else g['ntu']
        single, multi = expected_action_scores(oracle, ds, n_pose)
        if name == 'penn_multitask':
            want['eval_singleclip_generator'] = [single]
            want['eval_multiclip_dataset'] = [multi]
            want['eval_singleperson_pckh'] = [expected_pckh(oracle, g['x_val'], g['p_val'], g['afmat_val'], g['head_val'],
                                                            n_pose, clip=True)]
        else:
            want['eval_multiclip_dataset'] = [multi]
        model = action_model
    model_desc, split = describe_script_model(name, oracle, full, [model] if name in ('mpii', 'h36m') else g['models'])
    standin = {}
    if name == 'h36m':
        standin = {'pose_w': g['pw_val'].tolist(), 'uvd': g['puvd_val'].tolist(), 'scam': np.asarray(g['scam_val']).tolist()}
    print(json.dumps({
        'returned': returned, 'standin': standin, 'model': model_desc, 'split': split,
        'oracle': {k: [[float(s) for s in v] for v in vs] for k, vs in want.items()},
        'model_class': type(model).__module__ + '.' + type(model).__name__, 'n_outputs': len(model.outputs),
        'output_shape': [list(s) for s in model.output_shape], 'script_printed': printed.getvalue()[-600:],
        'forward': 'Model.predict' if ON_GPU else 'oracle (CPU stand-in)'}))


if __name__ == '__main__':
    main()
