"""tests/golden/ref_entry_scripts.json.gz: what the REFERENCE's own entry scripts end up with when they run unmodified on
deephar_b200 (tests/reference_dropin/run_reference_script.py, the forward being the oracle's): every score their
evaluators return, the recording of the model the script re-wired after load_weights (weight list, output expressions,
launches; for the multitask scripts the full model and split_model's views of it), and the cameras / poses of the
Human3.6M stand-in.  Runs where the reference tree exists; tests/test_keras_compat.py rebuilds the same re-wiring with
keras_compat, compares it with the recording and recomputes the scores from the oracle and from the product's own
Model.predict of the re-wired model (tests/reference_dropin/standins.py).

Before writing, the script checks what a run of the reference scripts shows and the file cannot hold: the evaluators
raised nothing (the multi-clip ones swallow predict() errors), they returned the scores recomputed from the oracle's
outputs, the re-wired model holds the loaded weights, its buffer plan replays memory-safe and, executed on the CPU,
computes the oracle's outputs; and, with the product's own Model.predict under the pose scripts' evaluators
(tests/fake_cuda.py --arithmetic), the scores agree with the oracle's to 1e-4.

    DEEPHAR_REFERENCE=<reference checkout> python tests/golden/make_entry_script_golden.py
"""
import gzip
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
RUNNER = os.path.join(TESTS, 'reference_dropin', 'run_reference_script.py')
PATH = os.path.join(HERE, 'ref_entry_scripts.json.gz')
CASES = ('mpii', 'h36m', 'penn_multitask', 'ntu_multitask')
ON_PREDICT = ('mpii', 'h36m')


def start(case, tmp, own_predict):
    work = os.path.join(tmp, case + ('_predict' if own_predict else ''))
    os.makedirs(os.path.join(work, 'checkout'))
    env = dict(os.environ, KERAS_HOME=os.path.join(work, 'keras'))
    cmd = [sys.executable, RUNNER, case, os.path.join(work, 'checkout')]
    if own_predict:
        env['DEEPHAR_B200_SCRIPT_ON_GPU'] = '1'
        cmd = [sys.executable, os.path.join(TESTS, 'fake_cuda.py'), '--arithmetic'] + cmd[1:]
    return subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env)


def finish(proc, own_predict):
    out, err = proc.communicate()
    assert proc.returncode == 0, err[-3000:]
    assert 'exception on sample' not in out + err
    got = json.loads([l for l in out.splitlines() if l.startswith('{')][-1])
    assert got['model_class'] == 'deephar_b200.keras_compat.Model'
    assert got['forward'] == ('Model.predict' if own_predict else 'oracle (CPU stand-in)')
    m = got['model']
    assert m['weights_are_the_files'] and m['plan_checked'] > m['launches'] and m['plan_emulation_max_err'] < 5e-4, m
    assert sorted(got['returned']) == sorted(got['oracle'])
    for fn, vs in got['returned'].items():
        assert len(vs) == 1
        for a, b in zip(vs[0], got['oracle'][fn][0]):
            assert abs(a - b) <= (1e-4 if own_predict else 1e-9) * abs(b) + 1e-12, (fn, a, b)
    return got


def main():
    if not os.path.isdir(os.environ.get('DEEPHAR_REFERENCE', '')):
        raise SystemExit('set DEEPHAR_REFERENCE to the reference checkout')
    blob = {}
    with tempfile.TemporaryDirectory() as tmp:
        runs = [(case, False, start(case, tmp, False)) for case in CASES]
        runs += [(case, True, start(case, tmp, True)) for case in ON_PREDICT]
        for case, own_predict, proc in runs:
            got = finish(proc, own_predict)
            print(case, '(Model.predict)' if own_predict else '', got['returned'], flush=True)
            if not own_predict:
                rec = {k: got['model'][k] for k in ('weight_specs', 'signatures', 'plan', 'optional_weights', 'output_shape')}
                blob[case] = {'returned': got['returned'], 'output_shape': got['output_shape'], 'standin': got['standin'],
                              'model': rec, 'split': got['split']}
    with open(PATH, 'wb') as f:
        f.write(gzip.compress(json.dumps(blob, sort_keys=True).encode(), 9, mtime=0))
    print('%s: %.0f KB' % (PATH, os.path.getsize(PATH) / 1024.0))


if __name__ == '__main__':
    main()
