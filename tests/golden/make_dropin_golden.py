"""tests/golden/ref_dropin_models.json.gz: the models the REFERENCE's own builder code records on the recording keras
(deephar_b200.dropin; tests/reference_dropin/run_reference_backbone.py), one entry per case -- weight lists with their
Keras auto-names, kernel plans, output shapes, output expression digests and the exceptions builders raise.  Runs where
the reference tree exists; tests/test_keras_compat.py checks deephar_b200's own builders against the file.

    DEEPHAR_REFERENCE=<reference checkout> python tests/golden/make_dropin_golden.py
"""
import gzip
import json
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
RUNNER = os.path.join(os.path.dirname(HERE), 'reference_dropin', 'run_reference_backbone.py')
PATH = os.path.join(HERE, 'ref_dropin_models.json.gz')

# run_reference_backbone.py arguments; the joined arguments are the case's key in the file
CASES = ('3', 'spnet', 'full2d 0', 'full2d 1', 'full3d', 'spnet_full penn', 'spnet_full ntu', 'merge 2', 'merge 3',
         'merge 2 v2', 'sweep')


def main():
    if not os.path.isdir(os.environ.get('DEEPHAR_REFERENCE', '')):
        raise SystemExit('set DEEPHAR_REFERENCE to the reference checkout')
    blob = {}
    for case in CASES:
        out = subprocess.run([sys.executable, RUNNER] + case.split(), capture_output=True, text=True, check=True)
        blob[case] = [json.loads(l) for l in out.stdout.splitlines() if l.startswith('{')]
        print(case, len(blob[case]), 'lines', flush=True)
    with open(PATH, 'wb') as f:
        f.write(gzip.compress(json.dumps(blob, sort_keys=True).encode(), 9, mtime=0))
    print('%s: %.0f KB' % (PATH, os.path.getsize(PATH) / 1024.0))


if __name__ == '__main__':
    main()
