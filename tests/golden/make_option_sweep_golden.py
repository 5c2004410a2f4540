"""tests/golden/ref_option_sweep.npz: outputs of the REFERENCE's own builder code for builder options OFF the BASELINE
configs (the tables OPTION_SWEEP_* of ref_cases.py).  Runs where the reference tree exists (DEEPHAR_REFERENCE).

For each configuration the reference's reception.build / spnet.build (unmodified) is EXECUTED on tests/golden/keras_shim
(eager float64) with the product's synthetic weights assigned by name -- the recipe of make_reference_golden.py, whose
helpers are reused -- on the seeded inputs of ref_cases.option_sweep_inputs().  Stored per configuration i: the
reference's trainable weight names (`names<i>`), its outputs in float64 (`out<i>_<k>`; of an output larger than
ref_cases.OPTION_SWEEP_SAMPLE its shape and a fixed sample of its values) and the CRC32 of the float32 input
(`x_crc32_<i>`).  tests/test_reference_golden.py executes the product's compiled plan on the same inputs and compares.

    DEEPHAR_REFERENCE=<reference checkout> python tests/golden/make_option_sweep_golden.py
"""
import os
import sys
import zlib

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import make_reference_golden as G  # noqa: E402  (puts the shim, the reference and the repo on sys.path)

import numpy as np  # noqa: E402
from ref_cases import option_sweep_inputs, option_sweep_store  # noqa: E402

from deephar.utils import pose as ref_pose  # noqa: E402
from deephar_b200 import config as pconfig  # noqa: E402


def record(blob, i, ref_model, prod_model, x, seed=1234):
    ws = G.collect(ref_model)
    trainable = {n: w for n, w, frozen in ws if not frozen}
    optional = set(prod_model.optional_weights)
    live = {n for n, _ in prod_model.weight_specs if n not in optional}
    assert live == set(trainable), (i, sorted(live ^ set(trainable))[:6])
    prod_model.init_synthetic_weights(seed)
    table = prod_model.get_weights()
    for n, w in trainable.items():
        w['value'] = np.asarray(table[n], dtype=np.float64)
    outs = ref_model.predict(np.asarray(x, dtype=np.float64))
    outs = outs if isinstance(outs, (list, tuple)) else [outs]
    blob['names%d' % i] = np.array(sorted(trainable))
    blob['x_crc32_%d' % i] = np.array(zlib.crc32(np.ascontiguousarray(x, dtype=np.float32).tobytes()))
    for k, o in enumerate(outs):
        option_sweep_store(blob, 'out%d_%d' % (i, k), o)


def main():
    blob = {}
    for i, (kind, spec, x) in enumerate(option_sweep_inputs()):
        G.fresh_process_state()
        if kind == 'reception':
            nj = 17 if spec['dim'] == 3 else 16
            record(blob, i, G.ref_reception.build((64, 64, 3), nj, **spec), G.reception.build((64, 64, 3), nj, **spec), x)
        else:
            shape, layout, kw = spec
            ref = G.ref_spnet.build(G.RefModelConfig(shape, getattr(ref_pose, layout), **kw))
            prod = G.spnet.build(pconfig.ModelConfig(shape, getattr(pconfig, layout), **kw))
            record(blob, i, ref, prod, x)
        print(i, kind, 'done', flush=True)
    path = os.path.join(HERE, 'ref_option_sweep.npz')
    np.savez_compressed(path, **blob)
    print('%s: %.0f KB' % (path, os.path.getsize(path) / 1024.0))


if __name__ == '__main__':
    main()
