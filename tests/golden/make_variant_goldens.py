"""Golden compiled models: every model variant that tests/test_model_variants.py and tests/test_model.py compile, as
`flybody_b200.compiler` compiled them from the reference's `fruitfly.xml`.  The tests compile afresh and compare with these, so a
change to the compiler's output shows; rerun this when such a change is intended.
    python tests/golden/make_variant_goldens.py [ASSETS_DIR]      -> tests/golden/model_variants.tar.xz
ASSETS_DIR defaults to tests/golden/fruitfly_assets.
The archive holds one uncompressed .npz per model (the layout of `compile_model.save_model`) and `index.json` (member ->
variant + compile_variant keyword arguments), xz-compressed as a whole: the variants differ in a few arrays, so the archive
is ~40 KB where separate compressed .npz files would take ~2.7 MB."""
import io
import json
import os
import sys
import tarfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'model_variants.tar.xz')

JOINT_FILTER, ADHESION_FILTER = 0.0123, 0.0234                     # the filter constants of tests/test_model_variants.py
USES = [(i, j, k, l) for i in range(2) for j in range(2) for k in range(2) for l in range(2)]
FILTERS = [(0, 0), (JOINT_FILTER, 0), (0, ADHESION_FILTER), (JOINT_FILTER, ADHESION_FILTER)]


def variants():
    """(variant, compile_variant kwargs) of every model the tests use"""
    out = [('walk', {}), ('flight', {})]                                # the shipped models, compiled afresh
    for use in USES:
        for flt in FILTERS:
            out.append(('walker', dict(use_legs=bool(use[0]), use_wings=bool(use[1]), use_mouth=bool(use[2]), use_antennae=bool(use[3]),
                                       joint_filter=flt[0], adhesion_filter=flt[1])))
    full = dict(use_legs=True, use_wings=True, use_mouth=True, use_antennae=True, joint_filter=0.01, adhesion_filter=0.02)
    out.append(('walker', dict(full, force_actuators=True)))
    for exact in (False, True):
        out.append(('walker', dict(full, dyntype_filterexact=exact)))
    # what flymodel.model_for asks for on behalf of the env factories' switches
    sw = dict(force_actuators=False, use_wings=None, use_legs=None, joint_filter=None)
    out.append(('walk', dict(sw, use_wings=True)))
    out.append(('walk', dict(sw, force_actuators=True, joint_filter=0.0)))
    out.append(('flight', dict(sw, use_legs=True, joint_filter=0.0002)))
    return out


def main():
    from flybody_b200.compiler import compile_model as cm
    src = sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(OUT), 'fruitfly_assets')
    mesh_cache = cm.load_mesh_cache(src)
    index = {}
    with tarfile.open(OUT, 'w:xz', preset=9) as tar:
        def add(name, data):
            ti = tarfile.TarInfo(name)
            ti.size = len(data)
            tar.addfile(ti, io.BytesIO(data))
        for i, (variant, kw) in enumerate(variants()):
            m = cm.compile_variant(variant, assets_dir=src, mesh_cache=mesh_cache, **kw)
            arrays = {k: v for k, v in m.items() if isinstance(v, np.ndarray) and not k.startswith('_')}
            meta = {k: v for k, v in m.items() if not isinstance(v, np.ndarray) and not k.startswith('_')}
            arrays['__meta__'] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
            buf = io.BytesIO()
            np.savez(buf, **arrays)
            name = f'{i:03d}_{variant}.npz'
            add(name, buf.getvalue())
            index[name] = dict(variant=variant, kwargs=kw)
        add('index.json', json.dumps(index, indent=1).encode())
    print(OUT, os.path.getsize(OUT), 'bytes,', len(index), 'models')


if __name__ == '__main__':
    main()
