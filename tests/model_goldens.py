"""The fly model the compiler is tested on, and what the compiler made of it.

golden/fruitfly_assets/fruitfly.xml is the upstream project's model file (see the README beside it).  golden/model_variants.tar.xz
holds the compiler's output for every variant the tests compile (written by tests/golden/make_variant_goldens.py): the regression
target of a fresh compile."""
import functools
import io
import json
import math
import os
import tarfile

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
ASSETS = os.path.join(GOLDEN, 'fruitfly_assets')
ARCHIVE = os.path.join(GOLDEN, 'model_variants.tar.xz')
RTOL = 1e-9


@functools.lru_cache(maxsize=1)
def _archive():
    with tarfile.open(ARCHIVE, 'r:xz') as tar:
        files = {ti.name: tar.extractfile(ti).read() for ti in tar.getmembers()}
    index = json.loads(files.pop('index.json'))
    return [(e['variant'], e['kwargs'], files[name]) for name, e in index.items()]


def read_saved(f):
    """(arrays, JSON metadata) of a model file in the layout of `compile_model.save_model` (a path or a file object)"""
    z = np.load(f)
    return {k: z[k] for k in z.files if k != '__meta__'}, json.loads(bytes(z['__meta__']).decode())


def stored(variant, **kwargs):
    """the stored output of `compile_variant(variant, **kwargs)`: (arrays, JSON metadata); KeyError if not stored"""
    for v, kw, data in _archive():
        if v == variant and kw == kwargs:
            return read_saved(io.BytesIO(data))
    raise KeyError(f'no stored compilation of {variant} {kwargs}: rerun tests/golden/make_variant_goldens.py')


def _same_meta(a, b):
    if isinstance(a, dict):
        return isinstance(b, dict) and a.keys() == b.keys() and all(_same_meta(a[k], b[k]) for k in a)
    if isinstance(a, list):
        return isinstance(b, list) and len(a) == len(b) and all(_same_meta(x, y) for x, y in zip(a, b))
    if isinstance(a, float) or isinstance(b, float):
        return math.isclose(a, b, rel_tol=RTOL, abs_tol=0.0)
    return a == b


def assert_matches_stored(arrays, meta, variant, **kwargs):
    """a compiled model (arrays + metadata) equals the stored compilation: integers exactly, floats to RTOL relative"""
    want_a, want_m = stored(variant, **kwargs)
    assert sorted(arrays) == sorted(want_a), (variant, kwargs, sorted(set(arrays) ^ set(want_a)))
    for k, want in want_a.items():
        got = np.asarray(arrays[k])
        assert got.shape == want.shape and got.dtype == want.dtype, (variant, kwargs, k, got.shape, want.shape, got.dtype, want.dtype)
        if want.dtype.kind == 'f':
            scale = float(np.abs(want).max()) if want.size else 0.0
            assert np.allclose(got, want, rtol=RTOL, atol=RTOL * scale), (variant, kwargs, k, float(np.abs(got - want).max()))
        else:
            assert np.array_equal(got, want), (variant, kwargs, k)
    assert _same_meta(json.loads(json.dumps(meta)), want_m), (variant, kwargs, 'metadata')


def compile_variant(variant, **kwargs):
    """`compile_model.compile_variant` on golden/fruitfly_assets, checked against the stored compilation"""
    from flybody_b200.compiler import compile_model as cm
    m = cm.compile_variant(variant, assets_dir=ASSETS, **kwargs)
    assert_matches_stored({k: v for k, v in m.items() if isinstance(v, np.ndarray) and not k.startswith('_')},
                          {k: v for k, v in m.items() if not isinstance(v, np.ndarray) and not k.startswith('_')}, variant, **kwargs)
    return m
