"""Loads the reference's own ops.py / model.py (UNMODIFIED, from a checkout of tachitachi/SR-WaveNet named by the
environment variable SRWN_REFERENCE_DIR) on top of the NumPy TensorFlow stand-in in tests/tf_shim.  Test
infrastructure; used by tests/test_reference_shim.py and tests/golden/make_reference_*golden.py.  The reference is
not part of this repository, so callers skip when ``available()`` is False; the committed fixtures
tests/golden/reference_*.npz hold what it computed."""
import contextlib
import importlib
import io
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REFERENCE = os.environ.get('SRWN_REFERENCE_DIR', '')
SHIM = os.path.join(HERE, 'tf_shim')


def available():
    return bool(REFERENCE) and os.path.exists(os.path.join(REFERENCE, 'ops.py')) and \
        os.path.exists(os.path.join(REFERENCE, 'model.py'))


_loaded = {}


def load():
    """-> (tf, ops, model): the stand-in and the reference modules imported through it.  The reference modules
    are registered under private names so the repo's own ``teacher`` / ``student`` / ``ops`` are never shadowed."""
    if _loaded:
        return _loaded['tf'], _loaded['ops'], _loaded['model']
    saved_path, saved_mods = list(sys.path), {k: sys.modules.get(k) for k in ('tensorflow', 'ops', 'model')}
    sys.path[:0] = [SHIM, REFERENCE]
    for k in ('tensorflow', 'ops', 'model'):
        sys.modules.pop(k, None)
    try:
        tf = importlib.import_module('tensorflow')
        assert tf.__file__.startswith(SHIM), 'a real TensorFlow is installed; the stand-in is not needed'
        ops = importlib.import_module('ops')
        model = importlib.import_module('model')
        assert ops.__file__.startswith(REFERENCE) and model.__file__.startswith(REFERENCE)
    finally:
        sys.path[:] = saved_path
        for k, v in saved_mods.items():
            if v is not None:
                sys.modules[k] = v
            else:
                sys.modules.pop(k, None)
    _loaded.update(tf=tf, ops=ops, model=model)
    return tf, ops, model


@contextlib.contextmanager
def quiet():
    """The reference prints from inside createNetwork (model.py:523-537)."""
    with contextlib.redirect_stdout(io.StringIO()):
        yield


def set_variables(graph, weights, strict_prefix=None):
    """Assigns name-keyed arrays to the graph's variables.  Every variable under ``strict_prefix`` must be given
    (that is the naming contract being tested) and every given name must exist."""
    import numpy as np
    missing = [n for n in graph.variables if strict_prefix and n.startswith(strict_prefix) and n not in weights]
    unknown = [n for n in weights if n not in graph.variables]
    assert not missing, 'reference variables without a value: %s' % missing[:5]
    assert not unknown, 'names the reference graph does not create: %s' % unknown[:5]
    for n, v in weights.items():
        var = graph.variables[n]
        assert tuple(var._shape) == tuple(v.shape), (n, var._shape, v.shape)
        var.value = np.asarray(v, dtype=np.float64)


class inject_uniforms(object):
    """Makes tf.random_uniform return the given arrays in call order (ops.py:187 then ops.py:196)."""

    def __init__(self, tf, arrays):
        self.tf, self.arrays, self.i = tf, list(arrays), 0

    def __enter__(self):
        self.saved = self.tf._random_hook

        def hook(shape, minval, maxval):
            a = self.arrays[self.i % len(self.arrays)]
            self.i += 1
            assert tuple(a.shape) == tuple(shape), (a.shape, shape)
            return a
        self.tf._random_hook = hook
        return self

    def __exit__(self, *a):
        self.tf._random_hook = self.saved
