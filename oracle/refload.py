"""Loader for the UNMODIFIED reference (nintendops/DynamicFusion_Body) -- test infrastructure only.

The reference is pure Python and is not part of this repository: put a checkout of it at oracle/_ref/ (ignored by git)
or name one with DFB_REFERENCE_ROOT.  This module is only used (a) by tests that are skipped when the
reference is absent and (b) by tests/golden/make_golden*.py, which execute the reference to
produce the committed golden fixtures.  Nothing in the product package imports it.

`import core` pulls TensorFlow-1, PyOpenGL, scikit-image and pyopencl (core/__init__.py:1-5,
core/fusion.py:41, core/fusion_dm.py:38), none of which are installed, so empty stand-in modules
are put in sys.modules first (SURVEY.md section 8c recipe).  No reference source is modified or copied.
"""
import contextlib
import io
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("DFB_REFERENCE_ROOT", os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref"))


def available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "core", "fusion.py"))


def _stub(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    m.__all__ = []
    sys.modules.setdefault(name, m)
    return sys.modules[name]


_loaded = None


def load():
    """Return (util_module, Fusion, FusionDM) from the unmodified reference."""
    global _loaded
    if _loaded is not None:
        return _loaded
    if not available():
        raise RuntimeError("reference not present at %s" % REFERENCE_ROOT)
    sk = _stub("skimage")
    sk.measure = _stub("skimage.measure")
    tf = _stub("tensorflow")
    tf.nn = types.SimpleNamespace(elu=None)
    tf.contrib = _stub("tensorflow.contrib")
    tf.contrib.slim = _stub("tensorflow.contrib.slim")
    gl = _stub("OpenGL")
    for sub in ("GL", "GLU", "GLUT"):
        setattr(gl, sub, _stub("OpenGL." + sub))
    _stub("pyopencl")
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    with contextlib.redirect_stdout(io.StringIO()):
        import core.util as util
        from core.fusion import Fusion
        from core.fusion_dm import FusionDM
    _loaded = (util, Fusion, FusionDM)
    return _loaded


def make_fusion(nodes, tsdf, tsdfw, tdist, knn, lw, vertices=None, normals=None,
                neighbor_look_up=None, correspondences=None):
    """Build a reference `Fusion` without its broken __init__ (core/fusion.py:51 NameError).

    nodes: list of (vertex_idx, pos(3,) f32, dq(8,), w) tuples exactly as core/fusion.py:113-116."""
    from scipy.spatial import KDTree
    import numpy as np
    _, Fusion, _ = load()
    f = object.__new__(Fusion)
    f._itercounter = 0
    f._curr_tsdf = None
    f._tdist = abs(tdist)
    f._lw = lw
    f._knn = knn
    f._nodes = list(nodes)
    f._kdtree = KDTree(np.array([n[1] for n in nodes]))
    f._verbose = False
    f._write_warpfield = False
    f._sess = None
    f._tsdf = tsdf
    f._tsdfw = tsdfw
    f._vertices = vertices
    f._normals = normals
    f._neighbor_look_up = neighbor_look_up if neighbor_look_up is not None else []
    f._correspondences = correspondences if correspondences is not None else []
    return f


@contextlib.contextmanager
def quiet():
    """The reference prints inside its hot loops (core/fusion.py:192-195, fusion_dm.py:182)."""
    with contextlib.redirect_stdout(io.StringIO()):
        yield
