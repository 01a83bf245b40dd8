"""ORACLE — test infrastructure only (never imported by the product path).

CPU restatement of READ's per-frame render path, used as the parity checker by
``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` / ``--impl
reference`` legs of ``bench.py``.  Nothing under ``read_b200/`` may import this
package.

Pieces (each cites the reference file:line it follows):
  * ``zbuffer.c``   — sequential z-buffer == point_render.cu:107-200
  * ``render_ref``  — MyRender.render == src/READ/gl/myrender.py:23-43
  * ``unet_ref``    — PointTexture / NetAndTexture / UNet in plain torch fp32
                      == READ/models/{texture,compose,unet}.py

Parity pinning: the reference has no tests or golden vectors for this path
(SURVEY.md §4: "parity unpinned" by the reference itself).  We pin the oracle
with (1) hand-derived known-answer tests, (2) golden fixtures computed by the
reference's own Python modules (tests/golden/make_golden.py and
make_reference_modules.py, fixtures committed), and (3) the index/depth maps the
reference ``pcpr`` extension, compiled from its own sources into ``oracle/_ref/``,
rendered on a B200 (tests/golden/make_reference_pcpr.py, fixture committed).
"""
import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "liboracle_zbuffer.so")
_lib = None


def build(force=False):
    """gcc the C restatement (seconds).  -ffp-contract=off: only explicit fmaf() fuses.  Returns the library's path: in the
    package, or in a temporary directory when the package directory is read-only and holds no current build."""
    global _SO
    src = os.path.join(_HERE, "zbuffer.c")
    if (not force) and os.path.exists(_SO) and os.path.getmtime(_SO) >= os.path.getmtime(src):
        return _SO
    out = _SO
    if not os.access(_HERE, os.W_OK):
        tmp = tempfile.mkdtemp(prefix="oracle_zbuffer_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, os.path.basename(_SO))
    cmd = ["gcc", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-mfma",
           "-o", out, src, "-lm"]
    subprocess.check_call(cmd)
    _SO = out
    return _SO


def _load():
    global _lib
    if _lib is None:
        lib = ctypes.CDLL(build())
        f32p = ctypes.POINTER(ctypes.c_float)
        lib.oracle_pcpr_forward.argtypes = [f32p, ctypes.c_int64, f32p, ctypes.c_int, ctypes.c_int,
                                            ctypes.c_int, f32p, f32p]
        lib.oracle_pcpr_forward.restype = None
        lib.oracle_count_degenerate.argtypes = [f32p, ctypes.c_int64, f32p]
        lib.oracle_count_degenerate.restype = ctypes.c_int64
        _lib = lib
    return _lib


def _fp(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))


def pcpr_forward(xyz, total_m, w, h):
    """Oracle of ``pcpr.forward`` (pcpr_cuda.cpp:23-37): xyz [N,3] f32, total_m [B,4,4] f32
    -> (index [B,h,w] f32, depth [B,h,w] f32), numpy."""
    xyz = np.ascontiguousarray(xyz, dtype=np.float32)
    total_m = np.ascontiguousarray(total_m, dtype=np.float32)
    assert xyz.ndim == 2 and xyz.shape[1] == 3
    assert total_m.ndim == 3 and total_m.shape[1:] == (4, 4), "batch_size check"
    B = total_m.shape[0]
    index = np.empty((B, h, w), np.float32)
    depth = np.empty((B, h, w), np.float32)
    _load().oracle_pcpr_forward(_fp(xyz), xyz.shape[0], _fp(total_m), B, int(w), int(h),
                                _fp(index), _fp(depth))
    return index, depth


def count_degenerate(xyz, M):
    xyz = np.ascontiguousarray(xyz, dtype=np.float32)
    M = np.ascontiguousarray(M, dtype=np.float32).reshape(16)
    return int(_load().oracle_count_degenerate(_fp(xyz), xyz.shape[0], _fp(M)))


def level_sizes(W, H, L):
    """src/READ/gl/myrender.py:33-34: w=int(W*0.5**i), h=int(H*0.5**i)."""
    return [(int(W * (0.5 ** i)), int(H * (0.5 ** i))) for i in range(L)]


def render_pyramid(xyz, proj_matrix, view_matrix, W, H, L, threads=1):
    """Oracle of MyRender.render (src/READ/gl/myrender.py:23-43) for one dataset id.

    proj_matrix, view_matrix: [B,4,4] float32.  total_m = proj @ inv(view) with the SAME
    numpy call the reference makes (myrender.py:28-30).  Returns (total_m, [index_l], [depth_l])
    with index_l/depth_l [B,1,h_l,w_l] float32.
    """
    proj = np.asarray(proj_matrix, dtype=np.float32)
    view = np.asarray(view_matrix, dtype=np.float32)
    total_m = (proj @ np.linalg.inv(view)).astype(np.float32)
    sizes = level_sizes(W, H, L)
    if threads > 1:
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(max_workers=min(threads, L)) as ex:
            res = list(ex.map(lambda s: pcpr_forward(xyz, total_m, s[0], s[1]), sizes))
    else:
        res = [pcpr_forward(xyz, total_m, w, h) for (w, h) in sizes]
    idx = [r[0][:, None] for r in res]
    dep = [r[1][:, None] for r in res]
    return total_m, idx, dep
