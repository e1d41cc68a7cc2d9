"""The CPU oracle with per-triangle materials (tests/oracle_tri_mats.c) — TEST INFRASTRUCTURE, the checker of
ipt_scene_set_triangle_materials.

`load()` compiles oracle/ipt_oracle.c, unchanged but for the hook of oracle_tri_mats.c, with the flags of oracle/Makefile
into a temporary directory (nothing is written into the tree) and returns an oracle_lib.Oracle over it that can also
attach an array of material indices to a scene description.
"""
from __future__ import annotations

import atexit
import contextlib
import ctypes as C
import glob
import os
import shutil
import subprocess
import tempfile
from pathlib import Path

import numpy as np

import oracle_lib

ROOT = Path(__file__).resolve().parent.parent


class TriMatsOracle(oracle_lib.Oracle):
    def set_triangle_materials(self, desc_ptr, materials):
        """ipt_oracle_set_triangle_materials: attach materials[k] to triangle k of the description (the oracle keeps a copy);
        None detaches. Every call on that description then reports materials[k] for a hit on triangle k."""
        m = None if materials is None else np.ascontiguousarray(materials, np.uint32)
        if m is not None:
            assert m.shape == (desc_ptr.contents.n_triangles,), m.shape
        rc = self.lib.ipt_oracle_set_triangle_materials(desc_ptr, None if m is None else m.ctypes.data_as(oracle_lib.u32p))
        assert rc == 0, {1: "material index out of range", 2: "table of attached arrays full"}.get(rc, rc)

    @contextlib.contextmanager
    def triangle_materials(self, desc_ptr, materials):
        """set_triangle_materials for the duration of a `with` block: a description's address may be reused once it is
        freed, so an attached array must not outlive it."""
        self.set_triangle_materials(desc_ptr, materials)
        try:
            yield
        finally:
            self.set_triangle_materials(desc_ptr, None)


_oracle = None


def load() -> TriMatsOracle:
    global _oracle
    if _oracle is None:
        tmp = tempfile.mkdtemp(prefix="ipt_oracle_tri_mats_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libipt_oracle_tri_mats.so")
        # oracle/Makefile's flags: the float arithmetic must be the oracle's own
        gomp = glob.glob("/usr/lib/gcc/x86_64-linux-gnu/*/libgomp.spec")
        cmd = [os.environ.get("CC", "gcc"), "-std=c11", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-fopenmp",
               *(["-B" + os.path.dirname(gomp[0]) + "/"] if gomp else []), "-Wall", f"-I{ROOT / 'include'}", f"-I{ROOT / 'oracle'}",
               "-o", so, str(ROOT / "tests" / "oracle_tri_mats.c"), "-lm"]
        subprocess.run(cmd, check=True, capture_output=True)
        _oracle = TriMatsOracle(C.CDLL(so))
    return _oracle
