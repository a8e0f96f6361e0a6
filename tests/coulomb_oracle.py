"""TEST INFRASTRUCTURE ONLY: the CPU oracle with Coulomb-pyramid friction (tests/coulomb_oracle.cc).

`CoulombWorld(world, mu)` wraps an `oracle.pyoracle.World` on the PGS solver: `step` runs the
oracle's step with Coulomb friction of coefficient `mu` (None: the oracle's own BOX step), and every
other attribute is the wrapped world's.  The library is compiled on first use with the flags of
oracle/Makefile into the temporary directory, keyed by the hash of its sources, so the repository
tree is never written."""
import ctypes as C
import hashlib
import math
import os
import subprocess
import tempfile

import numpy as np

from oracle import pyoracle as O

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "coulomb_oracle.cc")
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")
_FLAGS = ["-O2", "-DNDEBUG", "-march=native", "-ffp-contract=off", "-std=c++17", "-fPIC", "-shared"]   # oracle/Makefile
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        O.lib()   # the World handles come from liboracle.so
        h = hashlib.sha256(" ".join(_FLAGS).encode())
        for f in [_SRC] + sorted(os.path.join(_ORACLE, x) for x in os.listdir(_ORACLE) if x.endswith(".h")):
            with open(f, "rb") as fh:
                h.update(fh.read())
        so = os.path.join(tempfile.gettempdir(), f"eggshell_coulomb_oracle_{os.getuid()}_{h.hexdigest()[:16]}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}.tmp"
            subprocess.check_call([os.environ.get("CXX", "g++")] + _FLAGS + ["-o", tmp, _SRC])
            os.replace(tmp, so)
        _LIB = C.CDLL(so)
    return _LIB


class CoulombWorld:
    """An oracle World stepped with Coulomb friction `mu` (finite, >= 0; None: BOX).  The solver must be
    PGS when mu is set (`solver`, as given to set_params): the other solvers have no Coulomb path."""

    def __init__(self, world, mu, solver):
        if mu is not None:
            m = float(mu)
            if not (math.isfinite(m) and m >= 0) or solver != O.SOLVER_PGS:
                raise ValueError(f"Coulomb friction {mu!r}: mu must be finite and >= 0, and the solver PGS")
        self.world, self.mu = world, mu

    def __getattr__(self, name):
        return getattr(self.world, name)

    def step(self, dt):
        if self.mu is None:
            return self.world.step(dt)
        st = lib().coulomb_world_step(self.world.h, C.c_double(dt), C.c_double(float(self.mu)))
        assert st >= 0
        return st

    def friction_bound(self):
        """Per row of the last step: the bound b each tangent row was last projected with (inf: none)."""
        n = lib().coulomb_world_bound(self.world.h, None)
        out = np.zeros(n)
        lib().coulomb_world_bound(self.world.h, out.ctypes.data_as(C.POINTER(C.c_double)))
        return out

    def __del__(self):
        try:
            lib().coulomb_world_forget(self.world.h)
        except Exception:
            pass
