"""TEST INFRASTRUCTURE ONLY — the part of oracle/refbind's interface the tests use, served by the plain-C restatement
(oracle/libmcoracle.so, oracle/mc_oracle.c) instead of the compiled reference.

The unmodified reference's sources are not part of this repository, so oracle/_ref/libmcref.so exists only where
they were available at build time.  Everywhere else the tests that compare with the reference live compare with
this stand-in (the pytest header says which one a run used).  What the stand-in is worth, and where it is not
independent of the product:
  - tokenizer and evaluator: its own, walking the token list with two stacks like the reference; it shares no lowering
    with the product.  tests/test_oracle.py pins the values to the reference's golden vectors and the tokenizer's
    verdicts to the reference's known answers (Evaluator::test() and every equation of the golden runs).
  - lookup tables: the product's own (csrc/mcb_tables.h), so per-cube and soup comparisons do not test the table rows.
    Those are pinned to the reference separately: tests/test_host_logic.py checks every row its golden runs used
    against the triangles it emitted, and the ambiguity rule against its ambiguous and redirected cubes.
The restatement checked against the reference itself stays with the `unmodified_reference` fixture.
"""
import os

from oracle import oraclebind
from oracle.refbind import EXAMPLE_EQUATIONS, GYR34, GYR78, SPHERE, TORUS  # noqa: F401  (the inputs, same names)


def available():
    return oraclebind.available()


def parse_ok(eq):
    """Evaluator::tokenize's verdict on `eq` (the reference's tokenizer, without the restatement's underflow check)."""
    return bool(oraclebind.lib().mco_tokenize_ok(eq.encode()))


class Ref:
    """One Evaluator + Marching pair of the restatement, with refbind.Ref's methods.  The step is not range-checked:
    callers pass steps the reference accepts, or force them as refbind's force_step does."""

    def __init__(self, eq=None, step=None, scale=(1.0, 1.0, 1.0), iso=0.0, force_step=False):
        self.o = oraclebind.Oracle(eq, step, scale, iso)

    def coords(self):
        return self.o.coords()

    def eval_points(self, xyz, scaled=False):
        return self.o.eval_points(xyz, scaled=scaled)

    def sweep(self, k0=0, k1=None, soup=True):
        return self.o.sweep(k0, k1, soup=soup)

    def recalculate(self):
        return self.o.recalculate()

    def normals(self):
        return self.o.normals()


def sweep_rows_mt(eq, step, row0, row1, nthreads=None, scale=(1.0, 1.0, 1.0), iso=0.0, force_step=True):
    """refbind.sweep_rows_mt for whole cube layers: rows [row0, row1) with row = k*M + j."""
    r = Ref(eq, step, scale, iso)
    M, _ = r.coords()
    assert row0 % M == 0 and row1 % M == 0, "the restatement sweeps whole cube layers"
    return r.o.sweep(row0 // M, row1 // M, nthreads=nthreads or os.cpu_count())
