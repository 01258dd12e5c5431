"""CPU tier: pins the plain-C restatement (oracle/mc_oracle.c) against the golden vectors of the UNMODIFIED reference
(tests/golden/cases.npz) and, when oracle/_ref is present, against the reference executed live; also pins the
product's powf restatement (csrc/mcb_pow.h, host build) against libm's powf."""
import os

import numpy as np
import pytest

from .helpers import load_meta, same_bits
from . import mc_numpy

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def OB():
    from oracle import oraclebind
    if not oraclebind.available():
        pytest.skip("oracle/libmcoracle.so not built (run __graft_entry__.build())")
    return oraclebind


def _mk(OB, case, pow_mode=0):
    return OB.Oracle(case["eq"], case["step"], tuple(case["scale"]), case["iso"], pow_mode=pow_mode,
                     cons=[tuple(c) for c in case["cons"]])


def test_restatement_matches_reference_goldens(OB, golden):
    meta = load_meta(golden)
    for name, case in meta.items():
        for pow_mode in (0, 1):   # libm powf, and the product's restatement of it: must be indistinguishable
            o = _mk(OB, case, pow_mode)
            M, c = o.coords()
            assert M == case["M"] and same_bits(c, golden[name + "/coords"]), name
            sw = o.sweep(nthreads=4)
            assert np.array_equal(sw["code"], golden[name + "/code"]), name
            assert np.array_equal(sw["table_idx"], golden[name + "/table_idx"]), name
            assert np.array_equal(sw["ntri"], golden[name + "/ntri"]), name
            assert (sw["T"], sw["active"], sw["ambiguous"], sw["redirected"]) == \
                (case["T"], case["active"], case["ambiguous"], case["redirected"]), name
            assert same_bits(sw["soup"], golden[name + "/soup"]), name
            v, t = o.recalculate(nthreads=3)
            assert same_bits(v, golden[name + "/vertex_list"]) and np.array_equal(t, golden[name + "/tri_list"]), name + " weld"
            assert same_bits(o.normals(), golden[name + "/normals"]), name + " normal.h"


def test_restatement_repeating_surface_mode_matches_reference_goldens(OB):
    """marching.cpp:481-494 in the restatement: per-cube level for code and ambiguity, Marching::interp's own constant for
    the points — against the unmodified reference's runs (tests/golden/repeat_cases.npz)."""
    import json
    from .helpers import load_repeat_golden
    rep = load_repeat_golden(os.path.join(ROOT, "tests", "golden", "repeat_cases.npz"))
    for name, case in json.loads(bytes(rep["meta_json"]).decode()).items():
        o = OB.Oracle(case["eq"], case["step"], tuple(case["scale"]), case["iso"], cons=[tuple(c) for c in case["cons"]], repeat=case["dist"])
        sw = o.sweep(nthreads=4)
        act = (rep[name + "/code"] != 0) & (rep[name + "/code"] != 255)
        assert np.array_equal(sw["code"][act], rep[name + "/code"][act]) and np.array_equal((sw["code"] != 0) & (sw["code"] != 255), act), name
        assert np.array_equal(sw["table_idx"][act], rep[name + "/table_idx"][act]), name
        assert np.array_equal(sw["ntri"], rep[name + "/ntri"]), name
        assert (sw["T"], sw["active"], sw["ambiguous"], sw["redirected"]) == (case["T"], case["active"], case["ambiguous"], case["redirected"]), name
        assert same_bits(sw["soup"], rep[name + "/soup"]), name
        v, t = o.recalculate(nthreads=2)   # the restatement carries the reference's global std::set, so the weld is the reference's too
        assert same_bits(v, rep[name + "/vertex_list"]) and np.array_equal(t, rep[name + "/tri_list"]), name + " weld"
        assert same_bits(o.normals(), rep[name + "/normals"]), name + " normal.h"


def test_restatement_gradient_normals_match_numpy(OB, golden):
    """Two independent CPU statements of the product's normal definition (C in mc_oracle.c, numpy in mc_numpy.py)."""
    from .test_host_logic import _packed_rows
    rows = [[int(e) for e in r if e >= 0] for r in _packed_rows()]
    meta = load_meta(golden)
    for name in ("sphere_17", "eq8_ctor", "gyr34_9", "saddle_17", "nonuniform_scale"):
        case = meta[name]
        o = _mk(OB, case)
        sw = o.sweep(nthreads=2, grad_normals=True)
        M = case["M"]
        act = np.flatnonzero((sw["code"] != 0) & (sw["code"] != 255))
        cubes = [(int(a % M), int((a // M) % M), int(a // (M * M)), int(sw["code"][a]), int(sw["table_idx"][a])) for a in act]
        cs = mc_numpy.apron_coords(golden[name + "/coords"], case["step"])
        nref = mc_numpy.soup_gradient_normals(golden[name + "/field_ext"], cs, case["iso"], cubes, rows)
        assert same_bits(sw["grad_normals"], nref), name


def test_restatement_against_live_reference(OB, unmodified_reference):
    refbind = unmodified_reference
    rng = np.random.default_rng(3)
    pts = (rng.random((3000, 3), dtype=np.float32) * 4 - 2).astype(np.float32)
    eqs = list(refbind.EXAMPLE_EQUATIONS.values()) + [refbind.GYR78, "x-y+z", "x/y*z", "-x^2", "x*-y+z", "x^y^z",
                                                       "xy/z^-.22", "x^0.5+y"]
    for eq in eqs:
        for pm in (0, 1):
            o = OB.Oracle(eq, pow_mode=pm)
            assert same_bits(o.eval_points(pts), refbind.Ref(eq).eval_points(pts)), eq
    # a mid-size full run, welded, with a non-dyadic step, anisotropic scale and a non-zero iso value
    r = refbind.Ref(refbind.TORUS, 2.0 / 40, (1.05, 0.95, 1.0), 0.01)
    v, t = r.recalculate()
    o = OB.Oracle(refbind.TORUS, 2.0 / 40, (1.05, 0.95, 1.0), 0.01)
    v2, t2 = o.recalculate()
    assert same_bits(v, v2) and np.array_equal(t, t2)
    assert same_bits(r.normals(), o.normals())


def test_restatement_tokenizer_against_reference_verdicts(OB):
    """mco_tokenize_ok, which stands in for Evaluator::tokenize where oracle/_ref is not built, against verdicts of the
    reference itself: Evaluator::test()'s nine known answers and every equation (and constraint) its golden runs took."""
    import json
    from .helpers import load_repeat_golden
    from .test_host_logic import EVALUATOR_TEST_CASES
    for eq, ok in EVALUATOR_TEST_CASES:
        assert bool(OB.lib().mco_tokenize_ok(eq.encode())) == ok, eq
    metas = [load_meta(np.load(os.path.join(ROOT, "tests", "golden", f + ".npz"), allow_pickle=False)) for f in ("cases", "seed_cases")]
    metas.append(json.loads(bytes(load_repeat_golden(os.path.join(ROOT, "tests", "golden", "repeat_cases.npz"))["meta_json"]).decode()))
    eqs = {e for m in metas for case in m.values() for e in [case["eq"]] + [c[0] for c in case.get("cons", [])]}
    assert len(eqs) >= 15
    for eq in eqs:
        assert OB.lib().mco_tokenize_ok(eq.encode()), eq


def test_parse_accept_reject_matches_product(OB, mcb):
    for eq in ["x+y", "(x(y)", "x+", "-", "2x(y)3", "x^-y", "x--y", "--x", "", ".", "3.x", "((x))", "x)"]:
        assert bool(OB.lib().mco_parse_ok(eq.encode())) == mcb.parse_ok(eq), eq


POW_CHECK_SRC = r'''
#include <stdio.h>
#include <stdlib.h>
#include <math.h>
#include <pthread.h>
#include "mcb_pow.h"
static unsigned long long rng(unsigned long long* s){ *s ^= *s<<13; *s ^= *s>>7; *s ^= *s<<17; return *s; }
typedef struct { unsigned long long seed; long n, bad; int mode; } job;
static int same(float a, float b){ if (a!=a && b!=b) return 1; return mcb_f2u(a)==mcb_f2u(b); }
static void* run(void* p){ job* j=p; unsigned long long s=j->seed; long bad=0;
  static const float ys[] = {2,3,4,0.5f,-1,-2,1.5f,0.22f,-0.22f,7,8,0.333f,10,1,0};
  for(long i=0;i<j->n;i++){ float x,y; unsigned long long r=rng(&s);
    if (j->mode==0){ x = mcb_u2f((unsigned)r); y = mcb_u2f((unsigned)(r>>32)); }
    else if (j->mode==1){ x = (float)((double)(r&0xffffff)/0x1000000*2.75-1.375); y = ys[(r>>24)%15]; }
    else { x = (float)((double)(r&0xffffff)/0x1000000*4.0-2.0); y = (float)((double)((r>>24)&0xffffff)/0x1000000*16.0-8.0); }
    if(!same(powf(x,y), mcb_powf(x,y))) bad++; }
  j->bad=bad; return 0; }
int main(int argc,char**argv){ long n=atol(argv[1]); int T=atoi(argv[2]); pthread_t th[64]; job jb[64]; long bad=0;
  for(int m=0;m<3;m++){ for(int t=0;t<T;t++){ jb[t].seed=0x9E3779B97F4A7C15ull*(t+1+m*100); jb[t].n=n; jb[t].mode=m; pthread_create(&th[t],0,run,&jb[t]); }
    for(int t=0;t<T;t++){ pthread_join(th[t],0); bad+=jb[t].bad; } }
  printf("%ld\n", bad); return 0; }
'''


def test_powf_restatement_equals_libm():
    """csrc/mcb_pow.h (host build) vs glibc powf: >1e8 inputs incl. raw random bit patterns; zero mismatches."""
    import subprocess
    import tempfile
    inc = os.path.join(ROOT, "marching-cube-for-implicit-surfaces_b200", "csrc")
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "p.c"), "w").write(POW_CHECK_SRC)
        subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-I", inc, os.path.join(d, "p.c"), "-o",
                               os.path.join(d, "p"), "-lm", "-lpthread"])
        T = min(8, os.cpu_count() or 1)
        n = 36_000_000 // T
        out = subprocess.check_output([os.path.join(d, "p"), str(n), str(T)], text=True)
    assert int(out.strip()) == 0
