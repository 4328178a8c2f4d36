"""The GENERATED device sources (serl_b200/csrc/gen: fast mode, merged variants, pooled constants, table blob) are
checked on the CPU: compiled with gcc behind trivial macro definitions and compared with the oracle's exact restatement on
the reference-recorded right-hand-side vectors and the gust / test binaries' recorded states (tests/golden).  Also: the
committed generated files are reproducible from the reference binaries' byte copies under oracle/_ref (oracle/build.py)."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KAT = np.load(os.path.join(ROOT, 'tests', 'golden', 'plant_rhs_kat.npz'))
REFBIN = np.load(os.path.join(ROOT, 'tests', 'golden', 'refbin_kat.npz'))
VARIANTS = ['h2000_v90', 'ice', 'cg', 'cg_for', 'h2000_v150', 'h10000_v90']
LIVE = [0, 1, 2, 3, 4, 5, 6, 7, 9, 12, 15, 16, 17, 18]

HARNESS = r'''
#include <math.h>
#include <stdbool.h>
typedef %(real)s real;
#define __restrict__ restrict
#define __device__
#define PLANT_FN static
#define PLANT_XARGS , const real* restrict plant_tab
#define PLANT_TAB(name) (plant_tab + PT_OFF_##name)
#define PLANT_CONSTS(n) static const real plant_k[n]
#define PLANT_K(i) plant_k[i]
#define PLANT_IC_TABLE static const double plant_ic_table[8][19]
#define PLANT_IC(v) static const double plant_ic_unused_##v[19]
#define PLANT_PV_TABLE static const real plant_pv[8][PLANT_NPV]
#define PLANT_PV(k) plant_pvrow[k]
#define PLANT_XI(i) (i)
#define PLANT_DIV(a, b) ((a) / (b))
#define PLANT_SQRT sqrt%(sfx)s
#define PLANT_FABS fabs%(sfx)s
#define PLANT_SIN sin%(sfx)s
#define PLANT_COS cos%(sfx)s
#define PLANT_SINCOS sincos%(sfx)s
#define PLANT_TAN tan%(sfx)s
#define PLANT_EXP exp%(sfx)s
#define PLANT_LOG10 log10%(sfx)s
#define PLANT_POW pow%(sfx)s
#define _GNU_SOURCE
#include "%(support)s"
#include "%(gen)s/plant_tables_blob.h"
#include "%(gen)s/plant_consts.h"
#include "%(gen)s/plant_ic.h"
#include "%(gen)s/plant_rhs_common.h"
#include "%(gen)s/plant_rhs_nav.h"
void dev_rhs(int variant, const double* Xd, const double* Ud, double* out) {
    real X[19], U[4], xdot[19], nav[19];          /* U[3]: angle-of-attack offset of the gust build (0 otherwise) */
    for (int i = 0; i < 19; ++i) { X[i] = (real)Xd[i]; xdot[i] = 0; }
    for (int i = 0; i < 4; ++i) U[i] = (real)Ud[i];
    plant_rhs_common(X, U, xdot, plant_tables_blob, plant_pv[variant]);      /* one function for every variant */
    plant_rhs_nav(X, U, nav, plant_tables_blob);
    xdot[8] = nav[8]; xdot[10] = nav[10]; xdot[11] = nav[11];
    for (int i = 0; i < 19; ++i) out[i] = (double)xdot[i];
}
void dev_ic(int variant, double* X) { for (int i = 0; i < 19; ++i) X[i] = plant_ic_table[variant][i]; }
'''


@pytest.fixture(scope='module', params=['gen', 'gen_exact', 'gen_f32'])
def devlib(request, tmp_path_factory):
    d = tmp_path_factory.mktemp('devplant_' + request.param)
    src = d / 'h.c'
    src.write_text(HARNESS % {'support': os.path.join(ROOT, 'serl_b200', 'csrc', 'plant_support.h'),
                              'gen': os.path.join(ROOT, 'serl_b200', 'csrc', request.param),
                              'real': 'float' if request.param == 'gen_f32' else 'double', 'sfx': 'f' if request.param == 'gen_f32' else ''})
    so = d / 'h.so'
    subprocess.check_call(['gcc', '-O1', '-D_GNU_SOURCE', '-ffp-contract=off', '-fPIC', '-shared', '-o', str(so), str(src), '-lm'])
    lib = ctypes.CDLL(str(so))
    return request.param, lib


@pytest.mark.parametrize('variant', VARIANTS)
def test_generated_device_rhs_matches_reference_binary_vectors(devlib, variant):
    which, lib = devlib
    D = ctypes.c_double
    v = VARIANTS.index(variant)
    ic = (D * 19)()
    lib.dev_ic(v, ic)
    assert np.array_equal(np.array(ic[:]), KAT[variant + '_ic'])
    worst = 0.0
    for x, u, f in zip(KAT[variant + '_X'], KAT[variant + '_U'], KAT[variant + '_F']):
        xd = (D * 19)()
        lib.dev_rhs(v, (D * 19)(*x), (D * 4)(*u, 0.0), xd)
        got = np.array(xd[:])
        idx = LIVE + [8, 10, 11]
        if which == 'gen_exact':
            assert np.array_equal(got[idx], f[idx])          # reference operation order: bit-exact
        err = np.abs(got[idx] - f[idx]) / np.maximum(np.abs(f[idx]), 1e-3 if which != 'gen_f32' else 1.0)
        worst = max(worst, err.max())
    # fast mode (reciprocal tables / constants, merged rows): 1e-11; single-precision right-hand side: float round-off
    assert worst < (5e-4 if which == 'gen_f32' else 1e-11), worst


@pytest.mark.parametrize('build,sign', [('gust', 1.0), ('test', -1.0)])
def test_gust_build_is_the_nominal_rhs_with_an_angle_of_attack_offset(devlib, build, sign):
    """envs/gust ("vertical gust of 15 ft/s at 20 s"): ode5 over the generated right-hand side with U[3] = atan(w / V) for the
    stages inside 20 s <= t <= 23 s (last stage of native call 1999, calls 2000..2299, first stage of call 2300) reproduces
    the gust BINARY bit for bit (reference-order build) through both edges of the pulse.  envs/test is the same pulse with the
    opposite sign (U[3] = -atan(w / V)).  The binary's states before and after those calls, stepped from initialize() with
    cmd = 0.02 sin(0.01 k + [0, 1, 2]), are recorded in tests/golden/refbin_kat.npz."""
    import math
    which, lib = devlib
    if which == 'gen_f32':
        pytest.skip('double-precision check')
    D = ctypes.c_double
    B = [[1 / 5, 0, 0, 0, 0, 0], [3 / 40, 9 / 40, 0, 0, 0, 0], [44 / 45, -56 / 15, 32 / 9, 0, 0, 0],
         [19372 / 6561, -25360 / 2187, 64448 / 6561, -212 / 729, 0, 0], [9017 / 3168, -355 / 33, 46732 / 5247, 49 / 176, -5103 / 18656, 0],
         [35 / 384, 0, 500 / 1113, 125 / 192, -2187 / 6784, 11 / 84]]
    idx = LIVE + [8, 10, 11]
    w = float.fromhex('0x1.249ba5e353f7dp+2')          # include/serl_b200.h SERL_GUST_W
    h = 0.01

    def on(call, s):
        return (call == 1999 and s == 5) or (2000 <= call < 2300) or (call == 2300 and s == 0)

    def step(X, u, call):
        f, x = [], X.copy()
        for s in range(6):
            out = (D * 19)()
            lib.dev_rhs(0, (D * 19)(*x), (D * 4)(u[0], u[1], u[2], sign * (math.atan(w / x[3]) * 1.0) if on(call, s) else 0.0), out)
            f.append(np.array(out[:]))
            x = X.copy()
            for i in idx:
                acc = f[0][i] * (h * B[s][0])
                for j in range(1, s + 1):
                    acc += f[j][i] * (h * B[s][j])
                x[i] = X[i] + acc
        return x
    worst, active = 0.0, 0
    window = [k for k in range(2306) if 1996 <= k <= 2003 or 2296 <= k <= 2303 or k == 2150]
    assert REFBIN[build + '_k'].tolist() == window
    for k, X, Xb in zip(window, REFBIN[build + '_X0'], REFBIN[build + '_X1']):
        c = 0.02 * np.sin(0.01 * k + np.arange(3))
        Xn = step(X, c, k)
        err = np.abs(Xn[idx] - Xb[idx]).max()
        worst = max(worst, err / np.abs(Xb[idx]).max())
        if which == 'gen_exact':
            assert err == 0.0, (k, err)
        nominal = step(X, c, -1)
        active += int(np.abs(nominal[idx] - Xb[idx]).max() > 0)
    assert worst < 1e-12 and active >= 10        # fast build: <= 1 ulp per operation; the gust really is on in the window


def _have_ref_binaries():
    from oracle import build as obuild
    return all(os.path.exists(os.path.join(obuild.HERE, '_ref', 'citation_%s.so' % v)) for v in obuild.VARIANTS + obuild.REF_ONLY)


@pytest.mark.skipif(not _have_ref_binaries(), reason='needs the reference plant binaries under oracle/_ref (oracle/build.py)')
def test_committed_generated_sources_are_reproducible(tmp_path):
    """tools/lift regenerates byte-identical device sources from the reference binaries (oracle/_ref); the lifter's working
    copies of the binaries go to tmp_path."""
    code = ("import sys; sys.path.insert(0, %r); import gen_plant, gen_all as G, symtrace as S; "
            "gen_plant.REF = %r; init = S.Image.__init__; "
            "S.Image.__init__ = lambda self, so, workdir: init(self, so, %r); "
            "G.emit_set(%r, live=True)" %
            (os.path.join(ROOT, 'tools', 'lift'), os.path.join(ROOT, 'oracle', '_ref', 'citation_%s.so'), str(tmp_path / 'lift'),
             str(tmp_path / 'gen')))
    subprocess.check_call([sys.executable, '-c', code], stdout=subprocess.DEVNULL)
    for f in sorted(os.listdir(tmp_path / 'gen')):
        a = open(tmp_path / 'gen' / f).read()
        b = open(os.path.join(ROOT, 'serl_b200', 'csrc', 'gen', f)).read()
        assert a == b, f
