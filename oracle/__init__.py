"""CPU oracle for the scintools arc-measurement hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``scintools_b200/`` may import this
package.  The only legitimate users are ``tests/``, ``__graft_entry__.smoke()``
and the ``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` -- and
there only as the checker / CPU reference, never as the thing shipped.

Parity status
-------------
The reference repository (danielreardon/scintools @ 9b6d577) ships *no* test
suite and *no* golden vectors, so there is nothing upstream to pin against
(SURVEY.md section 8c).  The oracle is instead pinned against **outputs of the
reference itself, run in the build container**:

* ``oracle/ref_loader.py`` imports the unmodified reference from
  ``/root/reference`` with stub modules for the missing optional dependencies
  (matplotlib, astropy, lmfit, ...).  ``Dynspec.calc_sspec``, ``Dynspec.calc_acf``
  and ``scint_sim.Simulation`` then run unmodified.
* ``oracle/make_golden.py`` (committed) drives the reference through that loader
  on seeded synthetic inputs and writes the small fixtures in ``tests/golden/``.
  The numpy restatements in this package are checked against those fixtures in
  ``tests/test_oracle_golden.py``.
* ``ththmod`` needs real ``astropy.units`` arithmetic, which cannot be stubbed
  (astropy is not installable offline).  ``thth_oracle.py`` is a unit-free,
  line-by-line restatement; it is pinned by (i) executing the reference's own
  ``ththmod`` source through a *minimal arithmetic units shim*
  (``oracle/units_shim.py``, scale factors exactly 1.0 for us / mHz / s^3) in
  ``make_golden.py`` and (ii) the documented known answer eta ~= 44 s^3 on
  ``Sample_Data.npz`` (docs/source/tutorials/thth_intro.rst:101-104).
  Residual risk (stated in DESIGN.md): real astropy could apply a unit scale
  that differs from 1.0 in the last ulp; this cannot be checked offline.

Units convention of every unit-free function here: tau in us, fd / theta /
edges in mHz, eta in s^3, time in s, freq in MHz.  eta*theta^2 is numerically
already in us (s^3 * mHz^2 == 1e-6 s).
"""
import hashlib

import numpy as np


def complex_digest(a):
    """SHA-256 of ``a`` as C-ordered complex128 bytes.  Fixtures store this in place
    of reference arrays too large to commit; equal digests mean bit-identical arrays."""
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.complex128).tobytes()).hexdigest()


def retrieval_maps(g):
    """thth_red, rv_h and rv_n of the fixture tests/golden/retrieval_64x128.npz (``g``),
    rebuilt by the oracle from the fixture's inputs and checked bit for bit against
    the digests the fixture keeps of the reference's arrays."""
    from oracle import thth_oracle as TO
    eta = float(g["eta"])
    CS = TO.conjugate_spectrum(g["d0"], int(g["npad"]), None)
    out = {"thth_red": TO.thth_redmap(CS, g["tau"], g["fd"], eta, g["edges"])[0]}
    n = out["thth_red"].shape[0]
    rng = np.random.default_rng(int(g["tt_seed"]))
    tt = rng.normal(size=(n, n)) + 1j * rng.normal(size=(n, n))
    for herm, key in ((True, "rv_h"), (False, "rv_n")):
        out[key] = TO.rev_map(tt, g["tau"], g["fd"], eta, g["edges_red"], hermetian=herm)
    for key, a in out.items():
        assert a.shape == tuple(g[key + "_shape"]), key
        assert complex_digest(a) == str(g[key + "_sha256"]), key
    return out
