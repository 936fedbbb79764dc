"""TEST INFRASTRUCTURE ONLY -- harness that makes the REAL, UNMODIFIED reference run.

Nothing under ``pyrad_b200/`` may import this module.  It only works inside the
build container, where the upstream sources are mounted at ``/root/reference``;
on the GPU box that path does not exist and ``available()`` returns False.  It
is used by ``tests/golden/make_golden.py`` (to generate the committed golden
vectors) and by the CPU-side tests that pin ``oracle.physics`` against the real
reference code.

Why a harness is needed (reference file:line):
  * ``pyradUtilities.py:13``  imports ``bs4``                      -> stub module
  * ``pyradClasses.py:10``    imports ``matplotlib.pyplot``        -> stub package
  * ``pyradClasses.py:12``    imports ``pyradInteractive`` whose import never
    returns (``pyradInteractive.py:761-762``)                      -> stub module
  * ``pyradUtilities.py:16-27`` derives every path from ``os.getcwd()`` and
    truncates ``./logger.txt``                                     -> chdir to a scratch dir
  * ``pyradUtilities.py:64-88,1005`` ``setupDir()`` runs at import and would
    download ``molparam.txt`` unless every ``data/<id>/params.pyr`` exists
                                                                    -> pre-seeded
  * ``pyradClasses.py:704``   passes a float ``num`` to ``np.linspace``
    (TypeError on numpy >= 1.18)                                   -> ``int(num)`` shim
  * ``pyradClasses.py:1024``  lists ``./data/xsc`` at import        -> pre-created

The harness never modifies reference files and never copies them.
"""
import contextlib
import importlib
import io
import json
import os
import sys

import numpy as np

REFERENCE_DIR = os.environ.get("PYRAD_REFERENCE_DIR", "/root/reference")
STUB_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "stubs")

_REF_MODULES = ("pyradUtilities", "pyradLineshape", "pyradIntensity", "pyradPlanck",
                "pyradClasses", "pyradInteractive", "bs4", "matplotlib", "matplotlib.pyplot")

#: every global isotopologue id the reference's HITRAN_GLOBAL_ISO table mentions
#: (pyradUtilities.py:863-987) lies in 1..129; seeding 1..130 is a superset.
_ALL_GLOBAL_ISO = range(1, 131)


def available():
    return os.path.isfile(os.path.join(REFERENCE_DIR, "pyradClasses.py"))


def _linspace_int_shim():
    orig = np.linspace
    if getattr(orig, "_pyrad_shim", False):
        return

    def linspace(start, stop, num=50, *a, **kw):
        return orig(start, stop, int(num), *a, **kw)

    linspace._pyrad_shim = True
    np.linspace = linspace


def seed_workdir(workdir):
    """Create the cwd-relative ``data/`` tree the reference expects."""
    data = os.path.join(workdir, "data")
    os.makedirs(os.path.join(data, "curves"), exist_ok=True)
    os.makedirs(os.path.join(data, "xsc"), exist_ok=True)
    for gid in _ALL_GLOBAL_ISO:
        d = os.path.join(data, str(gid))
        os.makedirs(d, exist_ok=True)
        p = os.path.join(d, "params.pyr")
        if not os.path.isfile(p):
            write_params(workdir, gid, "x%d" % gid, 0, 0, 1.0, 1.0, 1, 1.0)


def write_params(workdir, global_iso, short_name, mol_num, iso_n, abundance, q296, gj, molmass):
    """``params.pyr`` row as parsed by readMolParams (pyradUtilities.py:464-477)."""
    d = os.path.join(workdir, "data", str(global_iso))
    os.makedirs(d, exist_ok=True)
    with open(os.path.join(d, "params.pyr"), "w") as f:
        f.write("# params\n")
        f.write("%d,%s,%d,%d,%r,%r,%d,%r\n" % (global_iso, short_name, mol_num, iso_n,
                                                 float(abundance), float(q296), gj, float(molmass)))


def write_q_table(workdir, global_iso, temps, qvals):
    """``q<iso>.txt`` rows ``T Q`` for integer T (readQFile, pyradUtilities.py:451-461)."""
    d = os.path.join(workdir, "data", str(global_iso))
    os.makedirs(d, exist_ok=True)
    with open(os.path.join(d, "q%d.txt" % global_iso), "w") as f:
        for t, q in zip(temps, qvals):
            f.write("%d %r\n" % (int(t), float(q)))


def write_line_segments(workdir, global_iso, mol_id, local_iso, lines, seg_min, seg_max):
    """HITRAN-online CSV ``<segment>.pyr`` files, one per 100 cm^-1 segment
    (gatherData pyradUtilities.py:173-189; columns readHitranOnlineFile :421-448:
    molec_id,local_iso_id,nu,sw,a,elower,gamma_air,gamma_self,delta_air,n_air).

    ``lines`` is a dict of equal-length float64 arrays with keys
    nu, sw, a, elower, gamma_air, gamma_self, delta_air, n_air, ascending in nu.
    Every segment in [seg_min, seg_max) is written (empty segments get a comment
    row only -- a missing file would trigger a network download attempt).
    Values are written with ``repr`` so ``float(text)`` round-trips bit-exactly.
    """
    d = os.path.join(workdir, "data", str(global_iso))
    os.makedirs(d, exist_ok=True)
    nu = np.asarray(lines["nu"], dtype=np.float64)
    seg = int(seg_min / 100) * 100
    while seg < seg_max:
        lo = np.searchsorted(nu, seg, side="left")
        hi = np.searchsorted(nu, seg + 100, side="left")
        with open(os.path.join(d, "%d.pyr" % seg), "w") as f:
            f.write("# synthetic HITRAN-online segment\n")
            for j in range(lo, hi):
                f.write("%d,%d,%r,%r,%r,%r,%r,%r,%r,%r\n" % (
                    mol_id, local_iso, float(nu[j]), float(lines["sw"][j]), float(lines["a"][j]),
                    float(lines["elower"][j]), float(lines["gamma_air"][j]),
                    float(lines["gamma_self"][j]), float(lines["delta_air"][j]),
                    float(lines["n_air"][j])))
        seg += 100


def write_xsc_file(workdir, name, temp, torr, rmin, rmax, res, wavenumber, intensity,
                   broadener="air", ident="00_00"):
    """xsc table named so that parseXscFileName's regexes match (pyradUtilities.py:611-641);
    two whitespace-separated columns (returnXscFileContents :680-696)."""
    d = os.path.join(workdir, "data", "xsc", name)
    os.makedirs(d, exist_ok=True)
    fname = "%s_%sK-%sTorr_%s-%s_%s_%s_%s.txt" % (name, temp, torr, rmin, rmax, res, broadener, ident)
    with open(os.path.join(d, fname), "w") as f:
        f.write("# synthetic xsc\n")
        for w, c in zip(wavenumber, intensity):
            f.write("%r     %r\n" % (float(w), float(c)))
    return fname


class Reference:
    """Namespace holding the imported real reference modules."""

    def __init__(self, workdir, mods):
        self.workdir = workdir
        self.utils = mods["pyradUtilities"]
        self.lineshape = mods["pyradLineshape"]
        self.intensity = mods["pyradIntensity"]
        self.planck = mods["pyradPlanck"]
        self.classes = mods["pyradClasses"]

    def set_base_resolution(self, res):
        """BASE_RESOLUTION is a module constant (pyradUtilities.py:804-805); 0.001 grids
        require overriding it after import and dynamicResolution=False (SURVEY 8(a) a11)."""
        self.utils.BASE_RESOLUTION = res


def reference_id_tables():
    """MOLECULE_ID and HITRAN_GLOBAL_ISO as the dict literals of the reference source (pyradClasses.py:951-1022), read
    without importing it; None where the sources are absent."""
    path = os.path.join(REFERENCE_DIR, "pyradClasses.py")
    if not os.path.isfile(path):
        return None
    with open(path) as f:
        src = f.read()
    ns = {}
    for name in ("HITRAN_GLOBAL_ISO", "MOLECULE_ID"):
        i = src.index(name + " = {")
        depth, j = 0, i
        while True:                                    # the dict literal: up to its matching brace
            ch = src[j]
            depth += ch == "{"
            depth -= ch == "}"
            j += 1
            if ch == "}" and depth == 0:
                break
        exec(src[i:j], ns)
    return {"MOLECULE_ID": ns["MOLECULE_ID"], "HITRAN_GLOBAL_ISO": ns["HITRAN_GLOBAL_ISO"]}


def id_tables_json(tables):
    """The layout of tests/golden/hitran_id_tables.json: the name table on one line, one isotopologue row per line."""
    rows = list(tables["HITRAN_GLOBAL_ISO"].items())
    out = ["{", ' "MOLECULE_ID": ' + json.dumps(tables["MOLECULE_ID"]) + ",", ' "HITRAN_GLOBAL_ISO": {']
    for k, (mol, isos) in enumerate(rows):
        out.append('  "%d": %s%s' % (mol, json.dumps({str(i): g for i, g in isos.items()}), "," if k < len(rows) - 1 else ""))
    return "\n".join(out + [" }", "}"]) + "\n"


@contextlib.contextmanager
def quiet():
    """The reference prints progress bars from inside the hot loop (pyradClasses.py:372-375)."""
    with contextlib.redirect_stdout(io.StringIO()):
        yield


def load_reference(workdir):
    """Import the real reference with cwd = ``workdir`` (seeded first).  Re-imports from
    scratch every call because module-level paths are frozen at import time."""
    if not available():
        raise RuntimeError("reference sources not present at %s" % REFERENCE_DIR)
    seed_workdir(workdir)
    _linspace_int_shim()
    for m in _REF_MODULES:
        sys.modules.pop(m, None)
    saved_path = list(sys.path)
    saved_cwd = os.getcwd()
    sys.path[:0] = [STUB_DIR, REFERENCE_DIR]
    os.chdir(workdir)
    try:
        with quiet():
            mods = {m: importlib.import_module(m) for m in
                    ("pyradUtilities", "pyradLineshape", "pyradIntensity", "pyradPlanck", "pyradClasses")}
    finally:
        sys.path[:] = saved_path
        # stay in workdir? no: paths are already frozen inside pyradUtilities (cwd at import)
        os.chdir(saved_cwd)
        for m in ("bs4", "matplotlib", "matplotlib.pyplot", "pyradInteractive"):
            sys.modules.pop(m, None)
    mods["pyradClasses"].Layer.hasAtmosphere = False
    return Reference(workdir, mods)
