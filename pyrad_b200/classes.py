"""Host-side mirror of the reference's object model (reference pyradClasses.py:237-821): the same class
names, constructor signatures, attribute names, getters and error behaviour, with every piece of physics
delegated to the CUDA engine through the C ABI.  This is the drop-in layer: menus and plots written
against ``Atmosphere > Layer > Molecule > Isotope > Line`` keep working, the numpy hot path is gone.

What runs where
  Isotope.createCrossSection  -> prb_upload_lines + prb_set_grid + prb_layer_prepass + prb_line_sum   (K0/K1/K2)
  absCoef / transmittance / transmission / planck                    -> prb_layer_stream / prb_planck  (K3)
  xsc Molecule ingest (np.interp + aligned placement)                -> prb_xsc_place                 (K3)
There is no CPU fallback: without the shared library or a B200 these calls raise EngineUnavailable.

Reference quirks kept on purpose (parity, SURVEY.md section 8(a)):
  * Q(T) is a dict lookup at the layer temperature: non-integer T raises KeyError (pyradClasses.py:389).
  * the grid index uses the UN-shifted wavenumber, widths and S(T) the pressure-shifted one (:388-390).
  * changePressure updates the cutoff and resolution but not effectiveRangeMin/Max (:745-752).
  * xAxis is linspace(rangeMin, rangeMax, N) -- spacing (max-min)/(N-1), not the resolution (:703-705).
  * an xsc molecule forces the layer's T and P to the file's (:488-491); the xsc path is only defined on
    a 0.01 cm-1 base grid (:493, :177-178).
"""
import numpy as np

from . import engine as _eng
from . import hitran_io as _io

# constants as the reference spells them (pyradClasses.py:15-23)
c = 299792458.0
k = 1.38064852E-23
h = 6.62607004e-34
pi = 3.141592653589793
t0 = 296
p0 = 1013.25
avo = 6.022140857E23

#: mirror of utils.BASE_RESOLUTION (pyradUtilities.py:804-805); assign to change the base grid
BASE_RESOLUTION = .01
#: root of the reference-format data tree (defaults to cwd, like the reference)
DATA_ROOT = None

#: largest grid span handed to one K2 launch: FP32 offsets must stay exact integers (< 2^24)
_MAX_SPAN = 1 << 23

import itertools as _it
#: unique tokens for "this object / this line list" in Layer._state_key (id() values are reused after a free)
_TOKEN = _it.count(1)

_ENGINE = None
#: state key of the Layer whose per-isotopologue rows the engine currently holds (Layer._device_rows)
_RESIDENT_KEY = None


def engine():
    """The process-wide CUDA engine (created on first use; raises EngineUnavailable without a B200)."""
    global _ENGINE
    if _ENGINE is None:
        set_engine(_eng.Engine(0))
    return _ENGINE


def set_engine(e):
    global _ENGINE, _RESIDENT_KEY
    _ENGINE = e
    _RESIDENT_KEY = None
    # spectra handed to the caller come from a pool of page-locked arrays that are reused once dropped (engine.ResultPool)
    if e is not None and getattr(e, "result_pool", None) is None:
        e.result_pool = _eng.ResultPool()


def _n_base(obj):
    return int((obj.rangeMax - obj.rangeMin) / BASE_RESOLUTION)


# ---------------------------------------------------------------------------------- module-level getters
def printProgress(text, obj):
    """Progress line of the reference's per-isotopologue loop (pyradClasses.py:98-102); kept for callers that print it."""
    print('Processing %s: %s; %s; isotope %s' % (text, obj.layer.name, obj.molecule.name, obj.name))


def cacheCurves():
    """The reference writes its memoised line-shape curves to disk here (pyradClasses.py:947-948, pyradLineshape.py).
    The device path evaluates every shape in place and keeps no curve cache: nothing to write."""
    return None


def integrateSpectrum(spectrum, unitAngle=pi, res=None):
    res = BASE_RESOLUTION if res is None else res
    return engine().integrate_spectrum(spectrum, unitAngle, res)          # device reduction (K4)


def getCrossSection(obj):
    if not obj.progressCrossSection:
        obj.createCrossSection()
    return obj.crossSection


def getAbsCoef(obj):
    if not obj.progressCrossSection:
        obj.createCrossSection()
    return obj.absCoef


def getTransmittance(obj):
    if not obj.progressCrossSection:
        obj.createCrossSection()
    return obj.transmittance


def getOpticalDepth(obj):
    if not obj.progressCrossSection:
        obj.createCrossSection()
    return engine().derived_spectra(obj.transmittance, want=("optical_depth",))["optical_depth"]


def getAbsorbance(obj):
    if not obj.progressCrossSection:
        obj.createCrossSection()
    return obj.absorbance


def getEmissivity(obj):
    if not obj.progressCrossSection:
        obj.createCrossSection()
    return obj.emissivity


def resetCrossSection(obj):
    if not isinstance(obj, Layer):
        if not obj.exotic:
            obj.crossSection = None                   # reads as np.zeros(N) (the reference's reset value), made on demand
            obj.progressCrossSection = False
    else:
        obj.progressCrossSection = False
        obj._cs = None                                # the layer's own sum is rebuilt from its molecules on demand
    if isinstance(obj, Isotope):
        return                                        # its children are lines (views): nothing to reset
    for child in obj:
        resetCrossSection(child)


def resetData(obj):
    for child in obj:
        if isinstance(child, Isotope):
            child.clearLines()
            child.getData()
        else:
            resetData(child)
    resetCrossSection(obj)


def totalConcentration(layer):
    return sum(m.concentration for m in layer)


def totalLineList(obj):
    if isinstance(obj, Isotope):
        return obj.linelist()
    out = []
    for item in obj:
        out += totalLineList(item)
    return out


def convertLength(value, units):
    return {"cm": value, "m": value * 100, "meter": value * 100, "ft": value * 30.48, "feet": value * 30.48,
            "in": value * 2.54, "inch": value * 2.54}.get(units)


def convertPressure(value, units):
    if units == "mbar":
        return value
    if units in ("atm", "atmospheres", "atmosphere"):
        return value * 1013.25
    if units in ("b", "bar"):
        return value * 1000
    if units in ("pa", "pascal", "pascals"):
        return value / 100


def convertRange(value, units):
    if units == "cm-1":
        return value
    if units in ("um", "micrometers", "micrometer"):
        return 10000 / value


def convertTemperature(value, units):
    u = units[0].upper()
    if u == "K":
        return value
    if u == "C":
        return value + 273
    if u == "F":
        return (value - 32) * 5 / 9 + 273


def isBetween(test, minValue, maxValue):
    return minValue <= test <= maxValue


def _merge_plan(newX, oldX):
    """Index plan of the reference's mergeArray (pyradClasses.py:165-233): (dst0, src0, count, out_len).
    Same 2-decimal rounding and first-match lookups; the last source sample is dropped (:226)."""
    nx = [round(float(v), 2) for v in np.asarray(newX).tolist()]
    ox = [round(float(v), 2) for v in np.asarray(oldX).tolist()]
    if max(nx) < min(ox) or min(nx) > max(ox):
        return 0, 0, 0, len(nx)
    if min(nx) <= min(ox):
        dst0, src0 = nx.index(min(ox)), 0
    else:
        dst0, src0 = 0, ox.index(min(nx))
    if max(nx) >= max(ox):
        final_new, final_old = dst0 + len(ox) - 1, len(ox) - 1
    else:
        final_new, final_old = len(nx) - 1, src0 + len(nx) - 1
    count = max(final_old - src0, 0)
    if src0 + count > len(ox):
        raise IndexError("list index out of range")               # the reference's copy loop runs off oldY (:224-226)
    out_len = dst0 + count + max(len(nx) - final_new, 0)          # ([0] * negative is an empty list, :229)
    return dst0, src0, count, out_len


def mergeArray(newX, oldX, oldY):
    """Aligned placement of (oldX, oldY) onto newX, zeros elsewhere -- on the device (prb_xsc_place)."""
    dst0, src0, count, out_len = _merge_plan(newX, oldX)
    if out_len != len(newX):
        raise ValueError("mergeArray: partially overlapping ranges are not supported (the reference returns a "
                         "wrong-length array here, pyradClasses.py:217-231)")
    return engine().xsc_place(len(newX), dst0, src0, count, None, np.asarray(oldY, dtype=np.float64), interp=False)


def interpolateArray(hiResXAxis, loResXAxis, loResYValues):
    """np.interp on the device for uniformly generated targets; falls back to per-point targets otherwise."""
    x = np.asarray(hiResXAxis, dtype=np.float64)
    if x.size >= 2:
        d = x[1] - x[0]
        if np.array_equal(x, x[0] + np.arange(x.size) * d):
            return engine().xsc_place(x.size, 0, 0, x.size, loResXAxis, loResYValues, interp=True, ax0=x[0], adelta=d)
    raise ValueError("interpolateArray: target axis must be start + i*step (np.arange / reference usage)")


# ---------------------------------------------------------------------------------- object model
class Line:
    """One transition; a view into the parent isotopologue's SoA columns (pyradClasses.py:237-263)."""
    __slots__ = ("isotope", "_i")

    def __init__(self, parent, index):
        self.isotope = parent
        self._i = index

    molecule = property(lambda s: s.isotope.molecule)
    layer = property(lambda s: s.isotope.molecule.layer)
    wavenumber = property(lambda s: float(s.isotope._cols["nu"][s._i]))
    intensity = property(lambda s: float(s.isotope._cols["sw"][s._i]))
    einsteinA = property(lambda s: float(s.isotope._cols["a"][s._i]))
    airHalfWidth = property(lambda s: float(s.isotope._cols["gamma_air"][s._i]))
    selfHalfWidth = property(lambda s: float(s.isotope._cols["gamma_self"][s._i]))
    lowerEnergy = property(lambda s: float(s.isotope._cols["elower"][s._i]))
    tempExponent = property(lambda s: float(s.isotope._cols["n_air"][s._i]))
    pressureShift = property(lambda s: float(s.isotope._cols["delta_air"][s._i]))

    @property
    def broadenedLine(self):
        return self.wavenumber + self.pressureShift * self.layer.P / p0

    @property
    def lorentzHW(self):
        q = self.molecule.concentration
        return float((1 - q) * self.airHalfWidth + q * self.selfHalfWidth) * (self.layer.P / p0) * \
            (t0 / self.layer.T) ** self.tempExponent

    @property
    def gaussianHW(self):
        return self.broadenedLine * np.sqrt(2 * k * self.layer.T / self.isotope.molMass / c ** 2)


class _LazyCrossSection:
    """crossSection of an Isotope / Molecule: an array, or None for "reset" -- which reads as np.zeros(N), built when
    somebody looks (resetting a layer of 3 M-point spectra is then free instead of eight 24 MB memsets)."""

    @property
    def crossSection(self):
        if self._cs is None:
            self._cs = np.zeros(_n_base(self))
        return self._cs

    @crossSection.setter
    def crossSection(self, value):
        self._cs = value


class _Spectral:
    """Pointwise spectra shared by Isotope / Molecule / Layer: all evaluated by K3 on the device."""

    def _sigma_rows(self):
        raise NotImplementedError

    def _stream(self, want, radiance_in=None):
        layer = self.layer if not isinstance(self, Layer) else self
        rows, weights = self._sigma_rows()
        axis = _eng.linspace_axis(layer.rangeMin, layer.rangeMax, _n_base(layer))
        return engine().layer_stream(rows, weights, layer.depth, layer.T, axis, radiance_in, want=want)

    @property
    def absCoef(self):
        return self._stream(("abs_coef",))[0]

    @property
    def transmittance(self):
        return self._stream(("transmittance",))[1]

    @property
    def emissivity(self):
        return engine().derived_spectra(self.transmittance, want=("emissivity",))["emissivity"]

    @property
    def emittance(self):
        return self.emissivity

    @property
    def absorbance(self):
        return engine().derived_spectra(self.transmittance, want=("absorbance",))["absorbance"]

    def transmission(self, surfaceSpectrum):
        return self._stream(("radiance",), np.asarray(surfaceSpectrum, dtype=np.float64))[2]


class Isotope(list, _Spectral, _LazyCrossSection):
    """An isotopologue and its lines.  The reference fills the list with one Line object per transition
    (pyradClasses.py:350-359); here the transitions live in SoA columns and the list protocol hands out Line VIEWS on
    demand (len / iteration / indexing / linelist()), so a 5 M-line list costs its columns, not 5 M Python objects."""

    def __init__(self, number, molecule):
        list.__init__(self)
        self.molecule = molecule
        self.layer = molecule.layer
        self.crossSection = None                      # zeros until computed (the reference copies the fresh layer's zeros)
        self.exotic = molecule.exotic
        self._cols = {kname: np.zeros(0) for kname in _io.LINE_COLUMNS}
        self._lines_token = next(_TOKEN)
        if not isinstance(number, str):
            p = _io.read_mol_params(number, DATA_ROOT)
            self.globalIsoNumber = p["globalIso"]
            self.shortName = p["shortName"]
            self.name = "Isotope %s" % self.globalIsoNumber
            self.molNum = p["molNum"]
            self.isoN = p["isoN"]
            self.abundance = p["abundance"]
            self.q296 = p["q296"]
            self.gj = p["gj"]
            self.molmass = p["molmass"]
            self.q = {}
            self.lineSurvey = np.zeros(_n_base(self.layer))
            self.progressCrossSection = False
        else:
            self.name = number

    P = property(lambda s: s.layer.P)
    T = property(lambda s: s.layer.T)
    depth = property(lambda s: s.layer.depth)
    rangeMin = property(lambda s: s.layer.rangeMin)
    rangeMax = property(lambda s: s.layer.rangeMax)
    resolution = property(lambda s: s.layer.resolution)
    distanceFromCenter = property(lambda s: s.layer.distanceFromCenter)
    yAxis = property(lambda s: np.copy(s.layer.yAxis))
    xAxis = property(lambda s: np.copy(s.layer.xAxis))

    @property
    def molMass(self):
        return self.molmass / 1000 / avo

    # -- the list protocol over the SoA columns (views are created when asked for)
    def __len__(self):
        return len(self._cols["nu"])

    def __bool__(self):
        return True

    def __iter__(self):
        return (Line(self, i) for i in range(len(self)))

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [Line(self, j) for j in range(*i.indices(len(self)))]
        n = len(self)
        if i < 0:
            i += n
        if not 0 <= i < n:
            raise IndexError("line index out of range")
        return Line(self, i)

    def __eq__(self, other):
        return self is other

    def __ne__(self, other):
        return self is not other

    __hash__ = object.__hash__

    def clearLines(self):
        self._cols = {kname: np.zeros(0) for kname in _io.LINE_COLUMNS}
        self._lines_token = next(_TOKEN)

    def setLines(self, cols, q_table=None):
        """Attach a line list directly (SoA float64 columns, ascending nu) instead of reading the data tree.  A column
        that is absent (the Einstein A of a synthetic list) reads as zeros."""
        n = len(cols["nu"])
        # the isotopologue owns its columns, in page-locked memory when a device is there: every later upload of the
        # list then runs at PCIe speed instead of through the driver's staging buffer
        block = _eng.PinnedBlock((8 * n + 64) * len(_io.LINE_COLUMNS))
        self._cols = {}
        for kname in _io.LINE_COLUMNS:
            a = block.array(n)
            a[:] = cols[kname] if kname in cols else 0.0
            self._cols[kname] = a
        self._cols_block = block
        self._lines_token = next(_TOKEN)
        if q_table is not None:
            self.q = q_table
        self.progressCrossSection = False

    def getData(self):
        global _RESIDENT_KEY
        _RESIDENT_KEY = None                          # the device parser replaces the engine's line list
        cols = _io.gather_lines(self.globalIsoNumber, self.layer.effectiveRangeMin, self.layer.effectiveRangeMax,
                                DATA_ROOT, engine())
        self.setLines(cols, _io.read_q_table(self.globalIsoNumber, DATA_ROOT))
        self.createLineSurvey()

    def createCrossSection(self):
        layer = self.layer
        res = layer.resolution
        n_res = int((self.rangeMax - self.rangeMin) / res)
        q_t = self.q[layer.T]                                  # KeyError on a non-tabulated T, as the reference
        rows = layer._group_rows() if isinstance(layer, Layer) else None
        if rows is not None and id(self) in rows:
            # ONE upload + ONE prepass + ONE line-sum launch made every isotopologue's row of this layer
            self.crossSection = rows[id(self)]
            self.progressCrossSection = True
            return
        global _RESIDENT_KEY
        _RESIDENT_KEY = None
        e = engine()
        window = _eng.window_len(layer.distanceFromCenter, res)
        wm = max(window - 2, 0)
        e.upload_lines(self._cols, n_groups=1)
        span = max(_MAX_SPAN - 2 * wm - 16384, 4096) // 4096 * 4096
        parts = []
        for a in range(0, max(n_res, 1), span):
            b = min(a + span, n_res)
            e.set_grid(self.rangeMin, res, n_res, a, b)
            e.layer_prepass(layer.T, layer.P, [self.molecule.concentration], [self.molmass], [q_t], [self.q296], window)
            parts.append(e.line_sum())
        sigma = np.concatenate(parts) if parts else np.zeros(0)
        if res != BASE_RESOLUTION:
            # np.interp(xAxis, linspace(rangeMin, rangeMax, n_res), sigma)   (pyradClasses.py:401-405)
            xr = np.linspace(self.rangeMin, self.rangeMax, n_res, endpoint=True)
            ax = _eng.linspace_axis(self.rangeMin, self.rangeMax, _n_base(self))
            sigma = e.xsc_place(ax[3], 0, 0, ax[3], xr, sigma, interp=True, ax0=ax[0], adelta=ax[1])
        self.crossSection = sigma
        self.progressCrossSection = True

    def createLineSurvey(self):
        """pyradClasses.py:409-428 on the device (K4): S296 summed per grid bin in line order, bit-exact."""
        n_out = _n_base(self)
        nu = self._cols["nu"]
        if nu.size:
            global _RESIDENT_KEY
            _RESIDENT_KEY = None
            e = engine()
            e.upload_lines(self._cols, 1)
            e.set_grid(self.layer.rangeMin, self.layer.resolution, max(n_out, 1))
            survey = e.line_survey(n_out)
        else:
            survey = np.zeros(n_out)
        self.lineSurvey = survey
        return survey

    def linelist(self):
        return [Line(self, i) for i in range(len(self))]

    def planck(self, temperature):
        return self.layer.planck(temperature)

    def _sigma_rows(self):
        w = _eng.number_density_weight(self.molecule.concentration, self.layer.P, self.layer.T)
        return self.crossSection[None, :], [w]


class Molecule(list, _Spectral, _LazyCrossSection):
    def __init__(self, shortNameOrMolNum, layer, isotopeDepth=1, **abundance):
        list.__init__(self)
        self.layer = layer
        self.concText = ""
        self.concentration = 0
        self.exotic = False
        self.crossSection = None                      # zeros until computed (the reference copies the fresh layer's zeros)
        self.progressCrossSection = False
        for key, val in abundance.items():
            if key == "ppm":
                self.setPPM(val)
            elif key == "ppb":
                self.setPPB(val)
            elif key in ("percentage", "perc", "%"):
                self.setPercentage(val)
            elif key == "concentration":
                self.setConcentration(val)
            else:
                print("Invalid concentration type. Use ppm, ppb, percentage, or concentration.")
        if type(shortNameOrMolNum) is dict:
            self._init_xsc(shortNameOrMolNum)
        else:
            self.isotopeDepth = isotopeDepth
            try:
                self.ID = int(shortNameOrMolNum)
                self.name = False
            except ValueError:
                self.name = shortNameOrMolNum
                self.ID = MOLECULE_ID[self.name]
            for gid in getGlobalIsotope(self.ID, isotopeDepth):
                iso = Isotope(gid, self)
                self.append(iso)
                if not self.name:
                    self.name = iso.shortName

    def _init_xsc(self, spec):
        """xsc branch (pyradClasses.py:466-505): table -> 0.01 grid (np.interp when coarser) -> aligned placement."""
        name, filename = list(spec.items())[0]
        wn, xs = _io.read_xsc_table(name, filename, DATA_ROOT, engine())
        info = _io.parse_xsc_filename(filename)
        rmin, rmax = (float(v) for v in info["RANGE"].split("-"))
        temp = int(float(info["TEMP"]))
        pressure = float(info["PRESSURE"]) / 0.75006
        low_res = float(info["RES"])
        self.name = name
        dummy = Isotope(name, self)
        self.exotic = True
        dummy.exotic = True
        if temp != self.layer.T:
            self.layer.changeTemperature(temp)
        if pressure != self.layer.P:
            self.layer.changePressure(pressure)
        x_axis = np.arange(rmin, rmax, .01)
        dst0, src0, count, out_len = _merge_plan(self.layer.xAxis, x_axis)
        n = len(self.layer.xAxis)
        if out_len != n:
            raise ValueError("xsc range partially overlaps the layer range: undefined in the reference (mergeArray)")
        if low_res > .01:
            a0 = float(x_axis[0])
            ad = float(x_axis[1] - x_axis[0]) if len(x_axis) > 1 else .01
            sigma = engine().xsc_place(n, dst0, src0, count, wn, xs, interp=True, ax0=a0, adelta=ad)
            self._xsc_plan = dict(n_out=n, dst0=dst0, src0=src0, count=count, file_x=wn, file_y=xs, interp=True, ax0=a0, adelta=ad)
        else:
            sigma = engine().xsc_place(n, dst0, src0, count, None, xs, interp=False)
            self._xsc_plan = dict(n_out=n, dst0=dst0, src0=src0, count=count, file_x=None, file_y=xs, interp=False)
        self._xsc_key = (name, filename)
        dummy.crossSection = sigma
        dummy.progressCrossSection = True
        self.crossSection = sigma
        self.progressCrossSection = True

    def __str__(self):
        return "%s: %s" % (self.name, self.concText)

    def __bool__(self):
        return True

    def returnCopy(self):
        value, unit = self.concText.split()
        m = Molecule(self.name, self.layer, isotopeDepth=int(self.isotopeDepth), **{unit: float(value)})
        m.getData()
        return m

    def setPercentage(self, percentage):
        self.concentration = percentage / 100
        self.concText = "%s %%" % percentage
        resetCrossSection(self)

    def setPPM(self, ppm):
        self.concentration = ppm * 10 ** -6
        self.concText = "%s ppm" % ppm
        resetCrossSection(self)

    def setPPB(self, ppb):
        self.concentration = ppb * 10 ** -8            # sic: the reference scales ppb by 1e-8 (pyradClasses.py:554)
        self.concText = "%s ppb" % ppb
        resetCrossSection(self)

    def setConcentration(self, concentration):
        self.setPPM(concentration * 1E6)
        resetCrossSection(self)

    def getData(self):
        for iso in self:
            iso.getData()

    def createCrossSection(self):
        total = np.zeros(_n_base(self))
        for iso in self:
            total += getCrossSection(iso)
        self.progressCrossSection = True
        self.crossSection = total

    def planck(self, temperature):
        return self.layer.planck(temperature)

    @property
    def lineSurvey(self):
        total = np.zeros(_n_base(self))
        for iso in self:
            total += iso.lineSurvey
        return total

    P = property(lambda s: s.layer.P)
    T = property(lambda s: s.layer.T)
    depth = property(lambda s: s.layer.depth)
    rangeMin = property(lambda s: s.layer.rangeMin)
    rangeMax = property(lambda s: s.layer.rangeMax)
    resolution = property(lambda s: s.layer.resolution)
    distanceFromCenter = property(lambda s: s.layer.distanceFromCenter)
    yAxis = property(lambda s: np.copy(s.layer.yAxis))
    xAxis = property(lambda s: np.copy(s.layer.xAxis))

    def _sigma_rows(self):
        return self.crossSection[None, :], [_eng.number_density_weight(self.concentration, self.layer.P, self.layer.T)]


class Layer(list, _Spectral):
    hasAtmosphere = False

    def __init__(self, depth, T, P, rangeMin, rangeMax, atmosphere=None, name="", dynamicResolution=True):
        list.__init__(self)
        self.rangeMin = rangeMin
        self.rangeMax = rangeMax
        self.T = T
        self.P = P
        self.depth = depth
        self.distanceFromCenter = self.P / 1013.25 * 5
        self.effectiveRangeMin = max(self.rangeMin - self.distanceFromCenter, 0)
        self.effectiveRangeMax = self.rangeMax + self.distanceFromCenter
        self.dynamicResolution = dynamicResolution
        self.resolution = self._pick_resolution()
        if not atmosphere:
            if not Layer.hasAtmosphere:
                self.atmosphere = Atmosphere("generic")
                Layer.hasAtmosphere = self.atmosphere
            else:
                self.atmosphere = Layer.hasAtmosphere
        else:
            self.atmosphere = atmosphere
            self.hasAtmosphere = atmosphere
        self._cs = np.zeros(int((rangeMax - rangeMin) / BASE_RESOLUTION))
        self._rows_cache = (None, None)
        self._token = next(_TOKEN)
        self.progressCrossSection = False
        self.exotic = False
        self.name = name or "layer %s" % self.atmosphere.nextLayerName()

    def _pick_resolution(self):
        if not self.dynamicResolution:
            return BASE_RESOLUTION
        return max(10 ** int(np.log10((self.P / 1013.25))) * .01, BASE_RESOLUTION)

    def __str__(self):
        return "%s; %s" % (self.name, "; ".join(str(m) for m in self))

    def __bool__(self):
        return True

    layer = property(lambda s: s)

    def createCrossSection(self):
        if self._device_rows():
            # the rows are on the device; the layer's own (unweighted) sum and its children's rows are fetched when
            # somebody asks for them (crossSection below, Isotope.createCrossSection)
            self._cs = None
            self.progressCrossSection = True
            return
        total = np.zeros(_n_base(self))
        for m in self:
            total += getCrossSection(m)
        self.progressCrossSection = True
        self.crossSection = total

    @property
    def crossSection(self):
        if self._cs is None:
            total = np.zeros(_n_base(self))
            for m in self:
                total += getCrossSection(m)
            self._cs = total
        return self._cs

    @crossSection.setter
    def crossSection(self, value):
        self._cs = value

    @property
    def lineSurvey(self):
        total = np.zeros(_n_base(self))
        for m in self:
            total += m.lineSurvey
        return total

    @property
    def yAxis(self):
        return np.zeros(int((self.rangeMax - self.rangeMin) / self.resolution))

    @property
    def xAxis(self):
        return np.linspace(self.rangeMin, self.rangeMax, _n_base(self), endpoint=True)

    @property
    def title(self):
        return "%s\nP: %smBars; T: %sK; depth: %scm" % (str(self), self.P, self.T, self.depth)

    def _sigma_rows(self):
        """One sigma row and one number-density weight per molecule: k_layer = sum_m sigma_m * w_m (:707-712)."""
        rows = [getCrossSection(m) for m in self]
        if not rows:
            return np.zeros((1, _n_base(self))), [0.0]
        return np.array(rows), [_eng.number_density_weight(m.concentration, self.P, self.T) for m in self]

    # -- the device-resident path of a layer: every isotopologue's line list uploaded as it is (grouped, no merge),
    #    ONE prepass, ONE line-sum launch with a row per isotopologue, xsc tables resident; k / T / transmission are then
    #    formed on the device from those rows and only the requested spectrum crosses PCIe
    def _isos(self):
        return [iso for m in self if not m.exotic for iso in m]

    def _state_key(self):
        isos = self._isos()
        return (self._token, self.T, self.P, self.rangeMin, self.rangeMax, self.resolution, self.distanceFromCenter, BASE_RESOLUTION,
                tuple((iso._lines_token, len(iso), iso.molmass, iso.q296, iso.molecule.concentration, iso.q.get(self.T))
                      for iso in isos),
                tuple(m._xsc_key for m in self if m.exotic))

    def _device_rows(self):
        """Make the engine hold this layer's per-isotopologue rows (and xsc tables); False when the one-pass path does
        not apply (dynamic resolution coarser than the base grid, a grid too long for one launch, no line-by-line
        molecule, more than eight xsc tables) -- callers then take the per-isotopologue path."""
        global _RESIDENT_KEY
        isos = self._isos()
        xmols = [m for m in self if m.exotic]
        n = _n_base(self)
        window = _eng.window_len(self.distanceFromCenter, self.resolution)
        if not isos or self.resolution != BASE_RESOLUTION or len(xmols) > 8 or \
                n + 2 * max(window - 2, 0) + 16384 >= _MAX_SPAN or n < 1:
            return False
        key = self._state_key()
        if _RESIDENT_KEY == key:
            return True
        _RESIDENT_KEY = None
        q_t = [iso.q[self.T] for iso in isos]                  # KeyError on a non-tabulated T, as the reference
        e = engine()
        e.upload_line_groups([iso._cols for iso in isos])
        e.set_grid(self.rangeMin, self.resolution, n)
        e.layer_prepass(self.T, self.P, [iso.molecule.concentration for iso in isos], [iso.molmass for iso in isos], q_t,
                        [iso.q296 for iso in isos], window)
        e.line_sum_groups(to_host=False)
        e.xsc_clear()
        for slot, m in enumerate(xmols):
            e.xsc_resident(slot, **m._xsc_plan)
        _RESIDENT_KEY = key
        return True

    def _group_rows(self):
        """{id(isotopologue): cross-section row} of the layer's one-pass result (one D2H for all rows, cached until the
        layer's state changes), or None when the one-pass path does not apply."""
        if not self._device_rows():
            return None
        key = self._state_key()
        if self._rows_cache[0] != key:
            rows = engine().line_sum_groups(to_host=True)
            self._rows_cache = (key, {id(iso): rows[g] for g, iso in enumerate(self._isos())})
        return self._rows_cache[1]

    def _stream(self, want, radiance_in=None):
        if self._device_rows():
            w = [_eng.number_density_weight(iso.molecule.concentration, self.P, self.T) for iso in self._isos()]
            xw = [_eng.number_density_weight(m.concentration, self.P, self.T) for m in self if m.exotic]
            return engine().layer_spectra_resident(w, self.depth, self.T, self.rangeMax, xw, radiance_in, want=want)
        return _Spectral._stream(self, want, radiance_in)

    def changeRange(self, rangeMin, rangeMax):
        self.rangeMin = rangeMin
        self.rangeMax = rangeMax
        self.effectiveRangeMax = self.rangeMax + self.distanceFromCenter
        self.effectiveRangeMin = max(self.rangeMin - self.distanceFromCenter, 0)
        self.crossSection = np.zeros(_n_base(self))
        resetData(self)

    def changeTemperature(self, temperature):
        self.T = temperature
        resetCrossSection(self)

    def changePressure(self, pressure):
        self.P = pressure
        self.distanceFromCenter = self.P / 1013.25 * 5
        self.resolution = self._pick_resolution()
        resetData(self)

    def changeDepth(self, depth):
        self.depth = depth

    def addMolecule(self, name, isotopeDepth=1, **abundance):
        molecule = Molecule(name, self, isotopeDepth, **abundance)
        self.append(molecule)
        self.progressCrossSection = False
        if totalConcentration(self) > 1:
            print("**Warning : Concentrations exceed 1.")
        if not molecule.exotic:
            molecule.getData()
        return molecule

    def returnCopy(self):
        new = Layer(self.depth, self.T, self.P, self.rangeMin, self.rangeMax, self.atmosphere,
                    name=self.atmosphere.nextLayerName(), dynamicResolution=self.dynamicResolution)
        for m in self:
            new.append(m.returnCopy())
        return new

    def returnMoleculeObjects(self):
        return list(self)

    def planck(self, temperature):
        axis = _eng.linspace_axis(self.rangeMin, self.rangeMax, _n_base(self))
        return engine().planck(axis, temperature)


class Atmosphere(list):
    def __init__(self, name):
        list.__init__(self)
        self.name = name

    def __str__(self):
        return self.name

    def __bool__(self):
        return True

    def addLayer(self, depth, T, P, rangeMin, rangeMax, name=None, dynamicResolution=True):
        layer = Layer(depth, T, P, rangeMin, rangeMax, atmosphere=self, name=name or self.nextLayerName(),
                      dynamicResolution=dynamicResolution)
        self.append(layer)
        return layer

    def nextLayerName(self):
        return "Layer %s" % (len(self) + 1)

    def returnLayerNames(self):
        return [l.name for l in self]

    def returnLayerObjects(self):
        return list(self)

    def transmission(self, surfaceSpectrum):
        """Fold of Layer.transmission bottom -> top over the layers in list order (the multi-layer path the
        reference's README announces but does not ship, SURVEY.md 3.5)."""
        spectrum = np.asarray(surfaceSpectrum, dtype=np.float64)
        for layer in self:
            spectrum = layer.transmission(spectrum)
        return spectrum

    def columnSpectrum(self, surfaceTemperature, continuum=None):
        """The whole column on the device in ONE engine call (prb_atmosphere): K1 for every layer, the batched line
        sums, and the fold  I <- T_l I + (1 - T_l) B(nu, T_l)  starting from I_0 = B(nu, surfaceTemperature).
        Returns (radiance, total transmittance) on the layers' common grid.  Same physics as ``transmission`` above,
        without one host round trip per layer and isotope; needs layers that share range and base resolution and carry
        the same line-by-line molecules in the same order.  xsc molecules (up to eight distinct tables over the column)
        stay resident on the device and enter every layer's k(nu) inside the line-sum kernel (prb_xsc_resident).
        continuum: None, or a water-vapour continuum table in MT_CKD's form for this call (Engine.set_continuum: a dict
        with nu, self, foreign, texp and optional t_ref, p_ref); its mole fraction in a layer is the summed concentration
        of the layer's line-by-line H2O (HITRAN id 1), 0 without one.  The continuum is an extension of the column path:
        ``transmission``, getTransmittance(layer) and Layer.transmission stay the reference's physics, without it.  The
        default gives the result described above, bit for bit."""
        return self._column(surfaceTemperature, lambda e: e.atmosphere_read(), continuum)

    def columnFluxes(self, surfaceTemperature, mu=None, weights=None, bands=None, surfaceEmissivity=None,
                     reflection="lambertian", topTemperature=0.0, solarIrradiance=None, solarMu=1.0, continuum=None):
        """Hemispheric fluxes, heating rates and slant radiances of the column (prb_atmosphere, then
        prb_atmosphere_fluxes on its device-resident k matrix; same requirements on the layers as columnSpectrum).
        For every node mu_i of the angular quadrature (default: 3-node Gauss-Legendre on [0, 1]; at most 4 nodes) the
        fold runs up from B(nu, surfaceTemperature) and down from 0 (by default no cosmic background, no sun) with
        T = exp(-k_l depth_l / mu_i); level j is the boundary below layer j (0 = surface, len(self) = top), and
        F[j] = 2 pi sum_i w_i mu_i integrateSpectrum(I_i(level j), 1, res).  A column with opaque bands is not
        isotropic, so F_up at the top differs from the pi x nadir radiance of integrateSpectrum(columnSpectrum(...)[0]).
        Returns a dict: flux_up, flux_down, net (= up - down) per level in W m-2; heating_rate per layer in K/day
        (heatingRate); rad_up_top and rad_down_surface, float32 (n_mu, n_points) -- the radiance leaving the top and
        reaching the surface along every mu_i; mu and weights.
        bands: optional band edges in cm-1 (1-d, at least 2, finite, strictly ascending); a grid point nu belongs to band
        b when bands[b] <= nu < bands[b+1] (prb_atmosphere_band_fluxes, on the same column run).  The dict then also holds
        band_edges, band_flux_up and band_flux_down (n_bands, L+1), band_net, and band_heating_rate (n_bands, L): each
        band's heating rate by heatingRate.
        surfaceEmissivity, reflection, topTemperature: the column's boundaries for this call (Engine.set_flux_boundaries).
        surfaceEmissivity is None (black), a scalar, or a pair (nu, eps) of 1-d arrays interpolated onto the grid (np.interp);
        the surface then emits eps B(nu, surfaceTemperature) and reflects 1 - eps of the downward radiance, diffusely
        ("lambertian") or along the same mu ("specular").  topTemperature > 0 sends B(nu, topTemperature) down from the top
        (2.725 for the cosmic background).
        solarIrradiance, solarMu: the Sun for this call (Engine.set_solar_source).  solarIrradiance is None (no Sun) or a
        pair (nu, S) of 1-d arrays, S the irradiance at the top in W m-2 (cm-1)-1 normal to the beam, interpolated onto
        the grid (np.interp, 0 outside the table); solarMu is the cosine of the solar zenith angle, in (0, 1].  The beam is
        absorbed on its way down and 1 - eps of it is reflected as the surface says; flux_down, net, heating_rate and the
        band arrays then include it (and flux_up its reflection).  The sunlight's share of any of them is the result with
        the Sun minus the result without it: the column is linear in its sources.
        continuum: a water-vapour continuum in the column's k matrix for this call, as in columnSpectrum.
        The defaults give the result described above, bit for bit."""
        _eng.flux_boundary_args(surfaceEmissivity, reflection, topTemperature)      # ValueError before the column runs
        _eng.solar_source_args(solarIrradiance, solarMu)
        if mu is None and weights is None:
            x, w = np.polynomial.legendre.leggauss(3)
            mu, weights = (x + 1) / 2, w / 2
        mu, weights = np.atleast_1d(np.asarray(mu, dtype=np.float64)), np.atleast_1d(np.asarray(weights, dtype=np.float64))
        if mu.shape != weights.shape or not 1 <= mu.size <= 4:
            raise ValueError("columnFluxes needs 1 to 4 quadrature nodes, as many weights as mu")
        if bands is not None:
            bands = np.asarray(bands, dtype=np.float64)
            if bands.ndim != 1 or bands.size < 2 or not np.all(np.isfinite(bands)) or not np.all(np.diff(bands) > 0):
                raise ValueError("columnFluxes: bands must be a 1-d array of at least 2 finite, strictly ascending edges")

        def result(e):
            e.set_flux_boundaries(surfaceEmissivity, reflection, topTemperature)
            try:
                e.set_solar_source(solarIrradiance, solarMu)
                return (e.atmosphere_fluxes(mu, weights, rows=True),
                        e.atmosphere_band_fluxes(mu, weights, bands) if bands is not None else None)
            finally:
                e.set_solar_source()
                e.set_flux_boundaries()

        (up, down, ru, rd), band = self._column(surfaceTemperature, result, continuum)
        layers = list(self)
        depth, T, P = [l.depth for l in layers], [l.T for l in layers], [l.P for l in layers]
        out = {"flux_up": up, "flux_down": down, "net": up - down, "heating_rate": heatingRate(up, down, depth, T, P),
               "rad_up_top": ru, "rad_down_surface": rd, "mu": mu, "weights": weights}
        if band is not None:
            bu, bd = band
            out.update(band_edges=bands, band_flux_up=bu, band_flux_down=bd, band_net=bu - bd,
                       band_heating_rate=np.array([heatingRate(u, d, depth, T, P) for u, d in zip(bu, bd)]))
        return out

    def _column(self, surfaceTemperature, result, continuum=None):
        """Run the column on the device (prb_atmosphere) and return result(engine) while its state is in place."""
        layers = list(self)
        if not layers:
            raise ValueError("atmosphere has no layers")
        # the continuum's gas is the layers' line-by-line H2O (HITRAN id 1); ValueError before the column runs
        h2o = [sum(m.concentration for m in l if not m.exotic and m.ID == 1) for l in layers] if continuum is not None \
            else None
        _eng.continuum_args(continuum, h2o)
        ref = layers[0]
        for l in layers:
            if (l.rangeMin, l.rangeMax) != (ref.rangeMin, ref.rangeMax) or l.resolution != BASE_RESOLUTION:
                raise ValueError("columnSpectrum needs layers on one grid at the base resolution "
                                 "(build them with dynamicResolution=False)")
            if [iso.globalIsoNumber for m in l if not m.exotic for iso in m] != \
                    [iso.globalIsoNumber for m in ref if not m.exotic for iso in m]:
                raise ValueError("columnSpectrum needs the same line-by-line isotopologues in every layer")
        # xsc tables of the column, in order of first appearance; a layer without a table carries it at mole fraction 0
        tables = {}
        for l in layers:
            for m in l:
                if m.exotic:
                    tables.setdefault(m._xsc_key, m)
        if len(tables) > 8:
            raise ValueError("columnSpectrum carries at most eight distinct xsc tables")
        # line source: the layer that read the widest wavenumber range from the data tree; every layer then takes part
        # with the lines of its OWN effective range only, as its getData kept them (prb_set_layer_line_range)
        widest = max(layers, key=lambda l: l.effectiveRangeMax - l.effectiveRangeMin)
        if any(l.effectiveRangeMin < widest.effectiveRangeMin or l.effectiveRangeMax > widest.effectiveRangeMax for l in layers):
            raise ValueError("columnSpectrum needs one layer whose loaded line range covers every other layer's")
        isos = [iso for m in widest if not m.exotic for iso in m]
        cols = {k: np.concatenate([iso._cols[k] for iso in isos]) if isos else np.zeros(0)
                for k in ("nu", "sw", "gamma_air", "gamma_self", "elower", "n_air", "delta_air")}
        group = np.concatenate([np.full(len(iso._cols["nu"]), g, dtype=np.int32) for g, iso in enumerate(isos)]) \
            if isos else np.zeros(0, dtype=np.int32)
        order = np.argsort(cols["nu"], kind="stable")
        lines = {k: np.ascontiguousarray(v[order]) for k, v in cols.items()}
        lines["group"] = np.ascontiguousarray(group[order])
        n = _n_base(ref)
        global _RESIDENT_KEY
        _RESIDENT_KEY = None
        e = engine()
        e.upload_lines(lines, n_groups=max(len(isos), 1))
        e.set_grid(ref.rangeMin, BASE_RESOLUTION, n)
        conc = [[m.concentration for m in l if not m.exotic for _ in m] for l in layers]
        q_t = [[iso.q[l.T] for m in l if not m.exotic for iso in m] for l in layers]   # KeyError on a non-tabulated T
        window = [_eng.window_len(l.distanceFromCenter, BASE_RESOLUTION) for l in layers]
        e.xsc_clear()
        try:
            for slot, m in enumerate(tables.values()):
                e.xsc_resident(slot, **m._xsc_plan)
            if tables:
                # several molecules of one table in a layer add up, like their absCoef terms do
                e.set_xsc_conc([[sum(m.concentration for m in l if m.exotic and m._xsc_key == key) for key in tables]
                                for l in layers])
            if not isos:                                           # xsc molecules only: an empty line list
                conc, q_t = [[0.0]] * len(layers), [[1.0]] * len(layers)
            if any((l.effectiveRangeMin, l.effectiveRangeMax) != (widest.effectiveRangeMin, widest.effectiveRangeMax)
                   for l in layers):
                e.set_layer_line_range([l.effectiveRangeMin for l in layers], [l.effectiveRangeMax for l in layers])
            e.set_continuum(continuum, h2o)
            e.atmosphere([l.depth for l in layers], [l.T for l in layers], [l.P for l in layers], conc,
                         [iso.molmass for iso in isos] or [1.0], q_t, [iso.q296 for iso in isos] or [1.0], window,
                         surfaceTemperature, ref.rangeMax)
            return result(e)
        finally:
            e.xsc_clear()
            e.set_layer_line_range()
            e.set_continuum()


#: dry air: molar mass (kg/mol), isobaric specific heat (J kg-1 K-1); molar gas constant (J mol-1 K-1, CODATA 2018 exact)
M_DRY_AIR = 0.0289647
CP_DRY_AIR = 1004.64
R_GAS = 8.314462618


def heatingRate(flux_up, flux_down, depth_cm, T, P):
    """Radiative heating rate of every layer in K/day from the level fluxes (L+1 values, level 0 = surface, W m-2):
    Q_l = -(F_net[l+1] - F_net[l]) / (rho_l c_p dz_l) * 86400 s/day with F_net = F_up - F_down, the layer's thickness
    dz_l = depth_cm / 100 m and its density rho_l = 100 P_l M_d / (R T_l) (ideal dry air; P in hPa as Layer holds it,
    T in K).  Constants: M_DRY_AIR, CP_DRY_AIR, R_GAS above.  Negative values are cooling."""
    net = np.asarray(flux_up, dtype=np.float64) - np.asarray(flux_down, dtype=np.float64)
    T, P = np.asarray(T, dtype=np.float64), np.asarray(P, dtype=np.float64)
    dz = np.asarray(depth_cm, dtype=np.float64) / 100
    if net.shape != (T.size + 1,) or T.shape != P.shape or dz.shape != T.shape:
        raise ValueError("heatingRate needs L+1 level fluxes and L depths, temperatures and pressures")
    rho = 100 * P * M_DRY_AIR / (R_GAS * T)
    return -(net[1:] - net[:-1]) / (rho * CP_DRY_AIR * dz) * 86400


def getGlobalIsotope(ID, isotopeDepth):
    return [HITRAN_GLOBAL_ISO[ID][i] for i in range(1, isotopeDepth + 1)]


def returnPlot(obj, propertyToPlot):
    if propertyToPlot == "transmittance":
        return getTransmittance(obj), 1
    if propertyToPlot == "absorption coefficient":
        return getAbsCoef(obj), 0
    if propertyToPlot == "cross section":
        return getCrossSection(obj), 0
    if propertyToPlot == "absorbance":
        return getAbsorbance(obj), 0
    if propertyToPlot == "optical depth":
        return getOpticalDepth(obj), 0
    if propertyToPlot == "line survey":
        return obj.lineSurvey, 0
    return False


# the reference's id tables (pyradClasses.py:951-1022), all 49 molecules
from .hitran_tables import HITRAN_GLOBAL_ISO, MOLECULE_ID  # noqa: E402
