"""Experiment orchestration, B200 version -- drop-in for the reference's Experiment.py.

Same class surface (Experiment.py:25-607): constructor keys, attributes, return tuples, error
messages and the report file.  The per-energy image-formation loops
(``computeSampleAndReferenceImages_RT`` / ``_Fresnel``) run on the GPU through
``paresis_b200.engine.ImageFormation``; only detector images return to the host.

Extensions read from ``exp_dict`` when present (the reference ignores unknown keys):
``poissonNoise`` (bool, default True), ``seed`` (int, default wall clock like Detector.py:113),
``returnDisplacement`` (bool, default True: Dx/Dy of point 0 are copied back), ``resultDtype`` ("float64" as
upstream, or "float32": counts are exact in float32 and cross PCIe at half the size -- what main.py saves anyway),
``membraneAhead`` (bool, default True: the next position's membrane map is cut and copied speculatively while this
position's images travel; see geometry.speculate_next_membrane).
"""
import time

import numpy as np

import _paresis_path  # noqa: F401
from Detector import Detector
from Sample import AnalyticalSample
from Source import Source
from getk import getk
from refractionFileNumba2 import fastRefraction, fastRefractionDF
from usefullScripts.getSamplingFactor import is_overSampling_ok
import torch

from paresis_b200 import darkfield, engine, geometry, host_api, hostmath, transfer
from paresis_b200.hostio import xmlparams


class Experiment:
    def __init__(self, exp_dict):
        """Experiment.py:26-137.

        Args:
            exp_dict (dict): experimentName, filepath, overSampling (int), nbExpPoints,
                simulation_type ("RayT" | "Fresnel"), expID.
        """
        self.xmlExperimentFileName = "xmlFiles/Experiment.xml"
        self.name = exp_dict['experimentName']
        self.exp_dict = exp_dict
        exp_dict.update({'studyPixelSize': 0., 'studyDimensions': (0., 0.), 'inVacuum': False, 'meanShotCount': 0,
                         'meanEnergy': 0, 'distSourceToMembrane': 0, 'distMembraneToObject': 0,
                         'distObjectToDetector': 0,
                         'studyPixelSize_unit': "um", 'studyDimensions_unit': "pixels", 'meanEnergy_unit': "keV",
                         'distSourceToMembrane_unit': "m", 'distMembraneToObject_unit': "m",
                         'distObjectToDetector_unit': "m"})
        self.mySampleofInterest = None
        self.mySampleType = ""
        self.myDetector = None
        self.mySource = None
        self.myMembrane = None
        self.myPlate = None
        self.myAirVolume = None
        self.Dxreal = []
        self.Dyreal = []
        self.imageSampleBeforeDetection = []
        self.imageReferenceBeforeDetection = []
        self.imagePropagBeforeDetection = []
        self._engine = None

        self.defineCorrectValues(exp_dict)
        self.myDetector.defineCorrectValuesDetector()
        self.mySource.defineCorrectValuesSource()
        self.mySampleofInterest.defineCorrectValuesSample()
        self.myAirVolume.defineCorrectValuesSample()
        d = self.exp_dict
        self.myAirVolume.myThickness = (d['distSourceToMembrane'] + d['distObjectToDetector'] + d['distMembraneToObject']) * 1e6
        if self.myPlate is not None:
            self.myPlate.defineCorrectValuesSample()
        self.myMembrane.defineCorrectValuesSample()

        d['magnification'] = (d['distSourceToMembrane'] + d['distObjectToDetector'] + d['distMembraneToObject']) / \
                             (d['distSourceToMembrane'] + d['distMembraneToObject'])
        self.getStudyDimensions()

        self.mySource.setMySpectrum(self.myDetector.det_param["photonCounting"])
        spectrum = self.mySource.mySpectrum
        for obj in (self.myAirVolume, self.myPlate, self.mySampleofInterest):
            if obj is not None:
                obj.getDeltaBeta(spectrum)
                obj.getMyGeometry(d['studyDimensions'], d['studyPixelSize'], d['overSampling'])
        self.myMembrane.getDeltaBeta(spectrum)
        self.myMembrane.membranePixelSize = d['studyPixelSize'] * d['distSourceToMembrane'] / \
                                            (d['distSourceToMembrane'] + d['distMembraneToObject'])
        if self.myDetector.det_param['myScintillatorMaterial'] is not None:
            self.myDetector.getBeta(spectrum)
            self.myDetector.getSpectralEfficiency()

        if d['simulation_type'] == "RayT" and d["overSampling"] < 2:
            print(f'/!\\/!\\ OVERSAMPLING FACTOR < MIN OVERSAMPLING FOR RAY-T MODEL: {d["overSampling"]} < 2')
        if d['simulation_type'] == "Fresnel":
            src = self.mySource.source_dict
            check_e = spectrum[-1][0] / 2 if src["myType"] == "Polychromatic" else src["Energy"]
            is_overSampling_ok(d, self.myDetector.det_param['myPixelSize'], check_e)
        self._banner()

    def _banner(self):
        d, det, src = self.exp_dict, self.myDetector, self.mySource.source_dict
        print('\nCurrent experiment:', self.name)
        print(f'  Experiment in Vacuum: {d["inVacuum"]}')
        print("  Magnification :", d['magnification'])
        print(f'  Study dimensions: {d["studyDimensions"]} pixels')
        print("  Sample pixel size =", d["studyPixelSize"], "um")
        print("  Over-overSampling factor: ", d["overSampling"])
        print("\nCurrent detector: ", det.myName)
        print(f'  Detector pixel size: {det.det_param["myPixelSize"]} um')
        if det.det_param['myScintillatorMaterial'] is not None:
            print(f'  Scintillator {det.det_param["myScintillatorMaterial"]} of {det.det_param["myScintillatorThickness"]}um')
        print("  Detectors dimensions: ", det.det_param["myDimensions"])
        print("\nCurrent source: ", self.mySource.myName)
        print("  Source type:", src["myType"])
        if src["myType"] == 'Monochromatic':
            print(f'Energy: {src["Energy"]} keV')
        else:
            if "myVoltage" in src:
                print(f'Source voltage: {src["myVoltage"]} kVp')
            if "myTargetMaterial" in src:
                print(f'Anode material: {src["myTargetMaterial"]}')
            if src.get("filterMaterial") is not None:
                print(f'filter: {src["filterMaterial"]} of {src["filterThickness"]} mm')
        print("\nCurrent sample:", self.mySampleofInterest.myName)
        print("\nCurrent membrane:", self.myMembrane.myName)

    def defineCorrectValues(self, exp_dict):
        """Experiment.py:140-197.

        Raises:
            Exception: sample type not defined.
            ValueError: experiment not found in xml file.
        """
        self.mySource = Source()
        self.myDetector = Detector(exp_dict)
        entry = xmlparams.find_entry(self.xmlExperimentFileName, "experiment", self.name)
        if entry is None:
            raise ValueError("experiment not found in xml file")
        d = self.exp_dict
        d['distSourceToMembrane'] = entry.get("distSourceToMembrane", float)
        d['distMembraneToObject'] = entry.get("distMembraneToObject", float)
        d['distObjectToDetector'] = entry.get("distObjectToDetector", float)
        d['meanShotCount'] = entry.get("meanShotCount", float)
        if entry.has("inVacuum"):
            d['inVacuum'] = entry.get("inVacuum") == "True"
        if entry.has("plateName"):
            self.myPlate = AnalyticalSample()
            self.myPlate.myName = entry.get("plateName")
        self.myAirVolume = AnalyticalSample()
        self.myAirVolume.myName = "air_volume"
        self.mySampleType = entry.get("sampleType")
        if self.mySampleType != "AnalyticalSample":
            raise Exception("sample type not defined")
        self.mySampleofInterest = AnalyticalSample()
        self.myMembrane = AnalyticalSample()
        self.myMembrane.myName = entry.get("membraneName")
        self.mySampleofInterest.myName = entry.get("sampleName")
        self.myDetector.myName = entry.get("detectorName")
        self.mySource.myName = entry.get("sourceName")

    def getText(self, node):
        return xmlparams.text_of(node)

    def getStudyDimensions(self):
        """Study grid = detector grid x oversampling; pixel size in the sample plane (Experiment.py:204-216)."""
        d, det = self.exp_dict, self.myDetector.det_param
        self.precision = det["myPixelSize"] / d['overSampling'] / d['distObjectToDetector']
        d['studyDimensions'] = det["myDimensions"] * int(d['overSampling'])
        d['studyDimensions'][0] = int(d['studyDimensions'][0])
        d['studyDimensions'][1] = int(d['studyDimensions'][1])
        d['studyPixelSize'] = det["myPixelSize"] / d['overSampling'] / d['magnification']

    # ------------------------------------------------------------------ stand-alone pieces
    def wavePropagation(self, waveToPropagate, propagationDistance, Energy, magnification):
        """Fresnel propagation of a complex field (Experiment.py:219-252)."""
        return host_api.wave_propagation(waveToPropagate, propagationDistance, Energy, magnification,
                                         self.exp_dict['studyDimensions'], self.exp_dict['studyPixelSize'])

    def refraction(self, intensityRefracted, phi, propagationDistance, Energy, magnification, darkField=0):
        """Ray-tracing propagation of an intensity map (Experiment.py:255-277)."""
        if type(darkField) == int or type(darkField) == float:
            return fastRefraction(intensityRefracted, phi, propagationDistance, Energy, magnification,
                                  self.exp_dict["studyPixelSize"])
        return fastRefractionDF(intensityRefracted, phi, propagationDistance, Energy, magnification,
                                self.exp_dict["studyPixelSize"], darkField)

    # ------------------------------------------------------------------ the hot path
    def _open_bins(self, pointNum):
        """Experiment.py:296-301 / :425-430: validate the detector bins, close the last one (in place)."""
        spectrum = self.mySource.mySpectrum
        thr = self.myDetector.det_param["myBinsThersholds"]
        if pointNum == 0:
            if any(t < spectrum[0][0] for t in thr) or any(t > spectrum[-1][0] for t in thr):
                raise Exception(f'At least one of your detector bin threshold is outside your source spectrum. \n'
                                f'Your source spectrum ranges from {spectrum[0][0]} to {spectrum[-1][0]}')
            thr.append(spectrum[-1][0])
        return thr

    @staticmethod
    def _lookup(pairs):
        return {e: v for e, v in pairs}

    def _layers(self, obj, materialise):
        geom = obj._device_geometry()
        entries = geom.device_entries(materialise=materialise)
        models = [darkfield.model_of(obj, m) for m in range(len(entries))]      # Sample.py:322-343
        return [engine.Layer(t, self._lookup(obj.delta[m]), self._lookup(obj.beta[m]),
                             hostmath.MODELS[models[m]] if models[m] is not None else None) for m, t in enumerate(entries)]

    def _uniform_attenuation(self, obj, energy):
        """exp(-2 k beta t) of an object made of uniform layers (air volume, plate: Sample.py:239-243, :347)."""
        geom = obj._device_geometry()
        k = getk(energy * 1000)
        arg = 0.0
        for m, t in enumerate(geom.entries):
            if not isinstance(t, float):
                t = float(np.asarray(geom[m]).flat[0])
            arg += 2 * k * self._lookup(obj.beta[m]).get(energy, 0.0) * t
        return float(np.exp(-arg))

    def _membrane_layers_per_position(self):
        """The segmented membrane as a batched scene sees it: the grain map is rasterised per position by
        the library (engine.PER_POSITION), the support plate is a uniform layer (getMembraneFromFile.py:168)."""
        mem = self.myMembrane
        entries = [engine.PER_POSITION, mem.myPMMAThickness * 1e-6]
        return [engine.Layer(t, self._lookup(mem.delta[m]), self._lookup(mem.beta[m])) for m, t in enumerate(entries)]

    def _scene(self, thresholds, per_position_membrane=False):
        d, det, src = self.exp_dict, self.myDetector, self.mySource

        def common(energy):
            f = 1.0
            if not d['inVacuum']:
                f *= self._uniform_attenuation(self.myAirVolume, energy)            # Experiment.py:452-453
            if det.det_param['myScintillatorMaterial'] is not None:
                if d['simulation_type'] == "RayT":
                    for e, eff in det.mySpectralEfficiency:                            # :456-459
                        if e == energy:
                            f *= eff
                else:
                    beta = dict(det.beta)[energy]                                      # :326-333
                    f *= 1 - np.exp(-2 * getk(energy * 1000) * det.det_param['myScintillatorThickness'] * 1e-6 * beta)
            return f

        plate = (lambda e: self._uniform_attenuation(self.myPlate, e)) if self.myPlate is not None else None
        return engine.Scene(
            d['studyDimensions'], d['studyPixelSize'], d['overSampling'], det.det_param['myDimensions'],
            det.det_param['myPixelSize'], det.det_param['myPSF'], d['distSourceToMembrane'], d['distMembraneToObject'],
            d['distObjectToDetector'], d['meanShotCount'], src.mySpectrum, src.source_dict["mySize"],
            src.source_dict["myEnergySampling"], thresholds,
            self._membrane_layers_per_position() if per_position_membrane else self._layers(self.myMembrane, materialise=False),
            self._layers(self.mySampleofInterest, materialise=True),
            common_factor=common, plate_factor=plate)

    def _get_engine(self):
        if self._engine is None:
            d, det = self.exp_dict, self.myDetector
            self._engine = engine.ImageFormation(d['studyDimensions'], d['overSampling'], det.det_param['myDimensions'],
                                                 seed=det.seed, poisson=det.poissonNoise)
        return self._engine

    def _membrane_ahead(self, pointNum=None):
        """Start the next position's membrane map while this position's images travel (geometry.speculate_next_membrane)."""
        mem = self.myMembrane
        if getattr(mem, "myGeometryFunction", "") == "getMembraneSegmentedFromFile" and self.exp_dict.get("membraneAhead", True):
            d = self.exp_dict
            geometry.speculate_next_membrane(mem, d['studyDimensions'][0], d['studyDimensions'][1], mem.membranePixelSize,
                                             mem.myPMMAThickness)

    def _finish(self, res, scene=None, ahead=False):
        """Device images -> the float64 [nbins, dimX, dimY] arrays the reference returns; images that were
        not computed (propagation / white beyond point 0) are zeros, as upstream (Experiment.py:433-434)."""
        dtype = torch.float32 if str(self.exp_dict.get("resultDtype", "float64")) == "float32" else torch.float64
        images = transfer.Pending(res["_stack"], dtype)            # one cast + one PCIe copy for all images
        if "aux" in res:
            # deferred bookkeeping: the per-energy sums and the status flag ride behind the images
            aux = transfer.Pending(res["aux"])
            if ahead:
                self._membrane_ahead()                             # queued behind the images and the sums: the link does not idle
            host = images.wait()
            num, den = self._get_engine().finish_deferred(scene, aux.wait())
        else:
            host = images.wait()
            num, den = res["mean_energy"]
        self.exp_dict['meanEnergy'] = (self.exp_dict['meanEnergy'] + num) / den      # Experiment.py:486, :523
        out = [host[i] for i in range(host.shape[0])]
        while len(out) < 4:
            out.append(self._zeros(out[0].shape))
        return out

    def _zeros(self, shape):
        """All-zero result images are shared, read-only arrays (allocating 8-32 MB of zeros per call costs
        more than the GPU work of a position)."""
        cache = self.__dict__.setdefault("_zero_cache", {})
        if shape not in cache:
            z = np.zeros(shape)
            z.setflags(write=False)
            cache[shape] = z
        return cache[shape]

    def computeSampleAndReferenceImages_Fresnel(self, pointNum):
        """All images of one membrane position with the Fresnel propagator (Experiment.py:279-405).

        Returns:
            SampleImage, ReferenceImage, PropagImage, detectedWhite: float64 arrays [nbins, dimX, dimY].
        """
        thresholds = self._open_bins(pointNum)
        for energy, _ in self.mySource.mySpectrum:
            print("Current Energy:", energy)
        res = self._get_engine().compute_fresnel(self._scene(thresholds), pointNum)
        out = self._finish(res)
        print("Mean energy detected in reference image", self.exp_dict['meanEnergy'])
        return tuple(out)

    def computeSampleAndReferenceImages_RT(self, pointNum):
        """All images of one membrane position with the ray-tracing model (Experiment.py:407-526).

        Returns:
            SampleImage, ReferenceImage, PropagImage, detectedWhite: float64 arrays [nbins, dimX, dimY],
            Dxreal, Dyreal: displacement maps of the sample-only beam, zero-padded by 15 (from point 0),
            darkFieldPropag: [N, N] dark-field map (zeros unless the sample has a dark-field model).
        """
        thresholds = self._open_bins(pointNum)
        for energy, _ in self.mySource.mySpectrum:
            print("Current Energy: %gkev" % energy)
        eng = self._get_engine()
        want_d = pointNum == 0 and bool(self.exp_dict.get("returnDisplacement", True))
        scene = self._scene(thresholds)
        try:
            res = eng.compute_rt(scene, pointNum, want_displacement=want_d, defer=True)
            out = self._finish(res, scene, ahead=True)
        except engine.InsaneValues as exc:
            raise Exception(str(exc))
        if want_d:
            self.Dxreal = transfer.fetch(eng.dx_pad, torch.float64)
            self.Dyreal = transfer.fetch(eng.dy_pad, torch.float64)
        if "dark_field" in res:
            self.darkFieldPropag = transfer.fetch(res["dark_field"], torch.float64)      # Experiment.py:491, from point 0
        elif not eng.scatters(scene):
            n = self.exp_dict['studyDimensions']
            self.darkFieldPropag = self._zeros((int(n[0]), int(n[1])))
        print("Mean detected energy in reference image", self.exp_dict['meanEnergy'])
        return out[0], out[1], out[2], out[3], self.Dxreal, self.Dyreal, self.darkFieldPropag

    # ------------------------------------------------------------------ report
    def saveAllParameters(self, time0, expDict):
        """Text report of all experiment and algorithm parameters (Experiment.py:530-607)."""
        fileName = expDict['filepath'] + self.name + '_' + str(expDict['expID']) + ".txt"
        print("file name: ", fileName)

        def block(fh, params):
            for key, value in params.items():
                if key.split('_')[-1] != 'unit':
                    unit = params.get(key + "_unit")
                    fh.write(f'\n    {key}: {value} {unit}' if unit is not None else f'\n    {key}: {value}')

        with open(fileName, "w+") as f:
            f.write("EXPERIMENT PARAMETERS - " + expDict['simulation_type'] + " - " + str(expDict['expID']))
            block(f, self.exp_dict)
            f.write("\n\nEntire computing time: %gs" % (time.time() - time0))
            f.write("\n\nSource parameters:")
            f.write("\nSource name: %s" % self.mySource.myName)
            block(f, self.mySource.source_dict)
            f.write("\n\nDetector parameters:")
            f.write("\nDetector name: %s" % self.myDetector.myName)
            block(f, self.myDetector.det_param)
            smp, mem = self.mySampleofInterest, self.myMembrane
            f.write("\n\nSample informations")
            f.write("\nSample name: %s" % smp.myName)
            f.write("\nSample type: %s" % self.mySampleType)
            f.write("\n    materials: %s" % smp.myMaterials)
            if smp.geom_parameters is not None:
                for key, value in smp.geom_parameters.items():
                    f.write(f'\n    {key}: {value[0]} {value[1]}')
            f.write("\n\nMembrane informations:")
            f.write("\nMembrane name: %s" % mem.myName)
            f.write("\nMembrane type: %s" % mem.myType)
            f.write("\n    materials: %s" % mem.myMaterials)
            f.write("\n    Membrane geometry function: %s" % mem.myGeometryFunction)
            if mem.geom_parameters is not None:
                # upstream lists the SAMPLE's geometry parameters under the membrane heading (Experiment.py:594-596
                # iterates mySampleofInterest.geom_parameters); kept, so that the report is the reference's line for line
                for key, value in (smp.geom_parameters or {}).items():
                    f.write(f'\n    {key}: {value[0]} {value[1]}')
            if mem.myGeometryFunction == "getMembraneFromFile":
                f.write("\nMembrane geometry file: %s" % mem.myMembraneFile)
            if self.myPlate is not None:
                f.write("\n\nDetectors protection Plate")
                f.write("Plate thickness: %s" % self.myPlate.myThickness)
                f.write("Plate Material: %s" % self.myPlate.myMaterials)
