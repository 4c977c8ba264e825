"""The host mirror keeps the reference's call signatures for the hot path (SURVEY.md §8b): every positional parameter of
the reference, same name, same order; ours may only append keyword extras.  The reference's signatures were parsed from its
sources (not imported) into tests/golden/reference_interface.json by tests/golden/make_golden.py --case reference_interface."""
import inspect
import json
import os

import pytest

from tardis_b200 import montecarlo as mc
from tardis_b200 import formal_integral as fim
from tardis_b200 import source_function as sfm
from tardis_b200 import spectrum as spm

with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_interface.json")) as _f:
    REF = json.load(_f)


def ours(obj):
    return [n for n, p in inspect.signature(obj).parameters.items()
            if n != "self" and p.kind in (p.POSITIONAL_ONLY, p.POSITIONAL_OR_KEYWORD)]


@pytest.mark.parametrize("ref_file,ref_name,mirror", [
    ("montecarlo_transport.py", "montecarlo_transport_with_vpackets", mc.montecarlo_transport_with_vpackets),
    ("iip/montecarlo_transport.py", "montecarlo_transport", mc.montecarlo_transport),
    ("classic/solver.py", "MCTransportSolverClassic.__init__", mc.MCTransportSolverB200.__init__),
    ("classic/solver.py", "MCTransportSolverClassic.from_config", mc.MCTransportSolverB200.from_config),
    ("classic/solver.py", "MCTransportSolverClassic.initialize_transport_state", mc.MCTransportSolverB200.initialize_transport_state),
    ("classic/solver.py", "MCTransportSolverClassic.run", mc.MCTransportSolverB200.run),
    ("iip/solver.py", "MCTransportSolverIIP.__init__", mc.MCTransportSolverB200IIP.__init__),
    ("iip/solver.py", "MCTransportSolverIIP.from_config", mc.MCTransportSolverB200IIP.from_config),
    ("iip/solver.py", "MCTransportSolverIIP.initialize_transport_state", mc.MCTransportSolverB200IIP.initialize_transport_state),
    ("iip/solver.py", "MCTransportSolverIIP.run", mc.MCTransportSolverB200IIP.run),
    ("../estimators/mc_rad_field_solver.py", "MCRadiationFieldPropertiesSolver.__init__", mc.MCRadiationFieldPropertiesSolverB200.__init__),
    ("../estimators/mc_rad_field_solver.py", "MCRadiationFieldPropertiesSolver.solve", mc.MCRadiationFieldPropertiesSolverB200.solve),
    ("../../../spectrum/formal_integral/source_function.py", "SourceFunctionSolver.__init__", sfm.SourceFunctionSolverB200.__init__),
    ("../../../spectrum/formal_integral/source_function.py", "SourceFunctionSolver.solve", sfm.SourceFunctionSolverB200.solve),
    ("../../../spectrum/formal_integral/formal_integral_solver.py", "FormalIntegralSolver.__init__", fim.FormalIntegralSolverB200.__init__),
    ("../../../spectrum/formal_integral/formal_integral_solver.py", "FormalIntegralSolver.solve", fim.FormalIntegralSolverB200.solve),
    ("../../../spectrum/formal_integral/base.py", "check_formal_integral_requirements", fim.check_formal_integral_requirements),
    ("../../../spectrum/base.py", "SpectrumSolver.__init__", spm.SpectrumSolverB200.__init__),
    ("../../../spectrum/base.py", "SpectrumSolver.setup_optional_spectra", spm.SpectrumSolverB200.setup_optional_spectra),
    ("../../../spectrum/base.py", "SpectrumSolver.solve", spm.SpectrumSolverB200.solve),
    ("../../../spectrum/base.py", "SpectrumSolver.from_config", spm.SpectrumSolverB200.from_config),
    ("../../../spectrum/spectrum.py", "TARDISSpectrum.__init__", spm.TARDISSpectrumB200.__init__),
])
def test_mirror_keeps_reference_parameters(ref_file, ref_name, mirror):
    ref = REF["signatures"][ref_file][ref_name]
    mine = ours(mirror)
    assert mine[:len(ref)] == ref, (ref_name, ref, mine)


def test_spectrum_solver_mirror_has_the_reference_s_properties():
    """every property / attribute list of SpectrumSolver (spectrum/base.py:14-202) exists on the mirror under the same name"""
    props = REF["spectrum_solver"]["properties"]
    assert len(props) >= 8
    for name in props:
        assert isinstance(getattr(spm.SpectrumSolverB200, name), property), name
    assert spm.SpectrumSolverB200.hdf_properties == REF["spectrum_solver"]["hdf_properties"] and spm.SpectrumSolverB200.hdf_name == "spectrum"
