"""Drop-in check of SURVEY.md 8(b): the reference's OWN Cython binding (python/py_corona_sim.pyx), compiled unchanged and
in place against this repository's observation_fit facade (oracle/build_pyx.py -> oracle/_ref/py_corona_sim/, module name
py_corona_sim_gpu as the reference's CUDA build), must build, expose every method of Pyobservation_fit, and -- on the
GPU -- give the numbers of the facade's C handles.  Built where B200RT_REFERENCE names the reference's source tree;
otherwise a module built before is used."""
import glob
import importlib
import os
import sys

import numpy as np
import pytest

from util import rel_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("B200RT_REFERENCE")     # the reference's source tree, where one is at hand
OUT = os.path.join(ROOT, "oracle", "_ref", "py_corona_sim")
PKG = "3d_planetary_rt_model_b200"

METHODS = """add_observation set_g_factor simulate_iph add_observation_ra_dec lc_from_T eff_from_T generate_source_function
generate_source_function_lc generate_source_function_effv generate_source_function_variable_thermosphere
generate_source_function_nH_asym generate_source_function_temp_asym generate_source_function_temp_asym_full
generate_source_function_tabular_atmosphere set_use_CO2_absorption set_use_temp_dependent_sH set_sza_method_uniform
set_sza_method_uniform_cos reset_H_lya_xsec_coef reset_H_lyb_xsec_coef reset_CO2_lya_xsec reset_CO2_lyb_xsec
get_CO2_exobase_density reset_CO2_exobase_density set_CO2_exobase_density save_influence_matrix
save_influence_matrix_O_1026 set_H_density_tweak set_H_density_tweak_values set_H_temp_tweak set_H_temp_tweak_values
brightness species_col_dens tau_species_final tau_absorber_final iph_brightness_observed iph_brightness_unextincted
D_brightness D_col_dens tau_D_final O_1026_generate_source_function O_1026_brightness
lyman_multiplet_generate_source_function lyman_multiplet_brightness lyman_singlet_generate_source_function
lyman_singlet_brightness corona_model_git_hash""".split()


@pytest.fixture(scope="module")
def module():
    if REF and os.path.exists(os.path.join(REF, "python", "py_corona_sim.pyx")):
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import build_pyx
        build_pyx.build(verbose=False)
    if not glob.glob(os.path.join(OUT, "py_corona_sim_gpu*.so")):
        pytest.skip("oracle/_ref/py_corona_sim not built (needs B200RT_REFERENCE; python oracle/build_pyx.py)")
    if OUT not in sys.path:
        sys.path.insert(0, OUT)
    return importlib.import_module("py_corona_sim_gpu")


def test_reference_binding_builds_against_the_facade(module):
    cls = module.Pyobservation_fit
    missing = [m for m in METHODS if not hasattr(cls, m)]
    assert not missing, missing
    assert module.Pyobservation_fit.corona_model_git_hash().startswith("b200rt-")
    assert os.path.exists(os.path.join(OUT, module.iph_sfn_basename))


@pytest.mark.gpu
def test_reference_binding_runs_on_the_device(module):
    synth = importlib.import_module(PKG + ".synth")
    hb = importlib.import_module(PKG + ".host_binding")
    locs, dirs = synth.random_los(300)
    P = module.Pyobservation_fit()
    P.add_observation(locs, dirs)
    P.generate_source_function(5e5, 200.0)
    b = np.array(P.brightness())
    F = hb.Pyobservation_fit(os.path.join(OUT, module.iph_sfn_basename))
    F.add_observation(locs, dirs)
    F.generate_source_function(5e5, 200.0)
    assert b.shape == (2, 300) and rel_err(b, F.brightness(), floor=1e-300) < 1e-12   # two runs: equal to rounding (atomics)
    assert rel_err(np.array(P.species_col_dens()), F.species_col_dens(), floor=1e-300) < 1e-12
    assert abs(P.lc_from_T(200.0) - F.lc_from_T(200.0)) < 1e-12
    # the IPH path through the real table the binding locates next to the module
    ra, dec = synth.random_sky(300)
    P.add_observation_ra_dec(np.array(synth.MARS_ECLIPTIC_POS), ra, dec)
    F.add_observation_ra_dec(synth.MARS_ECLIPTIC_POS, ra, dec)
    assert np.array_equal(np.array(P.iph_brightness_unextincted()), F.iph_brightness_unextincted())
    assert rel_err(np.array(P.brightness()), F.brightness(), floor=1e-300) < 1e-12
    # one call of every other model through the binding
    P.generate_source_function(5e5, 200.0, deuterium=True)
    F.generate_source_function(5e5, 200.0, deuterium=True)
    assert rel_err(np.array(P.D_brightness()), F.D_brightness(), floor=1e-300) < 1e-12
    P.O_1026_generate_source_function(2e7, 200.0, 1.69e-3)
    assert np.array(P.O_1026_brightness()).shape == (6, 300)
    P.lyman_multiplet_generate_source_function(5e5, 200.0)
    assert np.array(P.lyman_multiplet_brightness()).shape == (2, 300)
    d = P.get_example_tabular_atmosphere()
    alt = np.linspace(80.0, 50000.0, 200)
    d.update(alt_nH=alt, log_nH=np.log(1e6 * np.exp(-(alt - 80.0) / 800.0)), alt_nCO2=alt,
             log_nCO2=np.log(1e13 * np.exp(-(alt - 80.0) / 12.0) + 1e-30), alt_Temp=alt, Temp=np.full_like(alt, 200.0))
    P.generate_source_function_tabular_atmosphere(d)
    assert np.isfinite(np.array(P.brightness())).all()
