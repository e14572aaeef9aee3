"""The reference's own RT_grid, with its GPU members bound to libb200rt.so (SURVEY.md section 8(b): the drop-in seam).

integration/RT_b200.hpp defines RT_grid::RT_to_device / generate_S_gpu / brightness_gpu / emissions_influence_to_host
(declared at RT_grid.hpp:31-39,146,219,325; defined by the reference only in RT_gpu.cu:8-84,138-192,255-309) on top of
the C ABI.  oracle/Makefile (ref_b200) compiles it with the host compiler against the reference's headers, in place.
Here the reference's objects run both ways -- the CPU members the reference ships and the *_gpu members through the
binding -- and must agree within the bars of BASELINE.json (1e-6 double Real, 1e-4 float Real)."""
import numpy as np
import pytest

from util import TOL, TOL_AUX, UNDERFLOW, rel_err

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("shape,n_em", [((12, 8, 5, 6), 2), ((20, 12, 6, 8), 1)])
def test_reference_gpu_members_match_its_cpu_members(synth, prec, shape, n_em):
    from oracle import refbind
    if not refbind.available(prec, "b200"):
        pytest.skip("oracle/_ref/libref_b200_*.so not built (needs B200RT_REFERENCE at build time)")
    tol = TOL[prec]
    scn = synth.make_scenario(*shape, n_em=n_em, sza_T_contrast=0.1)
    cpu = refbind.RefModel(scn, prec, variant="b200")
    gpu = refbind.RefModel(scn, prec, variant="b200")
    cpu.generate_S()                       # RT_grid::generate_S (RT_grid.hpp:150-218)
    gpu.generate_S_gpu()                   # RT_grid::generate_S_gpu through integration/RT_b200.hpp
    gpu.influence_to_host()
    for e in range(n_em):
        a, b = cpu.vectors(e), gpu.vectors(e)
        for k in ("S0", "tau_species_ss", "tau_absorber_ss"):
            assert rel_err(a[k], b[k], floor=UNDERFLOW[prec]) < tol, k
        floor = 1e-30 if prec == "f64" else float(np.abs(a["S"]).max())
        assert rel_err(a["S"], b["S"], floor=floor) < tol
        Ka, Kb = cpu.K(e), gpu.K(e)
        kf = 1e-290 if prec == "f64" else 1e-30
        Ka, Kb = np.where(np.abs(Ka) > kf, Ka, 0.0), np.where(np.abs(Kb) > kf, Kb, 0.0)
        assert rel_err(Ka, Kb) < tol
        gpu.set_sourcefn(e, a["S"])        # same source function for the brightness comparison
    locs, dirs = synth.random_los(600, seed=4)
    _, bc = cpu.brightness(locs, dirs, 10)           # RT_grid::brightness (RT_grid.hpp:233-318)
    # a solved reference object that has never been on the device: brightness_gpu uploads tables + S itself
    fresh = refbind.RefModel(scn, prec, variant="b200")
    for e in range(n_em):
        fresh.set_sourcefn(e, cpu.vectors(e)["S"])
    bg = fresh.brightness_gpu(locs, dirs, 10)        # RT_grid::brightness_gpu through the binding
    for q in range(4):
        assert rel_err(bc[:, q], bg[:, q], floor=1e-300) < (tol if q == 0 else TOL_AUX[prec]), q
