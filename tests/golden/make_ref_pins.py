"""Write tests/golden/ref_pins.json and ref_pins_S.npz: what the comparisons with the reference's own source compared
against (see tests/ref_pins.py).  With the reference built (oracle/_ref, oracle/Makefile `ref`) the values come from it; without it
they come from the oracle, which those same comparisons hold bit for bit to the reference build (the source functions
to 1e-7: two different LUs).  The file records which one wrote it.
    python tests/golden/make_ref_pins.py"""
import importlib
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE)]
synth = importlib.import_module("3d_planetary_rt_model_b200.synth")
hb = importlib.import_module("3d_planetary_rt_model_b200.host_binding")
import ref_pins as P  # noqa: E402
from oracle import multbind, oraclebind, refbind  # noqa: E402


def main():
    use_ref = refbind.available("f64") and refbind.available("f32") and multbind.ref_available("f64") \
        and multbind.ref_available("f32")
    Model = refbind.RefModel if use_ref else oraclebind.OracleModel
    Mult = multbind.RefMultiplet if use_ref else multbind.OracleMultiplet
    pins = P.Pins("reference build (oracle/_ref)" if use_ref else "oracle (oracle/rt_oracle.c)")
    for prec in ("f64", "f32"):
        for shape in P.SINGLET_SHAPES:
            out, S, _ = P.singlet_case(synth, Model(synth.make_scenario(*shape, n_em=2, sza_T_contrast=0.1), prec))
            pins.store(f"singlet_{'x'.join(map(str, shape))}_{prec}", out, S)
        for shape in P.PP_SHAPES:
            out, S, _ = P.pp_case(Model(synth.make_scenario_pp(*shape, n_em=2), prec))
            pins.store(f"pp_{'x'.join(map(str, shape))}_{prec}", out, S)
        for kind in P.MULT_KINDS:
            for shape in P.MULT_SHAPES:
                scn = synth.make_multiplet_scenario(kind, *shape, sza_T_contrast=0.1)
                out, S, _ = P.mult_case(synth, Mult(scn, prec))
                pins.store(f"mult{kind}_{'x'.join(map(str, shape))}_{prec}", out, [S])
    out, S = P.grid_D_case(synth, Model(synth.make_scenario(40, 20, 7, 12, n_em=2), "f64"))
    pins.store("singlet_D", out, S)
    scn = synth.make_scenario(12, 8, 5, 6, n_em=1)
    rb = refbind.RefModel(scn, "f64", rmethod_inject=False).grid()["radial_boundaries"] if use_ref else scn.rb
    pins.store("rmethod_altitude", {"radial_boundaries": rb})
    pins.store("mult0_D", P.mult_grid_D_case(synth, Mult(synth.make_multiplet_scenario(0, 40, 20, 7, 12))))
    for shape, n_em in P.FILE_CASES:
        scn = synth.make_scenario(*shape, n_em=n_em, sza_T_contrast=0.1)
        pins.store(f"file_{'x'.join(map(str, shape))}_{n_em}", P.file_case(scn, Model(scn, "f64"), hb))
    pins.save()
    print("wrote", P.DIGESTS, "and", P.SOURCEFNS, "from the", pins.source)


if __name__ == "__main__":
    main()
