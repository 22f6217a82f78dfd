"""Host side of the product (loader, synthesis, grids, stream twins, C-ABI surface) -- CPU only.
No compute entry point is exercised here beyond checking that it refuses to run without a GPU."""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import REFERENCE, ROOT

have_ref = os.path.isdir(REFERENCE)


def test_abi_exports_every_declared_symbol(Q):
    """The shared library loads and exports every function include/qo100net.h declares."""
    hdr = open(os.path.join(ROOT, "include", "qo100net.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(qo_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 38
    lib = ctypes.CDLL(Q.LIB_PATH)
    missing = [s for s in sorted(declared) if not hasattr(lib, s)]
    assert not missing, missing
    assert declared == set(Q.EXPORTS), declared ^ set(Q.EXPORTS)


def test_no_torch_types_or_oracle_in_product(Q):
    """The product never links, imports or calls the oracle (it must fail loudly instead of falling back)."""
    import subprocess
    out = subprocess.run(["ldd", Q.LIB_PATH], capture_output=True, text=True).stdout
    assert "qo100ref" not in out and "torch" not in out
    for dirpath, _d, files in os.walk(os.path.join(ROOT, "qo-100-tools_b200")):
        for fn in files:
            if fn.endswith((".py", ".c", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, fn), errors="replace").read()
                assert "refbind" not in src and "qo100ref" not in src, fn


@pytest.mark.skipif(__import__("torch").cuda.is_available(), reason="checks the no-GPU behaviour")
def test_compute_refuses_without_gpu(Q):
    with pytest.raises(Q.QoError) as ei:
        Q.Context(device=0)
    assert ei.value.status == Q.ERR_NO_DEVICE
    with pytest.raises(Q.QoError) as ei:
        Q.Context(ngpus=2)
    assert ei.value.status == Q.ERR_NO_DEVICE


def test_golden_networks_match_survey_tables(golden_nets):
    """Element lists the loader produced from the reference files == SURVEY §2 tables."""
    n = golden_nets["util/if-bandpass-filter/schematic.svg"]
    assert (n["rs"], n["rl"]) == (50.0, 50.0)
    assert [e[0] for e in n["elements"]] == [7, 10, 7]
    assert n["elements"][0][1][:2] == [33e-9, 4.7e-12] and n["elements"][1][1][:2] == [4.7e-9, 33e-12]
    n = golden_nets["util/gpsdo-ouput-filters/10M/schematic.svg"]
    assert (n["rs"], n["rl"]) == (100.0, 50.0)
    assert [e[1][0] for e in n["elements"]] == [430e-12, 1.3e-6, 620e-12, 1.3e-6, 560e-12, 1.1e-6, 240e-12]
    assert [e[0] for e in n["elements"]] == [6, 3, 6, 3, 6, 3, 6]
    n = golden_nets["docs/gpsdo-filters/15M.svg"]
    assert [e[0] for e in n["elements"]] == [3, 9, 3, 9, 3, 9, 3]
    assert n["elements"][1][1][:2] == [82e-9, 270e-12]
    n = golden_nets["docs/upconverter/upconverter-lol-filter.svg"]
    assert [e[0] for e in n["elements"]] == [4, 8, 4, 8, 4, 8, 4, 5]
    assert n["elements"][1][1][:2] == [12e-9, 1.2e-12] and n["elements"][7][1][0] == 1.5e-12
    assert "2.100 GHz" in n["title"]
    n = golden_nets["util/pa-lpf-simulation/pa-lpf-simulation.sch"]
    kinds = [e[0] for e in n["elements"]]
    assert kinds.count(14) == 19 and kinds.count(15) == 12 and kinds.count(16) == 2 and kinds.count(17) == 2 and kinds[0] == 13
    assert n["elements"][0][1] == [4.5, 0.6e-3, 34.79e-6, 0.045, 1.68e-8, 0.15e-6]
    assert n["sweep"] == ["lin", 1e7, 1e10, 5000]
    # SURVEY App. A.6 cascade: main-line lengths in mm, in order
    main, side, in_side = [], [], False
    for k, p in n["elements"][1:]:
        if k == 16:
            in_side = True
        elif k == 17:
            in_side = False
        elif k == 14:
            (side if in_side else main).append(round(p[1] * 1e3, 5))
    assert main == [1.65, 1.40415, 1.65, 1.40415, 0.95, 0.95, 2.5, 3.45, 1.55, 0.95, 0.95, 0.8, 1.6, 1.75, 5.95]
    assert side == [0.15, 4.35, 2.5, 3.0]
    t = golden_nets["util/directional-couplers/dir_cpl_2.4g_20dB.trc"]
    assert (t["z0e"], t["z0o"], t["ang"], t["f0"]) == (55.2771, 45.2267, 95.4225, 2.4e9)
    t = golden_nets["util/directional-couplers/dir_cpl_2.4g_35dB_pa_250W.trc"]
    assert (t["ht"], t["f0"], t["s"]) == (15e-3, 2.4e9, 4e-3)


@pytest.mark.skipif(not have_ref, reason="the upstream qo-100-tools files are not in this repository: set QO100_REFERENCE to a checkout")
def test_loader_reads_every_reference_file(Q, golden_nets):
    for key, g in golden_nets.items():
        path = os.path.join(REFERENCE, key)
        if key.endswith(".svg"):
            n = Q.Net.from_rftools_svg(path)
        elif key.endswith(".sch"):
            n = Q.Net.from_qucs_sch(path)
            assert list(Q.qucs_sch_sweep(path)) == g["sweep"]
        else:
            assert Q.load_trc(path) == g
            continue
        assert n.terminations == (g["rs"], g["rl"])
        assert [[k, p] for k, p in n.elements] == g["elements"]


def test_workload_networks_equal_loaded_ones(Q, W, golden_nets):
    """The hard-coded BASELINE workloads are the reference files' element lists."""
    assert [[k, p] for k, p in W.if_bpf_net().elements] == golden_nets["util/if-bandpass-filter/schematic.svg"]["elements"]
    assert [[k, p] for k, p in W.pa_lpf_net().elements] == golden_nets["util/pa-lpf-simulation/pa-lpf-simulation.sch"]["elements"]
    bank = {name: net for name, net, _fc in W.gpsdo_bank()}
    assert [[k, p] for k, p in bank["10M"].elements] == golden_nets["util/gpsdo-ouput-filters/10M/schematic.svg"]["elements"]
    for nm in ("15M", "40M", "60M"):
        assert [[k, p] for k, p in bank[nm].elements] == golden_nets["docs/gpsdo-filters/%s.svg" % nm]["elements"]


def test_loader_errors(Q, tmp_path):
    with pytest.raises(Q.QoError) as ei:
        Q.Net.from_rftools_svg(str(tmp_path / "missing.svg"))
    assert ei.value.status == Q.ERR_IO
    p = tmp_path / "bad.svg"
    p.write_text("<svg><defs></defs><use xlink:href=\"#q_branch_weird\"/></svg>")
    with pytest.raises(Q.QoError) as ei:
        Q.Net.from_rftools_svg(str(p))
    assert ei.value.status == Q.ERR_UNSUPPORTED
    p.write_text("<svg>nothing</svg>")
    with pytest.raises(Q.QoError) as ei:
        Q.Net.from_rftools_svg(str(p))
    assert ei.value.status == Q.ERR_PARSE
    p = tmp_path / "x.sch"
    p.write_text("hello")
    with pytest.raises(Q.QoError) as ei:
        Q.Net.from_qucs_sch(str(p))
    assert ei.value.status == Q.ERR_PARSE
    p = tmp_path / "x.trc"
    p.write_text("<Microstrip>\n</Microstrip>\n")
    with pytest.raises(Q.QoError):
        Q.load_trc(str(p))
    with pytest.raises(Q.QoError):
        Q.Net.from_elements([(99, [1.0])])
    with pytest.raises(Q.QoError):
        Q.Net.from_elements([(Q.MLIN, [1e-3, 1e-3])])              # microstrip without SUBST
    with pytest.raises(Q.QoError):
        Q.Net.from_elements([(Q.SUBST, [4.5, 1e-3, 0, 0, 0, 0]), (Q.MTEE, [1e-3] * 3)])   # side arm not closed
    with pytest.raises(Q.QoError):
        Q.Net.cheby_lpf(10, 0.1, 1e6)                               # even order needs unequal terminations


def test_small_svg_and_sch_round_trip(Q, tmp_path):
    """A minimal hand-written rf-tools export and Qucs schematic (the formats, not the reference files)."""
    svg = ('<svg><defs><symbol id="x"><use xlink:href="#l_branch_series"/></symbol></defs>'
           '<use xlink:href="#s_branch_voltage" x="0"/><use xlink:href="#r_branch_series"/>'
           '<use xlink:href="#c_branch_shunt"/><use xlink:href="#lc_branch_series_parallel"/>'
           '<use xlink:href="#l_branch_shunt_half"/><use xlink:href="#r_branch_shunt"/>'
           '<text x="1">RS</text><text>75.00 Ω</text><text>C1</text><text>10.00 pF</text>'
           '<text>C2</text><text>1.500 nF</text><text>L2</text><text>2.200 uH</text>'
           '<text>L3</text><text>47.00 mH</text><text>RL</text><text>1.000 kΩ</text>'
           '<text>rf-tools.com | today</text><text>Demo filter</text></svg>')
    p = tmp_path / "t.svg"
    p.write_text(svg, encoding="utf-8")
    n = Q.Net.from_rftools_svg(str(p))
    assert n.terminations == (75.0, 1000.0) and n.title == "Demo filter"
    assert [(k, pp[:2]) for k, pp in n.elements] == [(Q.SHUNT_C, [10e-12, 0.0]), (Q.SER_LC_PAR, [2.2e-6, 1.5e-9]), (Q.SHUNT_L, [47e-3, 0.0])]
    sch = """<Qucs Schematic 0.0.19>
<Components>
  <Pac P1 1 100 100 18 -26 0 1 "1" 1 "75 Ohm" 1>
  <GND * 1 100 130 0 0 0 0>
  <MLIN MS1 1 160 70 -26 15 0 0 "S1" 1 "w0" 1 "2 mm" 1>
  <MCORN MS2 1 220 70 -26 15 0 0 "S1" 1 "w0" 1>
  <MLIN MS3 1 220 130 15 -26 0 1 "S1" 1 "1 mm" 1 "3.5 mm" 1>
  <Pac P2 1 220 190 18 -26 0 1 "2" 1 "50 Ohm" 1>
  <GND * 1 220 220 0 0 0 0>
  <SUBST S1 1 0 0 0 0 0 0 "3.5" 1 "0.762 mm" 1 "35 um" 1 "0.0013" 1 "2.4e-8" 1 "0" 1>
  <.SP SP1 1 0 0 0 0 0 0 "log" 1 "1 MHz" 1 "2 GHz" 1 "201" 1>
  <Eqn Eqn1 1 0 0 0 0 0 0 "w0=1.5e-3" 1 "foo=dB(S[2,1])" 1 "yes" 0>
</Components>
<Wires>
  <100 70 130 70 "" 0 0 0 "">
</Wires>
"""
    p = tmp_path / "t.sch"
    p.write_text(sch)
    n = Q.Net.from_qucs_sch(str(p))
    assert n.terminations == (75.0, 50.0)
    el = n.elements
    assert [k for k, _ in el] == [Q.SUBST, Q.MLIN, Q.MCORN, Q.MLIN]
    assert el[0][1] == [3.5, 0.762e-3, 35e-6, 0.0013, 2.4e-8, 0.0]
    assert el[1][1][:2] == [1.5e-3, 2e-3] and el[2][1][0] == 1.5e-3 and el[3][1][:2] == [1e-3, 3.5e-3]
    assert Q.qucs_sch_sweep(str(p)) == ("log", 1e6, 2e9, 201)


def test_synthesis_matches_oracle(Q, R):
    for order in (3, 5, 7, 11):
        net = Q.Net.cheby_lpf(order, 0.1, 10e6, 50.0).add_parasitics(10e6)
        ref = R.elems_to_list(R.ladder_lpf(R.cheby_g(order, 0.1), 10e6, 50.0, True, (60, 30, 0.1, 50)))
        for (k1, p1), (k2, p2) in zip(net.elements, ref):
            assert k1 == k2 and np.allclose(p1, p2, rtol=4e-16, atol=0)
    net = Q.Net.butter_lpf(11, 3e9, 50.0, series_first=False)
    ref = R.elems_to_list(R.ladder_lpf(R.butter_g(11), 3e9, 50.0, False))
    assert [k for k, _ in net.elements] == [k for k, _ in ref] and net.elements[0][0] == Q.SHUNT_C
    assert np.allclose([p[0] for _, p in net.elements], [p[0] for _, p in ref], rtol=4e-16)
    a, b = Q.Net.cheby_lpf(3, 0.5, 1e6, 75.0), Q.Net.butter_lpf(2, 1e6, 50.0)
    c = a.concat(b)
    assert len(c) == 5 and c.terminations == (75.0, 50.0)


def test_grids_bit_exact(Q, R, golden_dat):
    assert np.array_equal(Q.grid_lin(1e7, 1e10, 5000), golden_dat["frequency"])
    assert np.array_equal(Q.grid_log(4e6, 62.5e6, 4096), R.grid_log(4e6, 62.5e6, 4096))
    assert np.array_equal(Q.grid_lin(70e6, 4000e6, 4096), R.grid_lin(70e6, 4000e6, 4096))
    assert abs(Q.grid_lin(70e6, 4000e6, 4096)[2428] - 2400168498.17) < 0.01      # SURVEY §8d cfg 5
    assert Q.grid_lin(5.0, 9.0, 1)[0] == 5.0


def test_host_stream_twin_bit_exact_vs_oracle(Q, R):
    """qo_philox4x32_10 / qo_variate / qo_perturb_factor (product host twins) == the oracle's C stream."""
    assert Q.philox([0, 0, 0, 0], [0, 0]) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert Q.philox([0xffffffff] * 4, [0xffffffff] * 2) == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert Q.philox([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0]) == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]
    rng = np.random.default_rng(5)
    for _ in range(5000):
        seed, s, v = int(rng.integers(0, 2 ** 63)) * 2 + 1, int(rng.integers(0, 2 ** 40)), int(rng.integers(0, 64))
        for dist in (0, 1):
            assert Q.variate(seed, s, v, dist) == R.lib().ref_variate(seed, s, v, dist)
            assert Q.perturb_factor(seed, s, v, dist, 0.05) == R.lib().ref_perturb_factor(seed, s, v, dist, 0.05)


def test_lc_tolerances_helper(Q, W):
    w = W.cfg2(1000, 64)
    assert len(w.tols) == 11 and [t[2] for t in w.tols] == list(range(11))
    assert [t[4] for t in w.tols] == [0.05, 0.02] * 5 + [0.05]
    w5 = W.cfg5(1000, 4096)
    assert len(w5.net) == 12 and max(t[2] for t in w5.tols) == 13 and len(w5.specs) == 3
    assert sum(1 for f in w5.f if 2.3e9 <= f <= 2.5e9) == 209 and sum(1 for f in w5.f if f >= 3.9e9) == 105


def test_cpl_analyze_reproduces_trc_files_and_oracle(Q, R, golden_nets):
    """Row N1: QucsTranscalc CoupledMicrostrip analysis.  The product's host routine reproduces
    Z0e, Z0o, Ang_l of all four util/directional-couplers/*.trc:18-20 to the files' 6 digits and agrees
    with the oracle's independent restatement to rounding; derived checks: coupling k and sqrt(Z0e Z0o)."""
    n = 0
    for key, t in golden_nets.items():
        if not key.endswith(".trc"):
            continue
        n += 1
        args = (t["w"], t["s"], t["h"], t["t"], t["er"], t["ht"], t["f0"], t["l"])
        ze, zo, ae, ao = Q.cpl_analyze(*args)
        assert abs(ze / t["z0e"] - 1) < 5e-6 and abs(zo / t["z0o"] - 1) < 5e-6
        assert abs(np.sqrt(ae * ao) / t["ang"] - 1) < 5e-6
        assert ae > ao                                   # even mode is slower (more field in the dielectric)
        assert np.allclose([ze, zo, ae, ao], R.cpl_analyze(*args), rtol=1e-12, atol=0)
    assert n == 4
    t = golden_nets["util/directional-couplers/dir_cpl_2.4g_20dB.trc"]
    ze, zo, _, _ = Q.cpl_analyze(t["w"], t["s"], t["h"], t["t"], t["er"], t["ht"], t["f0"], t["l"])
    assert abs(20 * np.log10((ze - zo) / (ze + zo)) + 20.0) < 1e-3 and abs(np.sqrt(ze * zo) - 50.0) < 1e-3
    # zero strip thickness is a valid input; bad geometry is refused
    assert all(np.isfinite(Q.cpl_analyze(1.7e-3, 1e-3, 0.762e-3, 0.0, 3.5, 0.2, 2.4e9, 20e-3)))
    with pytest.raises(Q.QoError):
        Q.cpl_analyze(-1.0, 1e-3, 0.762e-3, 35e-6, 3.5, 0.2, 2.4e9, 20e-3)
    with pytest.raises(Q.QoError):
        Q.cpl_analyze(1.7e-3, 1e-3, 0.762e-3, 35e-6, 1.0, 0.2, 2.4e9, 20e-3)


def test_cpl_synthesize_recovers_trc_geometry(Q, golden_nets):
    """Row N1, the other button of QucsTranscalc: electrical -> physical.  From the Z0e / Z0o / Ang_l lines of the four
    util/directional-couplers/*.trc:18-20 the synthesis recovers the W / S / L lines :15-17 to the files' print precision
    (the impedances are printed to 6 digits: S moves in its 6th digit), and analysis(synthesis(x)) == x to 1e-9."""
    n = 0
    for key, t in golden_nets.items():
        if not key.endswith(".trc"):
            continue
        n += 1
        w, s, l = Q.cpl_synthesize(t["z0e"], t["z0o"], t["ang"], t["h"], t["t"], t["er"], t["ht"], t["f0"])
        assert abs(w / t["w"] - 1) < 2e-5 and abs(s / t["s"] - 1) < 2e-5 and abs(l / t["l"] - 1) < 2e-5, key
        ze, zo, ae, ao = Q.cpl_analyze(w, s, t["h"], t["t"], t["er"], t["ht"], t["f0"], l)
        assert abs(ze / t["z0e"] - 1) < 1e-9 and abs(zo / t["z0o"] - 1) < 1e-9 and abs(np.sqrt(ae * ao) / t["ang"] - 1) < 1e-9
    assert n == 4
    # a 10 dB coupler on 0.762 mm RO4350-like substrate needs a gap the model still covers; a 3 dB one does not exist in microstrip
    w, s, l = Q.cpl_synthesize(69.37, 36.04, 90.0, 0.762e-3, 35e-6, 3.5, 0.2, 2.4e9)
    assert 0 < s < w and 15e-3 < l < 25e-3
    with pytest.raises(Q.QoError):
        Q.cpl_synthesize(120.7, 20.7, 90.0, 0.762e-3, 35e-6, 3.5, 0.2, 2.4e9)
    with pytest.raises(Q.QoError):
        Q.cpl_synthesize(45.0, 55.0, 90.0, 0.762e-3, 35e-6, 3.5, 0.2, 2.4e9)      # Z0e must exceed Z0o


def test_qucs_dataset_round_trip(Q, golden_dat, tmp_path):
    """Row N2: Qucs dataset writer/reader.  A dataset built from the golden arrays is written in the layout of
    util/pa-lpf-simulation/pa-lpf-simulation.dat and read back bit-exactly; with the reference tree mounted,
    read -> write reproduces the reference file byte for byte."""
    f = golden_dat["frequency"]
    names = {"S[1,1]": "S11", "S[1,2]": "S12", "S[2,1]": "S21", "S[2,2]": "S22"}
    d = Q.Dataset.from_sweep(f, golden_dat["S11"], golden_dat["S12"], golden_dat["S21"], golden_dat["S22"])
    assert [v[0] for v in d.variables()] == ["frequency", "S11_dB", "S21_dB", "S[1,1]", "S[1,2]", "S[2,1]", "S[2,2]"]
    assert d.variables()[3] == ("S[1,1]", "frequency", 5000, True) and d.variables()[0] == ("frequency", "", 5000, False)
    p = tmp_path / "out.dat"
    d.write(str(p))
    head = open(p).read().split("\n")[:3]
    assert head[0] == "<Qucs Dataset 0.0.19>" and head[1] == "<indep frequency 5000>" and head[2] == "  +1.00000000000000000000e+07"
    r = Q.Dataset.read(str(p))
    assert np.array_equal(r["frequency"], f)
    for k, g in names.items():
        assert np.array_equal(r[k], golden_dat[g])
    # dB traces recomputed by the writer agree with Qucs' own to rounding
    assert np.max(np.abs(r["S21_dB"] - golden_dat["S21_dB"])) < 1e-12
    assert np.max(np.abs(r["S11_dB"] - golden_dat["S11_dB"])) < 1e-11
    # generic builder + error paths
    e = Q.Dataset()
    e.add_indep("zw", [0.75e-3])
    e.add_indep("frequency", f[:7])
    e.add_dep("gain", "frequency", np.arange(7.0))
    e.add_dep("S[2,1]", "frequency", golden_dat["S21"][:7])
    with pytest.raises(Q.QoError):
        e.add_dep("bad", "frequency", np.arange(3.0))          # length mismatch
    with pytest.raises(Q.QoError):
        e.add_dep("gain", "frequency", np.arange(7.0))         # duplicate
    with pytest.raises(Q.QoError):
        e.add_dep("x", "nope", np.arange(7.0))                 # unknown independent
    e.write(str(tmp_path / "e.dat"))
    r2 = Q.Dataset.read(str(tmp_path / "e.dat"))
    assert r2.variables() == e.variables() and np.array_equal(r2["S[2,1]"], golden_dat["S21"][:7]) and r2["zw"][0] == 0.75e-3
    (tmp_path / "junk.dat").write_text("<Qucs Dataset 0.0.19>\n<indep f 2>\n  +1.0e+00\n</indep>\n")
    with pytest.raises(Q.QoError):
        Q.Dataset.read(str(tmp_path / "junk.dat"))             # fewer values than the header says
    with pytest.raises(Q.QoError):
        Q.Dataset.read(str(tmp_path / "missing.dat"))
    ref = os.path.join(REFERENCE, "util/pa-lpf-simulation/pa-lpf-simulation.dat")
    if have_ref:
        rd = Q.Dataset.read(ref)
        assert [v[0] for v in rd.variables()] == ["zw", "frequency", "S11_dB", "S21_dB", "S[1,1]", "S[1,2]", "S[2,1]", "S[2,2]"]
        assert np.array_equal(rd["S[2,1]"], golden_dat["S21"]) and np.array_equal(rd["S11_dB"], golden_dat["S11_dB"])
        rd.write(str(tmp_path / "ref_copy.dat"))
        assert open(tmp_path / "ref_copy.dat", "rb").read() == open(ref, "rb").read()


def test_touchstone_loader_interp_and_inductor_fit(Q, golden_s2p, tmp_path):
    """Row N3 (host side).  The Touchstone loader against an independent numpy parse of the reference's three
    .s2p files (tests/golden/touchstone.npz; read live too when the tree is mounted), spot values from the files,
    SPfile interpolation against a numpy restatement, and the inductor-model fit against the part values."""
    from conftest import np_spfile
    files = {"11SQ39N": "util/pa-bias-simulation/11SQ39N.S2P", "06HP47N": "util/preamp-bias-simulation/06HP47N.s2p",
             "pa_20W": "docs/pa-driver/pa_20W_vdd_32V_idq_180mA.s2p"}
    blocks = {}
    for key, rel in files.items():
        fd, sd, z0 = golden_s2p[key + "_f"], golden_s2p[key + "_s"], float(golden_s2p[key + "_z0"])
        b = Q.SBlock.from_arrays(fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], z0)
        blocks[key] = (b, fd, sd)
        path = os.path.join(REFERENCE, rel)
        if have_ref:
            live = Q.SBlock.load(path)
            f, s11, s21, s12, s22 = live.data()
            assert len(live) == len(fd) and live.z0 == z0 and np.array_equal(f, fd)
            assert np.allclose(np.stack([s11, s21, s12, s22], 1), sd, rtol=1e-14, atol=0)
    # 11SQ39N.S2P:6  " 10  0.0241890116 81.640573  0.996771193 -1.37700407 ..." (# MHZ S MA R 50 at :3)
    b, fd, sd = blocks["11SQ39N"]
    assert len(b) == 659 and fd[0] == 10e6 and fd[-1] == 3300e6
    assert abs(sd[0, 0] - 0.0241890116 * np.exp(1j * np.deg2rad(81.640573))) < 1e-15
    assert abs(sd[0, 1] - 0.996771193 * np.exp(1j * np.deg2rad(-1.37700407))) < 1e-15
    # pa_20W_vdd_32V_idq_180mA.s2p:8 (# HZ S RI R 50 at :5): 1e7 Hz, S11 = 1.00031 - j0.0752988, S21 = 0.00209503 - j1.33393e-05
    _, fd3, sd3 = blocks["pa_20W"]
    assert len(fd3) == 501 and fd3[0] == 1e7 and sd3[0, 0] == complex(1.00031, -0.0752988) and sd3[0, 1] == complex(0.00209503, -1.33393e-05)
    # interpolation: at the data points exact, between them == numpy restatement, outside: end segment extrapolated
    for polar in (True, False):
        fq = np.concatenate([fd[:5], np.sqrt(fd[:-1] * fd[1:])[::7], [1e3, 5e9]])
        got = np.stack(b.interp(fq, polar=polar), 1)
        assert np.allclose(got, np_spfile(fq, fd, sd, polar), rtol=1e-12, atol=1e-15)
        assert np.allclose(got[:5], sd[:5], rtol=1e-14)
        assert not np.allclose(got[-1], sd[-1], rtol=1e-3) and not np.allclose(got[-2], sd[0], rtol=1e-3)
    # inductor fits (SURVEY 8f N3: 1111SQ-39N 38.4-39.0 nH, SRF > 3.3 GHz; 0603HP-47N ~47 nH,
    # R 0.30 Ohm @ 1 MHz -> 2.9 Ohm @ 680 MHz, SRF 3.29-3.44 GHz)
    r = blocks["11SQ39N"][0].fit_inductor(10e6, 500e6)
    assert 38.3e-9 < r["L"] < 39.0e-9 and 3.2e9 < r["srf"] < 3.6e9 and r["rms_rel"] < 0.01 and 0.05 < r["r0"] < 0.3
    h = blocks["06HP47N"][0]
    r = h.fit_inductor(10e6, 500e6)
    assert 46.5e-9 < r["L"] < 48.0e-9 and r["rms_rel"] < 0.01
    assert 0.2 < r["r0"] + r["r1"] * 1e3 < 0.45 and 2.3 < r["r0"] + r["r1"] * np.sqrt(680e6) < 3.3
    r = h.fit_inductor(1e6, 6e9)                       # the resonance lies inside the data: SRF from the sign change of Im Y
    assert 3.29e9 < r["srf"] < 3.44e9 and r["cp"] > 0
    with pytest.raises(Q.QoError):
        blocks["pa_20W"][0].fit_inductor(1e7, 1e10)    # an amplifier is not a series inductor
    # loader error paths and formats (DB, GHz, comments, wrapped lines)
    (tmp_path / "a.s2p").write_text("! c\n# GHz S DB R 75\n1.0 -20 90 -0.5 -10\n -0.5 -10 -20 90 ! tail\n2.0 -20 45 -1 -20 -1 -20 -20 45\n")
    a = Q.SBlock.load(str(tmp_path / "a.s2p"))
    f, s11, s21, s12, s22 = a.data()
    assert a.z0 == 75 and list(f) == [1e9, 2e9] and abs(s11[0] - 0.1j) < 1e-15 and abs(abs(s21[1]) - 10 ** (-1 / 20)) < 1e-15
    for bad in ("# MHz Y MA R 50\n1 0 0 0 0 0 0 0 0\n", "# MHz S MA R 50\n1 0 0 0 0\n", "# MHz S MA R 50\n", "# MHz S MA R 50\n2 1 0 1 0 1 0 1 0\n1 1 0 1 0 1 0 1 0\n"):
        (tmp_path / "bad.s2p").write_text(bad)
        with pytest.raises(Q.QoError):
            Q.SBlock.load(str(tmp_path / "bad.s2p"))
    # a net with blocks: concat re-indexes, raw element lists cannot smuggle a block index in
    n1 = blocks["11SQ39N"][0].as_net(polar=True)
    n2 = blocks["06HP47N"][0].as_net(polar=False)
    cat = n1.concat(Q.Net.from_elements([(Q.SHUNT_C, [2.2e-12, 3.0, 0.0])], 50, 50)).concat(n2)
    assert [(k, p[:2]) for k, p in cat.elements] == [(Q.SBLOCK, [0.0, 1.0]), (Q.SHUNT_C, [2.2e-12, 3.0]), (Q.SBLOCK, [1.0, 0.0])]
    with pytest.raises(Q.QoError):
        Q.Net.from_elements([(Q.SBLOCK, [0.0, 1.0])], 50, 50)


def test_physical_coupled_line_element_validation(Q):
    sub, cpl = (Q.SUBST, [3.5, 0.762e-3, 35e-6, 0, 0, 0]), (Q.CPL_MS, [1.69e-3, 0.99e-3, 20e-3, 0.2, 2.4e9, 50.0])
    n = Q.Net.from_elements([sub, cpl, (Q.SER_L, [1e-9, 0.1, 0.0])], 50, 50)
    assert [k for k, _ in n.elements] == [Q.SUBST, Q.CPL_MS, Q.SER_L]
    for bad in ([cpl], [sub, cpl, cpl], [sub, (Q.CPL_MS, [1.69e-3, -1.0, 20e-3, 0.2, 2.4e9, 50.0])]):
        with pytest.raises(Q.QoError):
            Q.Net.from_elements(bad, 50, 50)


def test_transfer_function_plan_analysis(Q, W, monkeypatch):
    """Host-only part of plan creation (qo_plan_analyze, no GPU): which jobs take the transfer-function kernel, the
    polynomial lengths the grid needs, the denominator form, and the self-check of the expansion against the
    per-element evaluation (<= 1e-10 on |den|^2; north_star asks 1e-9)."""
    for v in ("QO100NET_KERNEL", "QO100NET_TF_TOL", "QO100NET_TF_TRUNC", "QO100NET_TF_NO_FRONT"):
        monkeypatch.delenv(v, raising=False)
    w = W.cfg2()
    a = Q.plan_analyze(w.net, w.f, w.specs, w.tols, **w.hist)
    assert a["selected"] and a["reason"] == "ok" and a["numerator_chains"] == 2 and a["den_form"] == "E" and a["degree"] == 22
    assert a["kn"] < 12 and a["kd"] <= 16 and a["kd"] % 2 == 0      # the parasitic-order terms the grid cannot see are dropped
    assert a["self_check_err"] < 1e-11
    again = Q.plan_analyze(w.net, w.f, w.specs, w.tols, **w.hist)       # served from the analysis cache
    assert {k: v for k, v in again.items() if k != "seconds"} == {k: v for k, v in a.items() if k != "seconds"}
    monkeypatch.setenv("QO100NET_TF_TRUNC", "0")                     # keep every coefficient
    full = Q.plan_analyze(w.net, w.f, w.specs, w.tols, **w.hist)
    assert full["selected"] and full["kn"] == 12 and full["self_check_err"] < 1e-11
    monkeypatch.delenv("QO100NET_TF_TRUNC")
    w5 = W.cfg5()
    a5 = Q.plan_analyze(w5.net, w5.f, w5.specs, w5.tols, **w5.hist)
    assert a5["selected"] and a5["numerator_chains"] == 4 and a5["den_form"] == "E" and a5["kn"] <= a["kn"]   # grid ends at 1.33 fc
    # ideal ladder: no denominator at all; elliptic filter with traps resonating inside the grid: complex-D form
    ideal = Q.Net.cheby_lpf(11, 0.1, 10e6, 50.0, True)
    ai = Q.plan_analyze(ideal, w.f, w.specs, Q.lc_tolerances(ideal, 0.05, 0.02))
    assert ai["selected"] and ai["den_form"] == "none" and ai["degree"] == 11 and ai["kn"] == 6
    _, ell, fc = W.gpsdo_bank()[1]
    f = Q.grid_log(fc / 2.5, fc * 6.25, 1024)
    ae = Q.plan_analyze(ell, f, [(Q.SPEC_S21_MIN_DB, 0.0, 0.8 * fc, -1.0)], Q.lc_tolerances(ell, 0.05, 0.05))
    assert ae["selected"] and ae["den_form"] in ("D", "E") and ae["kn"] == 4 and ae["degree"] == 10   # 7th-order numerator inside a structural degree of 10
    f4 = Q.grid_log(fc / 2.5, fc * 6.25, 4096)                            # a grid point 1e-4 from a notch: E(y) loses digits there, D takes over
    assert Q.plan_analyze(ell, f4, [(Q.SPEC_S21_MIN_DB, 0.0, 0.8 * fc, -1.0), (Q.SPEC_S21_MAX_DB, 2.0 * fc, 1e99, -30.0)],
                          Q.lc_tolerances(ell, 0.05, 0.05))["den_form"] == "D"
    # jobs that stay on the chain kernels, with the reason
    a11 = Q.plan_analyze(w.net, w.f, [(Q.SPEC_S11_MAX_DB, 0.0, 8e6, -8.0)], w.tols)
    assert a11["selected"] and a11["numerator_chains"] == 4 and a11["den_form"] == "none"      # S11 = (P - Rs Q)/(P + Rs Q): denominators cancel
    a511 = Q.plan_analyze(w5.net, w5.f, [(Q.SPEC_S11_MAX_DB, 2.3e9, 2.5e9, -10.0)], w5.tols)          # |S11| behind the coupler: two row vectors of the block
    assert a511["selected"] and a511["numerator_chains"] == 4 and a511["den_form"] == "none"
    agd = Q.plan_analyze(w.net, w.f, [(Q.SPEC_GD_MAX, 0.0, 8e6, 1e-6), (Q.SPEC_S21_MIN_DB, 0.0, 9.5e6, -2.0)], w.tols)
    assert agd["selected"] and agd["den_form"] == "DD" and agd["kn"] == 12 and agd["self_check_err"] < 1e-10   # derivative polynomials: nothing dropped
    assert Q.plan_analyze(w.net, w.f, [(Q.SPEC_GD_MAX, 0.0, 8e6, 1e-6), (Q.SPEC_S11_MAX_DB, 0.0, 8e6, -8.0)], w.tols)["reason"] == \
        "group-delay specs mixed with a front block or |S11| specs"
    # a transmission line in FRONT of the ladder keeps the polynomial route (4 chains, row vector per point); inside the cascade it does not
    el = w.net.elements
    front = Q.Net.from_elements([(Q.TLINE, [75.0, 35.0, 10e6])] + el, 50.0, 50.0)
    af = Q.plan_analyze(front, w.f, w.specs, [(e + 1, p_, v, m, t) for (e, p_, v, m, t) in w.tols] + [(0, 0, 30, Q.TOL_REL, 0.05)])
    assert af["selected"] and af["numerator_chains"] == 4 and af["kn"] == a["kn"]
    monkeypatch.setenv("QO100NET_TF_NO_FRONT", "1")
    assert Q.plan_analyze(front, w.f, w.specs, [])["reason"] == "non-lumped element"
    monkeypatch.delenv("QO100NET_TF_NO_FRONT")
    inside = Q.Net.from_elements(el[:4] + [(Q.TLINE, [75.0, 35.0, 10e6])] + el[4:], 50.0, 50.0)
    assert Q.plan_analyze(inside, w.f, w.specs, [])["reason"] == "non-lumped element"
    assert Q.plan_analyze(w.net, w.f, w.specs, w.tols, precision=32)["reason"] == "not a reduce-only FP64 job on a lumped cascade"
    assert Q.plan_analyze(w.net, w.f, w.specs, w.tols, precision=32)["selected"] is False
    assert Q.plan_analyze(w.net, w.f, [], w.tols, mode=Q.MODE_FULL_S)["selected"] is False
    tl = Q.Net.from_elements(w.net.elements + [(Q.TLINE, [50.0, 90.0, 1e9])], 50.0, 50.0)       # a line at the load end
    assert Q.plan_analyze(tl, w.f, w.specs)["reason"] == "non-lumped element"
    assert Q.plan_analyze(W.pa_lpf_net(), w.f, w.specs)["selected"] is False
    monkeypatch.setenv("QO100NET_TF_TOL", "1e-16")
    assert Q.plan_analyze(w.net, w.f, w.specs, w.tols, **w.hist)["reason"] == "polynomial expansion is too ill-conditioned on this grid"
    monkeypatch.delenv("QO100NET_TF_TOL")
    monkeypatch.setenv("QO100NET_KERNEL", "ladder")
    assert Q.plan_analyze(w.net, w.f, w.specs, w.tols, **w.hist)["reason"] == "QO100NET_KERNEL override"
    monkeypatch.delenv("QO100NET_KERNEL")
    # a grid three decades wide: a 22nd-degree monomial basis cannot hold 1e-10 there -- the plan must notice
    wide = Q.plan_analyze(w.net, Q.grid_log(1e4, 1e9, 2048), [(Q.SPEC_S21_MIN_DB, 0.0, 1e9, -300.0)], w.tols)
    assert (not wide["selected"]) or wide["self_check_err"] <= 1e-10


def test_element_parameters_are_validated(Q):
    """Non-positive or non-finite L, C, Z0, f0 ... are refused when the network is built (they would only surface as inf / NaN
    on the device), with the element named in the error text."""
    ok = [(Q.SER_L, [1e-6, 0.1, 1e-13]), (Q.SHUNT_C, [1e-9, 0.05, 1e-10]), (Q.SER_R, [0.0]), (Q.TLINE, [50.0, 90.0, 1e9]),
          (Q.CPL_THRU, [55.0, 45.0, 90.0, 90.0, 1e9, 50.0])]
    Q.Net.from_elements(ok, 50.0, 50.0)
    bad = [(Q.SER_L, [0.0]), (Q.SER_L, [-1e-9]), (Q.SHUNT_C, [float("nan")]), (Q.SHUNT_C, [1e-9, -0.1]), (Q.SHUNT_R, [0.0]),
           (Q.SER_LC_SER, [1e-9, 0.0]), (Q.TLINE, [50.0, 90.0, 0.0]), (Q.TLINE, [float("inf"), 90.0, 1e9]),
           (Q.CPL_THRU, [55.0, -45.0, 90.0, 90.0, 1e9, 50.0]), (Q.CPL_THRU, [55.0, 45.0, 90.0, 90.0, 1e9, float("nan")])]
    for el in bad:
        with pytest.raises(Q.QoError) as ei:
            Q.Net.from_elements([ok[0], el], 50.0, 50.0)
        assert ei.value.status == Q.ERR_ARG and "element 1" in str(ei.value)
    with pytest.raises(Q.QoError):
        Q.Net.from_elements(ok, float("inf"), 50.0)


def test_plan_analysis_rejects_unknown_mode_and_precision(Q, W):
    w = W.cfg2(10, 64)
    assert Q.plan_analyze(w.net, w.f, w.specs, w.tols)["reason"] == "ok"
    assert Q.plan_analyze(w.net, w.f, w.specs, w.tols, mode=7)["reason"] == "network does not compile"
    assert "mode" in Q.lib().qo_last_error().decode()
    assert Q.plan_analyze(w.net, w.f, w.specs, w.tols, precision=16)["reason"] == "network does not compile"
    assert "precision" in Q.lib().qo_last_error().decode()


def test_integration_md_c_samples_compile_and_link(Q, tmp_path):
    """The C samples of INTEGRATION.md are real programs: extract them, compile them with the system C compiler against
    include/qo100net.h (-Wall -Werror: a drifted prototype or struct field fails here, not only in ctypes), link them against
    libqo100net.so and run them.  Without a GPU they must stop at the documented QO_ERR_NO_DEVICE path; with one they run."""
    import re
    import shutil
    import subprocess
    cc = shutil.which("gcc", path="/usr/bin") or shutil.which("gcc") or shutil.which("cc")
    if not cc:
        pytest.skip("no C compiler")
    md = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    blocks = re.findall(r"```c\n(.*?)```", md, flags=re.S)
    assert len(blocks) >= 2
    resim = next(b for b in blocks if "int main(void)" in b)
    frag = next(b for b in blocks if "qo_net_cheby_lpf" in b and "int main" not in b)
    # the yield fragment becomes a function body around which the declarations it assumes are supplied
    prog2 = ("#include <stdio.h>\n#include <stdlib.h>\n#include <stdint.h>\n#include \"qo100net.h\"\n"
             "int main(void)\n{\n    qo_ctx *ctx = NULL; double *f = malloc(4096 * sizeof *f);\n"
             "    qo_grid_log(10e6 / 2.5, 10e6 * 6.25, 4096, f);\n"
             "    if (qo_ctx_create(1, &ctx)) { fprintf(stderr, \"%s\\n\", qo_last_error()); return 3; }\n" + frag +
             "    printf(\"%llu %llu\\n\", (unsigned long long)res.n_pass, (unsigned long long)res.n_total);\n"
             "    qo_ctx_destroy(ctx); qo_net_free(net); free(f);\n    return 0;\n}\n")
    bias = next(b for b in blocks if "qo_nodal_jit_analyze" in b)
    prog3 = bias + "int main(void) { qo_ctx *ctx = NULL; if (qo_ctx_create(1, &ctx)) { fprintf(stderr, \"%s\\n\", qo_last_error()); return 3; } return bias_yield(ctx); }\n"
    libdir = os.path.dirname(Q.LIB_PATH)
    for name, src in (("resim", resim), ("yield", prog2), ("bias", prog3)):
        c = tmp_path / (name + ".c")
        c.write_text(src)
        exe = tmp_path / name
        r = subprocess.run([cc, "-std=gnu11", "-Wall", "-Werror", "-Wno-unused-value", str(c), "-I", os.path.join(ROOT, "include"), "-L", libdir,
                            "-Wl,-rpath," + libdir, "-lqo100net", "-lm", "-o", str(exe)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    # resim.c wants the reference schematic in its working directory: run it where it is not -> the loader's I/O error path
    r = subprocess.run([str(tmp_path / "resim")], cwd=str(tmp_path), capture_output=True, text=True)
    assert r.returncode == 1 and "pa-lpf-simulation.sch" in r.stderr
    import torch
    r = subprocess.run([str(tmp_path / "yield")], cwd=str(tmp_path), capture_output=True, text=True, timeout=300)
    if torch.cuda.is_available():
        assert r.returncode == 0 and r.stdout.split()[1] == "1000000"
    else:
        assert r.returncode == 3 and "CUDA" in r.stderr          # no device, no fallback


def test_chain_kernel_generator_compiles_without_gpu(Q, W, tmp_path, monkeypatch):
    """qo_chain_jit_analyze (host only: NVRTC compiles without a GPU): cascades the polynomial kernels cannot take -- a line inside
    the ladder, a coupler in front written out in full (dir_cpl_2.4g_20dB.trc:18-20), every lumped opcode of the rf-tools filters,
    group delay next to |S11| -- folded into the chain kernel's source and compiled for sm_100a.  The generated text carries one
    literal qo_chain_step per element and no opcode table; the cubin lands in QO100NET_CACHE_DIR and is found again."""
    w5 = W.cfg5(1000)
    a = Q.chain_jit_analyze(w5.net, w5.f, w5.specs, w5.tols, **w5.hist)
    if not a["compiled"] and "libnvrtc" in (a["error"] or ""):
        pytest.skip("libnvrtc is not loadable here: %s" % a["error"])
    assert a["compiled"] and a["cubin_bytes"] > 10000, a
    assert a["registers"] in (-1,) or 32 <= a["registers"] <= 128          # __launch_bounds__(256, 2); -1: NVRTC did not echo ptxas
    dump = tmp_path / "chain.cu"
    monkeypatch.setenv("QO100NET_CHAIN_JIT_DUMP", str(dump))
    monkeypatch.setenv("QO100NET_CACHE_DIR", str(tmp_path / "cache"))
    fs = Q.chain_jit_analyze(w5.net, w5.f[:500], [], w5.tols, mode=Q.MODE_FULL_S)
    assert fs["compiled"], fs["error"]
    src = dump.read_text()
    n_el = len(w5.net)
    assert src.count("qo_chain_step<T, TRIG, QO_ROW>(") == n_el + 1         # one call per element + the interpreter loop's (compiled out)
    assert "#define QO_JIT_ROW false" in src                                # FULL_S needs the whole 2x2 product
    assert "static constexpr bool FULL_S = true, TRIG = true, GD = false;" in src and "#define QO_JIT_NSPEC 0" in src
    assert len(list((tmp_path / "cache").glob("chain_*_sm100a.cubin"))) == 1
    # line inside a ladder + every rf-tools opcode + group delay and |S11| specs
    fc = 10e6
    lad = W.cheby11(fc).elements
    items = [(k, list(p)) for k, p in lad[:5]] + [(Q.TLINE, [75.0, 20.0, fc])] + [(k, list(p)) for k, p in lad[5:]]
    items += [(k, list(p)) for k, p in W.if_bpf_net().elements] + [(Q.SER_R, [1.0]), (Q.SHUNT_LC_SER, [1e-6, 1e-10])]
    net = Q.Net.from_elements(items, 50.0, 75.0)
    f = Q.grid_log(fc / 3, fc * 5, 300)
    specs = [(Q.SPEC_S21_MIN_DB, 0.0, fc, -3.0), (Q.SPEC_GD_MAX, 0.3 * fc, 0.9 * fc, 1e-6), (Q.SPEC_S11_MAX_DB, 0.0, 0.5 * fc, -9.0)]
    g = Q.chain_jit_analyze(net, f, specs, [(5, 0, 0, Q.TOL_REL, 0.05)], hist_bins=16, hist_spec=1, hist_lo=0.0, hist_hi=1e-6)
    assert g["compiled"], g
    src = dump.read_text()
    assert "GD = true" in src and "#define QO_JIT_HIST_KIND 4" in src and "#define QO_JIT_NEED_S11 1" in src
    assert src.count("qo_chain_step<T, TRIG, QO_ROW>(") == len(items) + 1
    assert "#define QO_JIT_ROW false" in src                                # an |S11| spec: both rows
    g2 = Q.chain_jit_analyze(net, f, specs[:2], [(5, 0, 0, Q.TOL_REL, 0.05)], hist_bins=16, hist_spec=1, hist_lo=0.0, hist_hi=1e-6)
    assert g2["compiled"] and "#define QO_JIT_ROW true" in dump.read_text()  # |S21| and group delay only: the row vector [1 Rs] M
    with pytest.raises(Q.QoError):                                           # microstrip networks have their own kernels
        Q.chain_jit_analyze(W.pa_lpf_net(), f)


def test_executed_profile_is_of_this_machine_code():
    """profiles/executed_fp64.json carries, next to the source hash, the per-kernel hash of the SASS its ncu captures were taken
    on.  build() writes the same hashes for the library just linked (qo-100-tools_b200/lib/sass_hashes.json): the headline kernels'
    machine code must be the profiled one, or the profile has to be re-captured."""
    import hashlib
    import json
    lib = os.path.join(ROOT, "qo-100-tools_b200", "lib")
    try:
        built = json.load(open(os.path.join(lib, "sass_hashes.json")))
    except OSError:
        pytest.skip("no sass_hashes.json next to the library (cuobjdump missing when build() ran)")
    if built.get("lib_sha256") != hashlib.sha256(open(os.path.join(lib, "libqo100net.so"), "rb").read()).hexdigest():
        pytest.skip("sass_hashes.json describes another build of the library")
    prof = json.load(open(os.path.join(ROOT, "profiles", "executed_fp64.json")))
    import bench
    same_source = prof.get("_src_hash") == bench.kernel_source_hash()
    stale = []
    for k in ("qo_mc_ts_kernel", "qo_mc_tf_kernel", "qo_mc_ladder_kernel"):
        same_sass = built["kernels"][k]["sha"] == prof["_sass"][k]
        ex = bench.executed_profile(k, "cfg2-cheby11")
        # the bench line says exactly what is true of this build
        assert bench.profile_match(ex, k) == ("source" if same_source else "sass" if same_sass else False), k
        if not (same_source or same_sass):
            stale.append(k)
    if stale:
        pytest.skip("machine code of %s differs from the profiled build: bench.py reports profile_match = false until the captures are "
                    "retaken (tools/profile_all.sh, tools/update_executed.py)" % ", ".join(stale))


def test_chain_kernel_generator_on_random_cascades(Q):
    """The generator of the compiled chain kernel on the differential fuzzer's random cascades (tools/fuzz_parity.py: all ten lumped
    branch kinds with and without parasitics; coupled line, physical coupled microstrip, transmission line or the measured two-port
    of pa-bias-simulation.sch:39 in front; a line / the measured block behind): every job compiles for sm_100a, reduce-only (row-vector
    and 2x2 flavours) and FULL_S.  Host only; the GPU side of the same networks is tools/fuzz_parity.py --chain-jit."""
    import importlib.util
    w = Q.Net.from_elements([(Q.SER_R, [1.0])], 50.0, 50.0)
    a = Q.chain_jit_analyze(w, [1e6, 2e6], [(Q.SPEC_S21_MIN_DB, 0.0, 1e9, -3.0)])
    if not a["compiled"] and "libnvrtc" in (a["error"] or ""):
        pytest.skip("libnvrtc is not loadable here: %s" % a["error"])
    assert a["compiled"], a
    spec = importlib.util.spec_from_file_location("fuzz_parity", os.path.join(ROOT, "tools", "fuzz_parity.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    fronts = set()
    for i in range(10):
        rng = np.random.default_rng([5, i])
        net, f, tols, fc = mod.random_net(Q, rng)
        rs, rl = net.terminations
        if i % 2 == 0:
            ne = len(net)
            net = net.concat(Q.Net.from_elements([(Q.TLINE, [60.0, 33.0, fc])], rs, rl))
            tols = list(tols) + [(ne, 0, 1 + max(t[2] for t in tols), Q.TOL_REL, 0.05)]
        if i % 3 == 0 and net.elements[0][0] != Q.SBLOCK:
            net = net.concat(mod._block(Q).as_net(True, rs, rl))
        fronts.add(net.elements[0][0] if net.elements[0][0] != Q.SUBST else net.elements[1][0])
        f = f[:64]
        lo, hi = float(f[0]), float(f[-1])
        s21 = [(Q.SPEC_S21_MIN_DB, lo, hi, -3.0), (Q.SPEC_S21_MAX_DB, lo, hi, -0.01)]
        for specs, mode, hist in ((s21, Q.MODE_REDUCE_ONLY, dict(hist_bins=16, hist_spec=0, hist_lo=-6.0, hist_hi=0.0)),
                                  (s21 + [(Q.SPEC_S11_MAX_DB, lo, hi, -10.0)], Q.MODE_REDUCE_ONLY, {}),
                                  ([], Q.MODE_FULL_S, {})):
            r = Q.chain_jit_analyze(net, f, specs, tols, mode=mode, **hist)
            assert r["compiled"], (i, mode, r["error"])
            assert r["registers"] == -1 or r["registers"] <= 128
    assert len(fronts) >= 3, fronts


def test_chain_kernel_full_s_with_an_older_nvrtc(tmp_path):
    """A process that imported torch carries torch's own libnvrtc (CUDA 12.8 here), whose PTX level predates the 256-bit global stores
    of the FULL_S path.  The chain generator prefers the toolkit's NVRTC; pointed at the older one (QO100NET_NVRTC) it must still
    produce a kernel -- with two 128-bit stores per plane (QO_NO_ST256) -- instead of failing in ptxas."""
    import glob
    import importlib.util
    import subprocess
    import sys
    sp = importlib.util.find_spec("nvidia.cuda_nvrtc")
    cands = []
    if sp is not None and sp.submodule_search_locations:
        for d in sp.submodule_search_locations:
            cands += glob.glob(os.path.join(d, "lib", "libnvrtc.so.*"))
    cands = [c for c in cands if "builtins" not in c]
    if not cands:
        pytest.skip("no pip-installed libnvrtc next to torch")
    dump = tmp_path / "fs.cu"
    code = ("import sys, json; sys.path.insert(0, %r)\n"
            "import qo100net as Q\nfrom qo100net import workloads as W\n"
            "w = W.cfg5(1000)\n"
            "print(json.dumps(Q.chain_jit_analyze(w.net, w.f[:200], [], w.tols, mode=Q.MODE_FULL_S)))\n") % os.path.join(ROOT, "qo-100-tools_b200", "python")
    env = dict(os.environ, QO100NET_NVRTC=cands[0], QO100NET_CHAIN_JIT_DUMP=str(dump))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stderr[-800:]
    import json
    a = json.loads(r.stdout.strip().splitlines()[-1])
    assert a["compiled"], a
    src = dump.read_text()
    import ctypes
    L = ctypes.CDLL(cands[0])
    mj, mn = ctypes.c_int(), ctypes.c_int()
    L.nvrtcVersion(ctypes.byref(mj), ctypes.byref(mn))
    assert ("#define QO_NO_ST256 1" in src) == ((mj.value, mn.value) < (12, 9)), (mj.value, mn.value)
