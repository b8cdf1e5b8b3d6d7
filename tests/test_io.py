"""Product-side readers / writers of the reference's on-disk formats."""
import os

import numpy as np
import pytest

from helpers import load_golden_tps
from oracle import vmc
from peps_b200 import io as pio
from peps_b200.api import SplitIndexTPS, Configuration

# The reference's own fixture files are not part of this repository. The fixtures below are written in its on-disk layout
# (SURVEY.md section 8c) from the golden tensors that tests/golden/make_golden.py and make_fermion_golden.py re-packed
# from those files. The hash fields stand in for TensorToolkit's: the readers skip them and the writers copy them from
# a template, which the byte-for-byte rewrites below check.
TPS_DIRS = (-1, 1, 1, -1)                                   # L, U legs IN; D, R legs OUT


def _hash(*key):
    """A fixed stand-in hash per key (key entries >= -1)."""
    return int(np.random.default_rng([k + 1 for k in key]).integers(1, 2 ** 63))


def qlten_dense_bytes(a, dirs):
    """One-block TrivialRepQN stream: rank; per index nsct dgnc sector-hash dir dim index-hash; nblocks and the block's
    coordinates; the row-major payload; a trailing newline."""
    head = [str(a.ndim)]
    for d, di in zip(a.shape, dirs):
        head += ["1", str(d), str(_hash(d, 0)), str(di), str(d), str(_hash(d, di))]
    head += ["1"] + ["0"] * a.ndim
    return ("\n".join(head) + "\n").encode() + np.ascontiguousarray(a).tobytes() + b"\n"


def qlten_fz2_bytes(a, par, dirs):
    """fZ2 stream of the dense array ``a``: per index nsct, per sector qnval qnhash dgnc hash (one sector per run of
    equal parity in ``par``), dir dim hash; then every block that holds a non-zero element, in lexicographic order, and
    their payloads."""
    legs = []
    for p in par:
        cuts = [0] + [i for i in range(1, len(p)) if p[i] != p[i - 1]] + [len(p)]
        legs.append([(int(p[lo]), lo, hi) for lo, hi in zip(cuts, cuts[1:])])
    head = [str(a.ndim)]
    for k, (scts, di) in enumerate(zip(legs, dirs)):
        head.append(str(len(scts)))
        for qn, lo, hi in scts:
            head += [str(qn), str(_hash(qn, 7)), str(hi - lo), str(_hash(qn, hi - lo))]
        head += [str(di), str(a.shape[k]), str(_hash(a.shape[k], di, len(scts)))]
    blocks = []
    for coord in np.ndindex(*[len(s) for s in legs]):
        blk = a[tuple(slice(legs[k][c][1], legs[k][c][2]) for k, c in enumerate(coord))]
        if np.any(blk != 0):
            blocks.append((coord, blk))
    head.append(str(len(blocks)))
    for coord, _ in blocks:
        head += [str(c) for c in coord]
    return ("\n".join(head) + "\n").encode() + b"".join(np.ascontiguousarray(b).tobytes() for _, b in blocks) + b"\n"


def write_tps_fixture(d, tps, dirs=TPS_DIRS):
    os.makedirs(d)
    open(os.path.join(d, "tps_meta.txt"), "w").write(f"{len(tps)} {len(tps[0])} {len(tps[0][0])}")
    for r, row in enumerate(tps):
        for c, site in enumerate(row):
            for s, t in enumerate(site):
                open(os.path.join(d, f"tps_ten{r}_{c}_{s}.qlten"), "wb").write(qlten_dense_bytes(t, dirs))
    return d


def heisenberg_4x4_fixture(d):
    """slow_tests/test_data/tps_square_heisenberg4x4D8Double with its configuration files."""
    tps, z = load_golden_tps("heis4x4_D8_double")
    write_tps_fixture(d, tps)
    for k, cfg in enumerate(z["configs"]):
        open(os.path.join(d, f"configuration{k}"), "w").write("".join(" ".join(map(str, row)) + "\n" for row in cfg))
    return d, tps, z


# reference fixture directory -> golden re-pack of it
FERMION_FIXTURES = {"spinless_fermion_tps_t2_2.100000_double_from_simple_update": "sf2x2_t2_+2.1_double_su",
                    "spinless_fermion_tps_t2_-2.500000_complexlowest": "sf2x2_t2_-2.5_complex_lowest",
                    "tj_model_tps_double_from_simple_update": "tj2x2_double_su"}


def fermion_fixture(d, name):
    """A test_data/<name> fZ2 TPS directory: site tensors (L in, D out, R out, U in, parity leg in of dim 1)."""
    from test_fermion_oracle import load_golden
    g, _ = load_golden(FERMION_FIXTURES[name])
    os.makedirs(d)
    rows, cols, phys = len(g.T), len(g.T[0]), len(g.T[0][0])
    open(os.path.join(d, "tps_meta.txt"), "w").write(f"{rows} {cols} {phys}")
    for r in range(rows):
        for c in range(cols):
            for s in range(phys):
                par = list(g.par[r][c]) + [np.array([g.phys_par[s]])]
                data = qlten_fz2_bytes(np.asarray(g.T[r][c][s])[..., None], par, (-1, 1, 1, -1, -1))
                open(os.path.join(d, f"tps_ten{r}_{c}_{s}.qlten"), "wb").write(data)
    return d


def test_tps_and_configuration_round_trip(tmp_path):
    tps = SplitIndexTPS(vmc.random_tps(3, 4, 2, 3, seed=1))
    pio.dump_tps(tps, str(tmp_path / "tps"))
    back = pio.load_tps(str(tmp_path / "tps"))
    assert np.array_equal(back.pack(), tps.pack())
    cfg = Configuration(vmc.shuffled_half_filled_config(3, 4, 9))
    pio.dump_configuration(cfg, str(tmp_path / "configuration0"))
    assert pio.load_configuration(str(tmp_path / "configuration0")) == cfg


def test_reads_reference_fixture_and_rewrites_it_byte_for_byte(tmp_path):
    d, gold, z = heisenberg_4x4_fixture(str(tmp_path / "tps_square_heisenberg4x4D8Double"))
    tps = pio.load_tps(d)
    assert np.array_equal(tps.pack(), SplitIndexTPS(gold).pack())
    assert np.array_equal(pio.load_configuration(os.path.join(d, "configuration3")).data, z["configs"][3])
    # with the fixture as header template the writer reproduces the reference's files exactly
    pio.dump_tps(tps, str(tmp_path / "out"), template_dir=d)
    for name in ("tps_ten1_1_0.qlten", "tps_ten0_0_1.qlten", "tps_ten3_3_0.qlten"):
        assert open(os.path.join(d, name), "rb").read() == open(tmp_path / "out" / name, "rb").read()


def test_read_qlten_checks_the_payload(tmp_path):
    a = np.arange(24, dtype=np.float64).reshape(2, 3, 4)
    p = str(tmp_path / "t.qlten")
    pio.write_qlten(p, a)
    assert np.array_equal(pio.read_qlten(p), a)
    raw = open(p, "rb").read()
    open(p, "wb").write(raw[:-17])                       # truncated payload
    with pytest.raises(ValueError):
        pio.read_qlten(p)
    with pytest.raises(ValueError):                      # a real file read as complex
        open(p, "wb").write(raw)
        pio.read_qlten(p, dtype=np.complex128)


def test_complex_fixture_is_detected(tmp_path):
    tps, _ = load_golden_tps("heis4x4_D8_double")
    rng = np.random.default_rng(3)
    ctps = [[[t * np.exp(1j * rng.uniform(0, 2 * np.pi, t.shape)) for t in site] for site in row] for row in tps]
    d = write_tps_fixture(str(tmp_path / "tps_square_heisenberg4x4D8Complex"), ctps)
    t = pio.read_qlten(os.path.join(d, "tps_ten1_1_0.qlten"))
    assert t.dtype == np.complex128 and t.shape == (8, 8, 8, 8)
    assert np.array_equal(t, ctps[1][1][0])
    with pytest.raises(ValueError):
        pio.read_qlten(os.path.join(d, "tps_ten1_1_0.qlten"), dtype=np.float64)


def test_measurement_stats_dump_layout(tmp_path):
    """MCPEPSMeasurer::DumpData layout (monte_carlo_peps_measurer_impl.h:266-330, 544-620): 2-D observables as
    <key>_mean.csv / <key>_stderr.csv (17 significant digits, scientific), flat ones as index,mean,stderr."""
    from peps_b200.api import dump_measurement_stats
    res = {"spin_z": (np.array([[0.5, -0.25], [0.125, 1 / 3]]), np.array([[0.1, 0.2], [0.3, 0.4]])),
           "energy": (np.array(-1.9952127879312345), np.array(1e-3))}
    dump_measurement_stats(res, str(tmp_path / "out"), {"lx": 2, "ly": 2})
    rows = open(tmp_path / "out" / "stats" / "spin_z_mean.csv").read().splitlines()
    assert rows[0] == "5.0000000000000000e-01,-2.5000000000000000e-01" and float(rows[1].split(",")[1]) == 1 / 3
    flat = open(tmp_path / "out" / "stats" / "energy.csv").read().splitlines()
    assert flat[0] == "index,mean,stderr" and flat[1].startswith("0,-1.9952127879312345e+00,")
    meta = open(tmp_path / "out" / "metadata.txt").read()
    assert meta.startswith("format_version 1\n") and "lx 2" in meta


def test_fermion_tps_loader_matches_repacked_fixture(tmp_path):
    """peps_b200.io.load_fermion_tps on an fZ2 fixture == the committed re-packed golden."""
    name = "spinless_fermion_tps_t2_2.100000_double_from_simple_update"
    d = fermion_fixture(str(tmp_path / name), name)
    from peps_b200.io import load_fermion_tps
    from test_fermion_oracle import load_golden
    f = load_fermion_tps(d)
    g, _ = load_golden("sf2x2_t2_+2.1_double_su")
    assert f.phys_par == g.phys_par == (1, 0)
    for r in range(2):
        for c in range(2):
            for s in range(2):
                assert np.array_equal(f.t[r][c][s], g.T[r][c][s])
            for k in range(4):
                assert np.array_equal(f.par[r][c][k], g.par[r][c][k])


@pytest.mark.parametrize("name", list(FERMION_FIXTURES))
def test_fermion_tps_writer_reproduces_reference_files(tmp_path, name):
    """dump_fermion_tps with the fixture as header template rewrites every fZ2 file byte for byte (double and complex);
    an edited state reloads with the edit."""
    d = fermion_fixture(str(tmp_path / name), name)
    f = pio.load_fermion_tps(d)
    assert np.iscomplexobj(f.t[0][0][0]) == ("complex" in name)
    pio.dump_fermion_tps(f, str(tmp_path / "out"), d)
    for fn in sorted(os.listdir(d)):
        if fn.endswith(".qlten") and fn.startswith("tps_ten"):
            assert open(os.path.join(d, fn), "rb").read() == open(tmp_path / "out" / fn, "rb").read(), fn
    g = f * 0.5
    g = type(f)(g.t, f.par, f.phys_par)
    pio.dump_fermion_tps(g, str(tmp_path / "half"), d)
    back = pio.load_fermion_tps(str(tmp_path / "half"))
    assert np.array_equal(back.pack(), 0.5 * f.pack())
    bad = type(f)([[[x + 1.0 for x in site] for site in row] for row in f.t], f.par, f.phys_par)   # parity-violating entries
    with pytest.raises(ValueError):
        pio.dump_fermion_tps(bad, str(tmp_path / "bad"), d)


def test_measurement_stats_dump_complex_values(tmp_path):
    """QLTEN_Complex measurement runs: ToCsvString(std::complex<double>) streams (re,im) (monte_carlo_peps_measurer_impl.h:31-36)."""
    from peps_b200.api import dump_measurement_stats
    res = {"bond_energy_h": (np.array([[0.5 + 0.25j, -1.0j]]), np.array([[0.1, 0.2]])), "energy": (np.array(-2.0 + 1e-3j), np.array(1e-4))}
    dump_measurement_stats(res, str(tmp_path / "out"))
    row = open(tmp_path / "out" / "stats" / "bond_energy_h_mean.csv").read().splitlines()[0]
    assert row == "(5.0000000000000000e-01,2.5000000000000000e-01),(-0.0000000000000000e+00,-1.0000000000000000e+00)" or \
        row == "(5.0000000000000000e-01,2.5000000000000000e-01),(0.0000000000000000e+00,-1.0000000000000000e+00)"
    flat = open(tmp_path / "out" / "stats" / "energy.csv").read().splitlines()
    assert flat[1].startswith("0,(-2.0000000000000000e+00,1.0000000000000000e-03),")
