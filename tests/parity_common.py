"""Parity checks shared by the hostsim (CPU, host-logic) tests and the GPU tests: the same scenario is run through
the C ABI (``lib`` decides which build) and through the oracle, and compared."""
import numpy as np

from oracle import vmc
from peps_b200.api import BMPSTruncateParams, SplitIndexTPS, WalkerBatch


def make_case(rows, cols, D, W, seed=1, signed=False):
    tps = vmc.random_tps(rows, cols, 2, D, seed=seed, signed=signed)
    cfgs = np.stack([vmc.neel_config(rows, cols)] +
                    [vmc.shuffled_half_filled_config(rows, cols, 10 + w) for w in range(1, W)])
    return tps, cfgs


def flat_holes(holes, rows, cols):
    return np.concatenate([holes[r][c].ravel() for r in range(rows) for c in range(cols)])


def run_pipeline_parity(lib, rows, cols, D, W, trunc, nsweeps=2, seed=1, signed=False, tol=1e-10, seeds0=100,
                        check_configs=True, j2=0.0, tfim_h=None, three_site=False, pinning00=0.0):
    """Sweeps + energy + holes for W walkers through the C ABI vs the oracle, walker by walker.
    tfim_h: transverse-field Ising model with the full-space (Suwa-Todo) updater instead of XXZ + exchange
    (BASELINE config #1); pinning00: the XXZ / J1-J2 model's pinning field on site (0, 0)."""
    tps, cfgs = make_case(rows, cols, D, W, seed, signed)
    tr = BMPSTruncateParams.SVD(*trunc)
    b = WalkerBatch(rows, cols, 2, D, W, tr, lib=lib)
    b.set_tps(SplitIndexTPS(tps))
    b.set_configs(cfgs)
    b.seed_rng(np.arange(seeds0, seeds0 + W))
    if j2 != 0.0:
        from peps_b200.api import SquareSpinOneHalfJ1J2XXZModelOBC
        b.set_model(SquareSpinOneHalfJ1J2XXZModelOBC(1.0, 1.0, j2, j2, pinning00))
    elif pinning00 != 0.0:
        from peps_b200.api import SquareSpinOneHalfXXZModelOBC
        b.set_model(SquareSpinOneHalfXXZModelOBC(1.0, 1.0, pinning00))
    if tfim_h is not None:
        from peps_b200.api import TransverseFieldIsingSquareOBC, MCUpdateSquareNNFullSpaceUpdate
        b.set_model(TransverseFieldIsingSquareOBC(tfim_h))
        b.set_updater(MCUpdateSquareNNFullSpaceUpdate())
    if three_site:
        from peps_b200.api import MCUpdateSquareTNN3SiteExchange
        b.set_updater(MCUpdateSquareTNN3SiteExchange())
    b.init_walkers()
    ws = [vmc.Walker(tps, cfgs[w], trunc) for w in range(W)]
    if three_site:
        ups = [vmc.TNN3SiteExchangeUpdater(seeds0 + w) for w in range(W)]
        model = vmc.XXZModel(1.0, 1.0, pinning00, j2, j2)
    elif tfim_h is not None:
        ups = [vmc.NNFullSpaceUpdater(seeds0 + w) for w in range(W)]
        model = vmc.TFIMModel(tfim_h)
    else:
        ups = [vmc.NNExchangeUpdater(seeds0 + w) for w in range(W)]
        model = vmc.XXZModel(1.0, 1.0, pinning00, j2, j2)
    amp0 = b.amplitudes()
    ref0 = np.array([w_.amplitude for w_ in ws])
    report = {"amp0": float(np.max(np.abs(amp0 / ref0 - 1)))}
    assert report["amp0"] < tol, report
    worst = dict(amp=0.0, eloc=0.0, hole=0.0, psi=0.0)
    for it in range(nsweeps):
        acc = b.sweep(1)
        racc = np.array([ups[w].sweep(tps, ws[w])[0] for w in range(W)])
        c = b.get_configs()
        if check_configs:
            for w in range(W):
                assert np.array_equal(c[w], ws[w].config), f"sweep {it}: configuration of walker {w} diverged"
            assert np.array_equal(acc, racc)
        amp = b.amplitudes()
        ramp = np.array([w_.amplitude for w_ in ws])
        e, psi = b.energy_and_holes(True, True)
        holes = b.holes()
        for w in range(W):
            ee, hh, pp = model.energy_and_holes(tps, ws[w], True)
            fh = flat_holes(hh, rows, cols)
            worst["eloc"] = max(worst["eloc"], abs(e[w] - ee) / max(1.0, abs(ee)))
            worst["hole"] = max(worst["hole"], float(np.max(np.abs(holes[w] - fh)) / np.max(np.abs(fh))))
            worst["psi"] = max(worst["psi"], float(np.max(np.abs(psi[:len(pp), w] / np.array(pp) - 1))))   # TFIM: rows only
        worst["amp"] = max(worst["amp"], float(np.max(np.abs(amp / ramp - 1))))
    report.update(worst)
    for k, v in worst.items():
        assert v < tol, (k, report)
    b.close()
    return report


def run_gradient_parity(lib, rows, cols, D, W, trunc, nsamples=3, seed=2, tol=1e-10):
    """peps_sample x nsamples + accumulators vs the oracle's EnergyGradEvaluator (walker == rank)."""
    tps, cfgs = make_case(rows, cols, D, W, seed)
    tr = BMPSTruncateParams.SVD(*trunc)
    b = WalkerBatch(rows, cols, 2, D, W, tr, lib=lib)
    b.set_tps(SplitIndexTPS(tps))
    b.set_configs(cfgs)
    b.seed_rng(np.arange(500, 500 + W))
    b.init_walkers()
    b.zero_accumulators()
    energies = np.zeros((W, nsamples))
    for s in range(nsamples):
        e, _ = b.sample(1)
        energies[:, s] = e
    osum, eosum = b.accumulators()
    ev = vmc.EnergyGradEvaluator(tps, vmc.XXZModel(), trunc, 1)
    rr = []
    for w in range(W):
        rr.append(ev.sample_rank(vmc.Walker(tps, cfgs[w], trunc), vmc.NNExchangeUpdater(500 + w), nsamples))
    ref_e = np.array([r["energies"] for r in rr])
    assert np.max(np.abs(energies - ref_e) / np.maximum(1, np.abs(ref_e))) < tol
    like = SplitIndexTPS(tps)
    ref_o = sum((SplitIndexTPS(r["ostar_sum"]) for r in rr[1:]), SplitIndexTPS(rr[0]["ostar_sum"])).pack()
    ref_eo = sum((SplitIndexTPS(r["eloc_ostar_sum"]) for r in rr[1:]), SplitIndexTPS(rr[0]["eloc_ostar_sum"])).pack()
    assert np.max(np.abs(osum - ref_o)) < tol * np.max(np.abs(ref_o))
    assert np.max(np.abs(eosum - ref_eo)) < tol * np.max(np.abs(ref_eo))
    energy, err, grad = ev.combine(rr)
    from peps_b200.api import combine_energy_bins
    e2, err2 = combine_energy_bins(energies)
    assert abs(e2 - energy) < 1e-12 * max(1, abs(energy))
    g2 = (eosum - e2 * osum) / (nsamples * W)
    gref = SplitIndexTPS(grad).pack()
    assert np.max(np.abs(g2 - gref)) < tol * max(np.max(np.abs(gref)), 1e-300)
    b.close()
    return dict(energy=energy, gnorm=float(np.sum(gref ** 2)))


def run_plaquette_trace_parity(lib, rows=4, cols=5, D=2, W=3, tol=1e-10):
    """peps_probe_plaquette_trace (ReplaceNNNSiteTrace / ReplaceSqrt5DistTwoSiteTrace, both link directions and both MPS
    orientations) vs the oracle amplitude of the configuration with the two corner spins exchanged."""
    tps = vmc.random_tps(rows, cols, 2, D, seed=12)
    cfgs = np.stack([vmc.shuffled_half_filled_config(rows, cols, 3 + w) for w in range(W)])
    trunc = (1, 1000, 0.0)
    b = WalkerBatch(rows, cols, 2, D, W, BMPSTruncateParams.SVD(*trunc), lib=lib)
    b.set_tps(SplitIndexTPS(tps))
    b.set_configs(cfgs)
    b.init_walkers()
    worst = 0.0
    for kind in (0, 1):
        for d in (0, 1):
            for o in (0, 1):
                r1, c1 = 1, 1
                h, wd = (2, 2) if kind == 0 else ((2, 3) if o == 0 else (3, 2))
                a_, b_ = ((r1, c1), (r1 + h - 1, c1 + wd - 1)) if d == 0 else ((r1 + h - 1, c1), (r1, c1 + wd - 1))
                psi = b.probe_plaquette_trace(kind, r1, c1, d, o)
                for w in range(W):
                    c2 = cfgs[w].copy()
                    c2[a_], c2[b_] = cfgs[w][b_], cfgs[w][a_]
                    ref = vmc.Walker(tps, c2, trunc).amplitude
                    worst = max(worst, abs(psi[w] / ref - 1))
                    assert abs(psi[w] / ref - 1) < tol, (kind, d, o, w, psi[w], ref)
    b.close()
    return worst


def spin_one_matrices(j1=1.0, j2=0.3, dz=0.4, hx=0.2):
    """Spin-1 test model: J1/J2 Heisenberg bonds, single-ion anisotropy dz (Sz)^2 and a transverse field hx Sx (d = 3)."""
    sz = np.diag([1.0, 0.0, -1.0])
    sp = np.zeros((3, 3)); sp[0, 1] = sp[1, 2] = np.sqrt(2.0)
    sm = sp.T
    hb = np.kron(sz, sz) + 0.5 * (np.kron(sp, sm) + np.kron(sm, sp))
    h1 = dz * sz @ sz + hx * 0.5 * (sp + sm)
    return j1 * hb, j2 * hb, h1


def run_table_model_parity(lib, tol=1e-10):
    """Seam B2 as data: (i) the XXZ / J1-J2 tables reproduce the built-in solver exactly, (ii) the TFIM tables reproduce
    the built-in TFIM solver, (iii) a spin-1 (phys = 3) J1-J2 model with single-ion anisotropy and a transverse field --
    a model the engine has no branch for -- matches the oracle's generic restatement of the reference traversal."""
    from peps_b200.api import TableModel, SquareSpinOneHalfJ1J2XXZModelOBC, TransverseFieldIsingSquareOBC
    rows, cols, D, W = 3, 4, 2, 3
    tps = vmc.random_tps(rows, cols, 2, D, seed=21)
    cfgs = np.stack([vmc.shuffled_half_filled_config(rows, cols, 30 + w) for w in range(W)])
    trunc = (1, 64, 0.0)
    b = WalkerBatch(rows, cols, 2, D, W, BMPSTruncateParams.SVD(*trunc), lib=lib)
    b.set_tps(SplitIndexTPS(tps)); b.set_configs(cfgs); b.init_walkers()
    b.set_model(SquareSpinOneHalfJ1J2XXZModelOBC(1.0, 0.8, 0.5, 0.35, 0.0))
    e_builtin, psi_b = b.energy_and_holes(True, True)
    h_builtin = b.holes()
    b.set_model(TableModel.xxz(1.0, 0.8, 0.5, 0.35))
    e_tab, psi_t = b.energy_and_holes(True, True)
    assert np.array_equal(psi_b, psi_t) and np.array_equal(h_builtin, b.holes())
    assert np.max(np.abs(e_tab - e_builtin)) < 1e-13 * np.max(np.abs(e_builtin))
    b.set_model(TransverseFieldIsingSquareOBC(0.7))
    e_builtin = b.energy_and_holes(False)
    b.set_model(TableModel.tfim(0.7))
    e_tab = b.energy_and_holes(False)
    assert np.max(np.abs(e_tab - e_builtin)) < 1e-12 * np.max(np.abs(e_builtin))
    b.close()
    # spin-1
    h2, h2n, h1 = spin_one_matrices()
    tps3 = vmc.random_tps(rows, cols, 3, D, seed=22)
    rng = np.random.default_rng(5)
    cfg3 = rng.integers(0, 3, size=(W, rows, cols))
    b3 = WalkerBatch(rows, cols, 3, D, W, BMPSTruncateParams.SVD(*trunc), lib=lib)
    b3.set_tps(SplitIndexTPS(tps3)); b3.set_configs(cfg3); b3.init_walkers()
    b3.set_model(TableModel(3, h2, h2n, h1))
    e3, psi3 = b3.energy_and_holes(True, True)
    holes3 = b3.holes()
    om = vmc.TableModel(3, h2, h2n, h1)
    worst = 0.0
    for w in range(W):
        wk = vmc.Walker(tps3, cfg3[w], trunc)
        ee, hh, pp = om.energy_and_holes(tps3, wk, True)
        worst = max(worst, abs(e3[w] - ee) / max(1.0, abs(ee)))
        assert np.max(np.abs(holes3[w] - flat_holes(hh, rows, cols))) < tol * np.max(np.abs(holes3[w]))
    assert worst < tol, worst
    b3.close()
    return worst


def run_structure_factor_parity(lib, rows=3, cols=4, D=2, W=3, chi=64, tol=1e-10, complex_=False):
    """peps_measure_structure_factor vs the oracle's restatement of MeasureStructureFactor, pair by pair."""
    tps = complex_tps(rows, cols, D, 17) if complex_ else vmc.random_tps(rows, cols, 2, D, seed=17)
    cfgs = np.stack([vmc.shuffled_half_filled_config(rows, cols, 5 + w) for w in range(W)])
    trunc = (1, chi, 0.0)
    b = WalkerBatch(rows, cols, 2, D, W, BMPSTruncateParams.SVD(*trunc), lib=lib)
    if complex_:
        b.set_complex()
    b.set_tps(SplitIndexTPS(tps)); b.set_configs(cfgs); b.init_walkers()
    pairs, vals = b.measure_structure_factor()
    worst = 0.0
    for w in range(W):
        ref = vmc.measure_structure_factor(tps, vmc.Walker(tps, cfgs[w], trunc))
        assert len(ref) == len(pairs)
        scale = max(abs(r[4]) for r in ref)
        for k, r in enumerate(ref):
            assert tuple(pairs[k]) == r[:4]
            assert (r[4] == 0.0) == (vals[w, k] == 0.0)
            worst = max(worst, abs(vals[w, k] - r[4]) / scale)
    assert worst < tol, worst
    b.close()
    return worst


def run_variational_parity(lib, scheme, rows=5, cols=5, D=3, chi=5, W=2, iters=3, tol=1e-9, complex_=False):
    """BMPS::MultiplyMPO with VARIATION2Site (1) / VARIATION1Site (2) through the C ABI vs the oracle restatement, same
    number of sweeps (convergence_tol = 0): amplitudes closed on several rows, with a truncating chi."""
    from oracle.contractor import BMPSContractor
    from oracle.bmps import LEFT, RIGHT, HORIZONTAL
    tps = complex_tps(rows, cols, D, 33) if complex_ else vmc.random_tps(rows, cols, 2, D, seed=33)
    cfgs = np.stack([vmc.shuffled_half_filled_config(rows, cols, 8 + w) for w in range(W)])
    mk = BMPSTruncateParams.Variational2Site if scheme == 1 else BMPSTruncateParams.Variational1Site
    b = WalkerBatch(rows, cols, 2, D, W, mk(1, chi, 0.0, 0.0, iters), lib=lib)
    if complex_:
        b.set_complex()
    b.set_tps(SplitIndexTPS(tps)); b.set_configs(cfgs); b.init_walkers()
    worst = 0.0
    for row in (0, rows // 2, rows - 1):
        psi = b.probe_trace_row(row)
        for w in range(W):
            tn = vmc.project(tps, cfgs[w])
            c = BMPSContractor(rows, cols)
            c.init(tn)
            c.set_truncate_params(1, chi, 0.0)
            c.set_compress_scheme(scheme, 0.0, iters)
            c.grow_bmps_for_row(tn, row)
            c.init_bten(tn, LEFT, row)
            c.grow_full_bten(tn, RIGHT, row, 2, True)
            ref = c.trace(tn, (row, 0), HORIZONTAL)
            worst = max(worst, abs(psi[w] / ref - 1))
    assert worst < tol, worst
    # and the variational boundary is a good approximation: close to the exact amplitude
    exact = np.array([vmc.Walker(tps, cfgs[w], (1, 1000, 0.0)).amplitude for w in range(W)])
    assert np.max(np.abs((b.amplitudes_c() if complex_ else b.amplitudes()) / exact - 1)) < 0.2
    b.close()
    return worst


# ---------------------------------------------------------------------------------------------------------------------
# fermion mode (fZ2-graded tensors as sign-dressed dense tensors)
# ---------------------------------------------------------------------------------------------------------------------
def fermion_configs(rows, cols, W, phys, seed=10):
    """Half-filled (spinless) / two-holes-per-... configurations with an even fermion number, one per walker."""
    out = []
    n = rows * cols
    for w in range(W):
        rng = np.random.default_rng(seed + w)
        if phys == 2:
            base = np.array([0] * (n // 2 - (n // 2) % 2) + [1] * (n - n // 2 + (n // 2) % 2))
        else:                                   # t-J: up / down / empty, even number of electrons
            ne = (2 * n // 3) - ((2 * n // 3) % 2)
            base = np.array([0] * (ne // 2) + [1] * (ne - ne // 2) + [2] * (n - ne))
        out.append(rng.permutation(base).reshape(rows, cols))
    return np.stack(out)


def run_fermion_pipeline_parity(lib, rows, cols, D, W, trunc, model="spinless", nsweeps=2, seed=3, tol=1e-10, seeds0=200,
                                t2=0.6, check_holes=True, jastrow=False, complex_=False, updater="exchange", state=None):
    """Sweeps + E_loc + O* of W walkers through the C ABI in fermion mode vs oracle/fermion.py, walker by walker:
    configurations and acceptance counts bit-identical, |amplitudes|, E_loc, O* to `tol` (relative)."""
    from oracle import fermion as F
    from peps_b200.api import FermionSplitIndexTPS, TableModel
    phys_par = (1, 0) if model == "spinless" else (1, 1, 0)
    if state is not None:                       # (oracle FermionTPS, configurations): a given physical state
        f, given_cfgs = state
        assert tuple(f.phys_par) == phys_par
    else:
        f = F.FermionTPS.random(rows, cols, D, seed, phys_par=phys_par, complex_=complex_)
    ftps = FermionSplitIndexTPS(f.T, f.par, phys_par)
    if model == "spinless":
        omodel = F.SpinlessFermionModel(1.0, t2, 0.3)
        tmodel = TableModel.spinless_fermion(1.0, t2, 0.3)
    else:
        omodel = F.tJModel(1.0, 0.3, mu=0.2, V=0.075, t2=t2 if model == "tj_nnn" else 0.0)
        tmodel = TableModel.tj(1.0, 0.3, V=0.075, mu=0.2, t2=t2 if model == "tj_nnn" else 0.0)
    cfgs = given_cfgs if state is not None else fermion_configs(rows, cols, W, len(phys_par))
    tr = BMPSTruncateParams.SVD(*trunc)
    b = WalkerBatch(rows, cols, len(phys_par), D, W, tr, lib=lib)
    if complex_:
        b.set_complex()
    b.set_fermion(ftps)
    b.set_tps(ftps)
    b.set_model(tmodel)
    jas = None
    if jastrow:                                 # JastrowDress: v_ij = 0.3 / (1 + distance^2), density = fermion number
        n = rows * cols
        yy, xx = np.divmod(np.arange(n), cols)
        v = 0.3 / (1.0 + (yy[:, None] - yy[None, :]) ** 2 + (xx[:, None] - xx[None, :]) ** 2)
        np.fill_diagonal(v, 0.0)
        jas = (v, np.array(phys_par, dtype=np.int32))
        b.set_jastrow(*jas)
        omodel.jastrow = jas
    b.set_configs(cfgs)
    b.seed_rng(np.arange(seeds0, seeds0 + W))
    b.init_walkers()
    ws = [F.FermionWalker(f, cfgs[w], trunc) for w in range(W)]
    ups = [F.FermionNNExchangeUpdater(seeds0 + w, jastrow=jas) for w in range(W)]
    if updater == "full_space":                 # MCUpdateSquareNNFullSpaceUpdateOBC on fZ2 tensors (fermion number not conserved)
        from peps_b200.api import MCUpdateSquareNNFullSpaceUpdate
        b.set_updater(MCUpdateSquareNNFullSpaceUpdate())
        ups = [F.FermionNNFullSpaceUpdater(seeds0 + w) for w in range(W)]
    elif updater == "three_site":               # MCUpdateSquareTNN3SiteExchange on fZ2 tensors
        from peps_b200.api import MCUpdateSquareTNN3SiteExchange
        b.set_updater(MCUpdateSquareTNN3SiteExchange())
        ups = [F.FermionTNN3SiteExchangeUpdater(seeds0 + w) for w in range(W)]
    amps = b.amplitudes_c if complex_ else b.amplitudes
    a0 = np.abs(amps())
    r0 = np.abs(np.array([w_.amplitude for w_ in ws]))
    assert np.max(np.abs(a0 / r0 - 1)) < tol
    worst = dict(amp=0.0, eloc=0.0, ostar=0.0)
    for it in range(nsweeps):
        acc = b.sweep(1)
        racc = np.array([ups[w].sweep(ws[w])[0] for w in range(W)])
        c = b.get_configs()
        for w in range(W):
            assert np.array_equal(c[w], ws[w].config), (it, w)
        assert np.array_equal(acc, racc), (acc, racc)
        amp = amps()
        ramp = np.array([w_.amplitude for w_ in ws])
        worst["amp"] = max(worst["amp"], float(np.max(np.abs(np.abs(amp) / np.abs(ramp) - 1))))
        e = b.energy_and_holes(check_holes)
        holes = (b.holes_c() if complex_ else b.holes()) if check_holes else None
        for w in range(W):
            re, rost, _ = omodel.energy_and_holes(ws[w], check_holes)
            worst["eloc"] = max(worst["eloc"], abs(e[w] - re) / max(1.0, abs(re)))
            if check_holes:
                ref = np.concatenate([rost[r][c_].ravel() for r in range(rows) for c_ in range(cols)])
                got = np.conj(holes[w] / amp[w])              # O* = conj(finished hole / cached amplitude)
                worst["ostar"] = max(worst["ostar"], float(np.max(np.abs(got - ref)) / np.max(np.abs(ref))))
    assert worst["amp"] < tol and worst["eloc"] < tol and worst["ostar"] < tol, worst
    b.close()
    return worst


def run_sector_truncation_case(lib, nr=160, nc=192, t=24, W=3, seed=4):
    """Standalone truncation (peps_test_truncate) of Theta matrices with the Z2 structure of fermion mode: rows and columns
    fall into two parity sectors (interleaved at random), entries outside the two diagonal blocks are exact zeros. With
    PEPS_Z2_SECTORS=1 the block-Jacobi schedule regroups the rows and skips cross-sector pairs; the kept right singular
    subspace must equal the exact one (projector to 1e-11) and the kept rows must be orthonormal."""
    import ctypes as C
    rng = np.random.default_rng(seed)
    th = np.zeros((W, nr, nc))
    projs = []
    for w in range(W):
        rsec = rng.integers(0, 2, nr)
        csec = rng.integers(0, 2, nc)
        pi = int(rng.integers(0, 2))
        idx = [(np.flatnonzero(rsec == (s ^ pi)), np.flatnonzero(csec == s)) for s in (0, 1)]
        ks = [min(len(ri), len(ci)) for ri, ci in idx]
        # flat spectrum (full rank, nothing deflates) with a clear gap at the cut, dealt to the two sectors at random
        allsv = np.sort(0.5 + rng.random(ks[0] + ks[1]))[::-1]
        allsv[:t] += 0.05
        owner = rng.permutation(np.array([0] * ks[0] + [1] * ks[1]))
        for s, (ri, ci) in enumerate(idx):
            k = ks[s]
            u, _ = np.linalg.qr(rng.standard_normal((len(ri), k)))
            v, _ = np.linalg.qr(rng.standard_normal((len(ci), k)))
            th[w][np.ix_(ri, ci)] = (u * allsv[owner == s]) @ v.T
        _, s_all, vt = np.linalg.svd(th[w])
        assert s_all[t - 1] - s_all[t] > 0.04
        projs.append(vt[:t].T @ vt[:t])
    b = np.empty((W, t, nc))
    kept = np.empty(W, dtype=np.int32)
    sweeps = C.c_int32()
    dp = lambda x: x.ctypes.data_as(C.POINTER(C.c_double))
    rc = lib.peps_test_truncate(0, W, nr, nc, t, t, 0.0, dp(th), dp(b), kept.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(sweeps))
    assert rc == 0, lib.peps_last_error(None)
    for w in range(W):
        assert kept[w] == t
        assert np.max(np.abs(b[w] @ b[w].T - np.eye(t))) < 1e-12
        assert np.max(np.abs(b[w].T @ b[w] - projs[w])) < 1e-11
    return sweeps.value


# ---------------------------------------------------------------------------------------------------------------------
# complex (QLTEN_Complex) states
# ---------------------------------------------------------------------------------------------------------------------
def complex_tps(rows, cols, D, seed, phys=2):
    """uniform [0,1) real parts and uniform [-0.5, 0.5) imaginary parts, NormalizeAllSite."""
    rng = np.random.default_rng(seed)
    tps = vmc.random_tps(rows, cols, phys, D, seed=seed, dtype=np.complex128)
    for row in tps:
        for site in row:
            for s in range(len(site)):
                site[s] = site[s] + 1j * (rng.random(site[s].shape) - 0.5) * np.max(np.abs(site[s]))
    return vmc.normalize_all_site(tps)


def run_complex_pipeline_parity(lib, rows, cols, D, W, trunc, nsweeps=2, seed=6, tol=1e-10, seeds0=300, j2=0.0,
                                tfim_h=None, three_site=False, table=None):
    """Sweeps + E_loc + holes + accumulators of W walkers on a COMPLEX state through the C ABI vs the oracle (which is
    pinned on the reference's complex goldens, K5): configurations and acceptance counts bit-identical, amplitudes,
    E_loc = sum ... conj(psi_ex / psi), O* = conj(hole / psi), sum O* and sum conj(E_loc) O* to `tol` (relative).
    tfim_h: transverse-field Ising + full-space (Suwa-Todo) updater; three_site: the 3-site exchange updater;
    table = "xxz": the XXZ / J1-J2 model as tables (seam B2), "spin1": the phys = 3 table model of run_table_model_parity."""
    phys = 3 if table == "spin1" else 2
    tps = complex_tps(rows, cols, D, seed, phys)
    if phys == 2:
        cfgs = np.stack([vmc.neel_config(rows, cols)] + [vmc.shuffled_half_filled_config(rows, cols, 20 + w) for w in range(1, W)])
    else:
        cfgs = np.random.default_rng(seed).integers(0, 3, size=(W, rows, cols))
    b = WalkerBatch(rows, cols, phys, D, W, BMPSTruncateParams.SVD(*trunc), lib=lib)
    b.set_complex()
    b.set_tps(SplitIndexTPS(tps))
    from peps_b200.api import (SquareSpinOneHalfJ1J2XXZModelOBC, TransverseFieldIsingSquareOBC, TableModel,
                               MCUpdateSquareNNFullSpaceUpdate, MCUpdateSquareTNN3SiteExchange)
    model = vmc.XXZModel(1.0, 1.0, 0.0, j2, j2)
    ups = [vmc.NNExchangeUpdater(seeds0 + w) for w in range(W)]
    if table == "xxz":
        b.set_model(TableModel.xxz(1.0, 1.0, j2, j2))
    elif table == "spin1":
        h2, h2n, h1 = spin_one_matrices()
        b.set_model(TableModel(3, h2, h2n, h1))
        model = vmc.TableModel(3, h2, h2n, h1)
    elif j2 != 0.0:
        b.set_model(SquareSpinOneHalfJ1J2XXZModelOBC(1.0, 1.0, j2, j2, 0.0))
    if tfim_h is not None:
        b.set_model(TransverseFieldIsingSquareOBC(tfim_h))
        model = vmc.TFIMModel(tfim_h)
    if tfim_h is not None or table == "spin1":
        b.set_updater(MCUpdateSquareNNFullSpaceUpdate())
        ups = [vmc.NNFullSpaceUpdater(seeds0 + w) for w in range(W)]
    if three_site:
        b.set_updater(MCUpdateSquareTNN3SiteExchange())
        ups = [vmc.TNN3SiteExchangeUpdater(seeds0 + w) for w in range(W)]
    b.set_configs(cfgs)
    b.seed_rng(np.arange(seeds0, seeds0 + W))
    b.init_walkers()
    ws = [vmc.Walker(tps, cfgs[w], trunc) for w in range(W)]
    a0 = b.amplitudes_c()
    r0 = np.array([w_.amplitude for w_ in ws])
    assert np.max(np.abs(a0 / r0 - 1)) < tol, np.max(np.abs(a0 / r0 - 1))
    worst = dict(amp=0.0, eloc=0.0, ostar=0.0, acc=0.0)
    b.zero_accumulators()
    osum = np.zeros(b.tps_size, dtype=complex)
    eosum = np.zeros(b.tps_size, dtype=complex)
    like = SplitIndexTPS(tps)
    for it in range(nsweeps):
        acc = b.sweep(1)
        racc = np.array([ups[w].sweep(tps, ws[w])[0] for w in range(W)])
        c = b.get_configs()
        for w in range(W):
            assert np.array_equal(c[w], ws[w].config), (it, w)
        assert np.array_equal(acc, racc)
        amp = b.amplitudes_c()
        ramp = np.array([w_.amplitude for w_ in ws])
        worst["amp"] = max(worst["amp"], float(np.max(np.abs(amp / ramp - 1))))
        e, psi = b.energy_and_holes(True, True)
        holes = b.holes_c()
        b.accumulate_ostar()
        for w in range(W):
            re, rh, pp = model.energy_and_holes(tps, ws[w], True)
            worst["eloc"] = max(worst["eloc"], abs(e[w] - re) / max(1.0, abs(re)))
            worst["psi"] = max(worst.get("psi", 0.0), float(np.max(np.abs(psi[:len(pp), w] / np.array(pp) - 1))))
            ost_ref = flat_holes(rh, rows, cols) * np.conj(1.0 / ws[w].amplitude)          # inverse_amplitude * holes (:245-272)
            ost = np.conj(holes[w] / amp[w])
            worst["ostar"] = max(worst["ostar"], float(np.max(np.abs(ost - ost_ref)) / np.max(np.abs(ost_ref))))
            off = hoff = 0
            for r in range(rows):
                for cc in range(cols):
                    sz = tps[r][cc][0].size
                    s_ = int(ws[w].config[r, cc])
                    osum[off + s_ * sz: off + (s_ + 1) * sz] += ost_ref[hoff:hoff + sz]
                    eosum[off + s_ * sz: off + (s_ + 1) * sz] += np.conj(re) * ost_ref[hoff:hoff + sz]
                    off += phys * sz
                    hoff += sz
    go, geo = b.accumulators_c()
    worst["acc"] = max(float(np.max(np.abs(go - osum)) / np.max(np.abs(osum))), float(np.max(np.abs(geo - eosum)) / np.max(np.abs(eosum))))
    assert all(v < tol for v in worst.values()), worst
    b.close()
    return worst


def run_complex_k5_golden(lib):
    """K5 (complex) through the C ABI: exact summation over the six S_z = 0 configurations of the reference's 2x2 complex
    Heisenberg fixture with device amplitudes / E_loc / holes: energy -2 and the reference's gradient signatures
    kGradNorm = 2.277663798157925e-08, kGradProbe = (7.37963070602707e-09, 1.708247848617349e-10)
    (tests/test_algorithm/test_exact_summation_evaluator.cpp:578-597; their tolerance is 1e-8 absolute, here relative)."""
    import itertools
    from helpers import load_golden_tps
    tps, z = load_golden_tps("heis2x2_complex_lowest")
    cfgs = np.stack([np.array(p).reshape(2, 2) for p in sorted(set(itertools.permutations([0, 0, 1, 1])))])
    W = len(cfgs)
    D = max(max(x.shape) for row in tps for site in row for x in site)
    b = WalkerBatch(2, 2, 2, D, W, BMPSTruncateParams.SVD(1, 1000, 0.0), lib=lib)
    b.set_complex()
    b.set_tps(SplitIndexTPS(tps))
    b.set_configs(cfgs)
    b.init_walkers()
    b.energy_and_holes(True)
    amp, e, holes = b.amplitudes_c(), b.eloc_c(), b.holes_c()
    wt = np.abs(amp) ** 2
    energy = np.sum(wt * e) / np.sum(wt)
    assert abs(energy - float(z["exp_energy"])) < float(z["exp_energy_tol"])
    s_o = np.zeros(b.tps_size, dtype=complex)
    s_eo = np.zeros(b.tps_size, dtype=complex)
    for w in range(W):
        off = hoff = 0
        for r in range(2):
            for c in range(2):
                sz = tps[r][c][0].size
                s_ = int(cfgs[w, r, c])
                inc = amp[w] * np.conj(holes[w, hoff:hoff + sz])
                s_o[off + s_ * sz: off + (s_ + 1) * sz] += inc
                s_eo[off + s_ * sz: off + (s_ + 1) * sz] += np.conj(e[w]) * inc
                off += 2 * sz
                hoff += sz
    grad = (s_eo - np.conj(energy) * s_o) / np.sum(wt)
    gn = float(np.sum(np.abs(grad) ** 2))
    assert abs(gn / float(z["exp_grad_norm"]) - 1) < 1e-5, (gn, float(z["exp_grad_norm"]))
    probe = 0.0
    off = 0
    for r in range(2):
        for c in range(2):
            for i in range(2):
                sz = tps[r][c][i].size
                base = complex(0.012 * ((r + 1) * 11 + (c + 1) * 5 + (i + 1) * 2), 0.0025 * ((r + 1) + (i + 1)))
                t = grad[off:off + sz]
                probe = probe + np.sum(np.conj(t) * (t * base))
                off += sz
    assert abs(probe.real / float(z["exp_grad_probe_re"]) - 1) < 1e-5 and abs(probe.imag / float(z["exp_grad_probe_im"]) - 1) < 1e-5
    b.close()


def run_complex_k8_goldens(lib):
    """K8 in QLTEN_Complex through the C ABI: exact summation with device amplitudes / E_loc over the reference's complex fZ2
    fixtures (tests/test_algorithm/test_exact_summation_evaluator.cpp:137-151, 353-425, 807): the spinless-fermion energies
    for t2 = 2.1 / 0 / -2.5 (simple-update and lowest states) and the t-J energy."""
    from test_fermion_oracle import load_golden, perms
    from peps_b200.api import FermionSplitIndexTPS, TableModel
    out = {}
    cases = [(f"sf2x2_t2_{t2:+.1f}_complex_{kind}", TableModel.spinless_fermion(1.0, t2, 0.0), [0, 0, 1, 1], (8, 8, 1e-16))
             for t2 in (2.1, 0.0, -2.5) for kind in ("su", "lowest")]
    cases += [(f"tj2x2_complex_{kind}", TableModel.tj(1.0, 0.3, V=0.3 / 4, mu=0.0), [0, 1, 2, 2], (4, 4, 0.0)) for kind in ("su", "lowest")]
    for name, model, occ, trunc in cases:
        f, z = load_golden(name)
        cfgs = np.stack(perms(occ, 2, 2))
        ftps = FermionSplitIndexTPS(f.T, f.par, f.phys_par)
        assert np.iscomplexobj(ftps.t[0][0][0])
        b = WalkerBatch(2, 2, len(f.phys_par), ftps.bond_dim(), len(cfgs), BMPSTruncateParams.SVD(*trunc), lib=lib)
        b.set_complex()
        b.set_fermion(ftps)
        b.set_tps(ftps)
        b.set_model(model)
        b.set_configs(cfgs)
        b.init_walkers()
        e = b.energy_and_holes(False)
        w = np.abs(b.amplitudes_c()) ** 2
        energy = np.sum(w * e) / np.sum(w)
        out[name] = energy
        tol = float(z["exp_energy_tol"])                      # the reference test's own tolerance for this fixture
        assert abs(energy.real - float(z["exp_energy"])) < tol and abs(energy.imag) < tol, (name, energy, float(z["exp_energy"]))
        b.close()
    return out


def run_complex_measure_parity(lib, j2=0.5, fermion=False):
    """EvaluateObservables on a complex state: every (complex) bond energy, the row correlator channels and the energy
    against the oracle; the arrays cross the ABI as planes."""
    rows, cols, D, W = 3, 4, 2, 3
    from peps_b200.api import SquareSpinOneHalfJ1J2XXZModelOBC
    tps = complex_tps(rows, cols, D, 31)
    cfgs = np.stack([vmc.shuffled_half_filled_config(rows, cols, 70 + w) for w in range(W)])
    b = WalkerBatch(rows, cols, 2, D, W, BMPSTruncateParams.SVD(4, 4, 0.0), lib=lib)
    b.set_complex()
    b.set_tps(SplitIndexTPS(tps))
    b.set_configs(cfgs)
    b.set_model(SquareSpinOneHalfJ1J2XXZModelOBC(1.0, 0.8, j2, 0.7 * j2, 0.3))
    b.init_walkers()
    obs = b.measure()
    model = vmc.XXZModel(1.0, 0.8, 0.3, j2, 0.7 * j2)
    for w in range(W):
        ref = model.measure(tps, vmc.Walker(tps, cfgs[w], (4, 4, 0.0)))
        for k, v in ref.items():
            assert np.allclose(obs[k][w], v, rtol=1e-10, atol=1e-12), (k, w)
    assert np.max(np.abs(obs["bond_energy_h"].imag)) > 1e-3                # genuinely complex records
    e = b.energy_and_holes(False)
    assert np.allclose(e, obs["energy"], rtol=1e-12)
    b.close()


def run_complex_sr(lib, rows=3, cols=3, D=2, W=3, n=4, chi=4, diag_shift=1e-3):
    """SR on a complex state: the store keeps the real embedding of the O* samples (x = [o_r; o_i], y = J x), the matvec and the
    CG run with the real kernels on planar vectors. Checked against the dense Hermitian S = <(O - Obar)(O - Obar)^H> of the
    oracle chain (SRSMatrix::operator* with the conjugating SplitIndexTPS inner product) and its dense solve."""
    from oracle import sr as osr
    from peps_b200 import sr
    from peps_b200.api import (MCEnergyGradEvaluator, MonteCarloParams, SquareSpinOneHalfXXZModelOBC, MCUpdateSquareNNExchange)
    tps_l = complex_tps(rows, cols, D, 8)
    tps = SplitIndexTPS(tps_l)
    cfgs = np.stack([vmc.shuffled_half_filled_config(rows, cols, 60 + w) for w in range(W)])
    mc = MonteCarloParams(num_samples=n * W, num_warmup_sweeps=0, sweeps_between_samples=1, is_warmed_up=True)
    ev = MCEnergyGradEvaluator(mc, BMPSTruncateParams.SVD(chi, chi, 0.0), tps, SquareSpinOneHalfXXZModelOBC(1, 1, 0),
                               MCUpdateSquareNNExchange(31), walkers=W, configs=cfgs, lib=lib)
    res = ev.Evaluate(collect_sr_buffers=True)
    assert ev.batch.sr_count() == n * W and res.total_samples == n * W
    model = vmc.XXZModel()
    ostars = []
    for w in range(W):
        wk = vmc.Walker(tps_l, cfgs[w], (chi, chi, 0.0))
        up = vmc.NNExchangeUpdater(31 + w)
        for _ in range(n):
            up.sweep(tps_l, wk)
            _, holes, _ = model.energy_and_holes(tps_l, wk, True)
            inv = np.conj(1.0 / wk.amplitude)
            sample = {(r, c): (int(wk.config[r, c]), holes[r][c] * inv) for r in range(rows) for c in range(cols)}
            ostars.append(osr.dense_ostar(sample, tps_l))
    o = np.stack(ostars)
    obar = o.mean(axis=0)
    assert np.max(np.abs(res.Ostar_mean.pack() - obar)) < 1e-12 * np.max(np.abs(obar))
    rng = np.random.default_rng(0)
    v = rng.standard_normal(obar.size) + 1j * rng.standard_normal(obar.size)
    # S v = (1/N) sum_i (<O_i, v> - <Obar, v>) O_i + shift v,  <a, b> = sum conj(a) b   (stochastic_reconfiguration_smatrix.h:45-91)
    ref = sum((np.vdot(oi, v) - np.vdot(obar, v)) * oi for oi in o) / len(o) + diag_shift * v
    smat = sr.SRSMatrix(ev.batch, res.Ostar_mean.pack(), res.total_samples, diag_shift)
    assert np.max(np.abs(smat(v) - ref)) < 1e-11 * np.max(np.abs(ref))
    g = res.gradient.pack()
    params = sr.ConjugateGradientParams(max_iter=300, relative_tolerance=1e-10)
    nat, iters, resid = ev.CalculateNaturalGradient(res, diag_shift, params)
    oc = o - obar
    s_dense = oc.T @ oc.conj() / len(o) + diag_shift * np.eye(obar.size)      # S_ab = <(O - Obar)_a conj((O - Obar)_b)>
    x_dense = np.linalg.solve(s_dense, g)
    assert np.max(np.abs(nat.pack() - x_dense)) < 1e-6 * np.max(np.abs(x_dense)), np.max(np.abs(nat.pack() - x_dense)) / np.max(np.abs(x_dense))
    return iters


def run_tj_pairing_parity(lib, rows=3, cols=4, D=2, W=4, trunc=(4, 4, 0.0), complex_=False, tol=1e-10):
    """t-J model with a singlet-pair pinning field (SetSingletPairPinningField, square_tJ_model.h:86-137, 256-289) and the
    bond-singlet SC observable (EvaluateBondSC -> SC_bond_singlet_h / _v, base/square_nnn_model_measurement_solver.h:116-131)
    through the C ABI in fermion mode against oracle/fermion.py (pair rule checked against the graded contraction):
    pinned E_loc, the difference to the unpinned model = delta * (delta_dag + delta) on that bond, and (conj(delta_dag) +
    delta) / 2 on every bond."""
    from oracle import fermion as F
    from peps_b200.api import FermionSplitIndexTPS, TableModel
    phys_par = (1, 1, 0)
    f = F.FermionTPS.random(rows, cols, D, 23, phys_par=phys_par, complex_=complex_)
    ftps = FermionSplitIndexTPS(f.T, f.par, phys_par)
    rng = np.random.default_rng(8)
    cfgs = []
    while len(cfgs) < W:                                   # any even-parity configuration: empty pairs and up/down pairs occur
        c = rng.integers(0, 3, size=(rows, cols))
        if f.parities(c).sum() % 2 == 0:
            cfgs.append(c)
    cfgs = np.stack(cfgs)
    delta = 0.07
    worst = 0.0
    dd, d = TableModel.tj_singlet_pair_tables()
    for pin in (((0, 1), (0, 0)), ((1, 2), (2, 2))):       # a horizontal bond (sites given in reverse order) and a vertical one
        b = WalkerBatch(rows, cols, 3, D, W, BMPSTruncateParams.SVD(*trunc), lib=lib)
        if complex_:
            b.set_complex()
        b.set_fermion(ftps)
        b.set_tps(ftps)
        b.set_configs(cfgs)
        b.init_walkers()
        base = TableModel.tj(1.0, 0.3, mu=0.2)
        b.set_model(base)
        e0 = b.energy_and_holes(False)
        pinned = TableModel.tj(1.0, 0.3, mu=0.2).SetSingletPairPinningField(pin[0], pin[1], delta)
        b.set_model(pinned)
        e1 = b.energy_and_holes(False)
        sc_h, sc_v = b.measure_sc_bond_singlet()
        assert np.array_equal(b.energy_and_holes(False), e1)                 # the observable leaves the model untouched
        b.set_model(pinned.ClearSingletPairPinningField())
        assert np.array_equal(b.energy_and_holes(False), e0)
        a_, b_ = sorted(pin)
        omodel = F.tJModel(1.0, 0.3, mu=0.2)
        opinned = F.tJModel(1.0, 0.3, mu=0.2)
        opinned.pin = (a_, b_, delta * (dd + d))
        for w in range(W):
            wk = F.FermionWalker(f, cfgs[w], trunc)
            r0 = omodel.energy_and_holes(wk, False)[0]
            r1 = opinned.energy_and_holes(wk, False)[0]
            worst = max(worst, abs(e0[w] - r0) / max(1.0, abs(r0)), abs(e1[w] - r1) / max(1.0, abs(r1)))
            hdd, vdd = omodel.measure_bond_table(dd, wk)
            hd, vd = omodel.measure_bond_table(d, wk)
            rh, rv = (np.conj(hdd) + hd) / 2, (np.conj(vdd) + vd) / 2
            worst = max(worst, float(np.max(np.abs(sc_h[w] - rh))), float(np.max(np.abs(sc_v[w] - rv))))
            src = (hdd + hd)[a_] if a_[0] == b_[0] else (vdd + vd)[a_]   # the pinned energy adds delta * (delta_dag + delta) on the bond
            assert abs((e1[w] - e0[w]) - delta * src) < 1e-10
        assert np.max(np.abs(sc_h)) + np.max(np.abs(sc_v)) > 1e-3
        b.close()
    assert worst < tol, worst
    # a bond outside the lattice is an error (ValidateSingletPairPinningBondInLattice_)
    from peps_b200.api import PepsError
    b = WalkerBatch(rows, cols, 3, D, 1, BMPSTruncateParams.SVD(*trunc), lib=lib)
    b.set_fermion(ftps)
    try:
        b.set_model(TableModel.tj(1.0, 0.3).SetSingletPairPinningField((rows, 0), (rows, 1), delta))
        raise AssertionError("out-of-lattice pin accepted")
    except PepsError:
        pass
    b.close()
    return worst


def run_boson_bond_observable_parity(lib):
    """peps_measure_bond_term on a bosonic context: the XXZ bond operator as a table reproduces the per-bond energies of the
    built-in measurement, for a table model too (whose measure() now records its bond energies)."""
    from peps_b200.api import SquareSpinOneHalfXXZModelOBC, TableModel
    rows, cols, D, W = 3, 4, 2, 3
    tps = vmc.random_tps(rows, cols, 2, D, seed=31)
    cfgs = np.stack([vmc.shuffled_half_filled_config(rows, cols, 70 + w) for w in range(W)])
    b = WalkerBatch(rows, cols, 2, D, W, BMPSTruncateParams.SVD(4, 4, 0.0), lib=lib)
    b.set_tps(SplitIndexTPS(tps)); b.set_configs(cfgs); b.init_walkers()
    b.set_model(SquareSpinOneHalfXXZModelOBC(1.0, 0.8, 0.0))
    obs = b.measure()
    oh, ov = b.measure_bond_observable(TableModel.xxz(1.0, 0.8).h2)
    assert np.allclose(oh, obs["bond_energy_h"], rtol=1e-12, atol=1e-13) and np.allclose(ov, obs["bond_energy_v"], rtol=1e-12, atol=1e-13)
    b.set_model(TableModel.xxz(1.0, 0.8, 0.5, 0.35))
    obs_t = b.measure()
    b.set_model(__import__("peps_b200.api", fromlist=["x"]).SquareSpinOneHalfJ1J2XXZModelOBC(1.0, 0.8, 0.5, 0.35, 0.0))
    obs_b = b.measure()
    for k in ("energy", "bond_energy_h", "bond_energy_v", "bond_energy_dr", "bond_energy_ur"):
        assert np.allclose(obs_t[k], obs_b[k], rtol=1e-12, atol=1e-13), k
    b.close()


def run_tfim_measure_parity(lib, complex_=False):
    """TransverseFieldIsingSquareOBC::EvaluateObservables through peps_measure_site_term: sigma_x per site, energy, spin_z and
    SzSz_row against the oracle; the model state is untouched."""
    from peps_b200.api import TransverseFieldIsingSquareOBC, MCPEPSMeasurer, MCUpdateSquareNNFullSpaceUpdate
    from peps_b200.api import MonteCarloParams, Configuration
    rows, cols, D, W = 3, 4, 2, 3
    tps = complex_tps(rows, cols, D, 31) if complex_ else vmc.random_tps(rows, cols, 2, D, seed=31)
    cfgs = np.stack([vmc.shuffled_half_filled_config(rows, cols, 70 + w) for w in range(W)])
    b = WalkerBatch(rows, cols, 2, D, W, BMPSTruncateParams.SVD(4, 4, 0.0), lib=lib)
    if complex_:
        b.set_complex()
    b.set_tps(SplitIndexTPS(tps)); b.set_configs(cfgs); b.init_walkers()
    b.set_model(TransverseFieldIsingSquareOBC(0.7))
    e0 = b.energy_and_holes(False)
    obs = b.measure_tfim()
    model = vmc.TFIMModel(0.7)
    for w in range(W):
        ref = model.measure(tps, vmc.Walker(tps, cfgs[w], (4, 4, 0.0)))
        for k, v in ref.items():
            assert np.allclose(obs[k][w], v, rtol=1e-10, atol=1e-12), (k, w)
    assert np.array_equal(b.energy_and_holes(False), e0)
    # E = diagonal part - h sum sigma_x (transverse_field_ising_square_obc.h:95-122)
    diag = np.array([model.diag_energy(cfgs[w]) for w in range(W)])
    assert np.allclose(obs["energy"], diag - 0.7 * obs["sigma_x"].sum(axis=(1, 2)), rtol=1e-11)
    b.close()
    out = MCPEPSMeasurer(MonteCarloParams(6, 0, 1, Configuration(cfgs[0]), True), BMPSTruncateParams.SVD(4, 4, 0.0), SplitIndexTPS(tps),
                         TransverseFieldIsingSquareOBC(0.7), MCUpdateSquareNNFullSpaceUpdate(seed=3), 3, lib=lib).Execute()
    assert set(out) == {"energy", "spin_z", "sigma_x", "SzSz_row"} and out["sigma_x"][0].shape == (rows, cols)


def ipeps_tj_state(rows, cols):
    """An OBC t-J state tiled from the reference's iPEPS unit cell (tests/golden/ipeps_tj_ab.npz, re-packed from
    tests/test_data/ipeps_tJ_t{a,b}_doping0.125.qlten): tensor a / b on the two sublattices, boundary legs reduced to dimension 1
    by the dominant singular vector, NormalizeAllSite, times 3 -- the construction of ProjectedtJTensorNetwork
    (tests/test_2d_tn/test_bmps_contractor.cpp:762-847) except that the boundary vector is taken from the EVEN sector of the
    leg (the reference keeps the overall dominant one, which is odd for a's R and b's L leg; boundary legs are even here).
    Returns an oracle FermionTPS with phys = (up, down, empty)."""
    import os
    from oracle import fermion as F
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "ipeps_tj_ab.npz"))
    bp = z["leg_par"][0].astype(np.int32)
    assert all((z["leg_par"][k] == bp).all() for k in range(4)) and list(bp) == [0, 0, 1, 1] and list(z["phys_par"]) == [1, 1, 0]
    one = np.zeros(1, dtype=np.int32)

    def project(t, axis):
        m = np.moveaxis(t, axis, 0).reshape(t.shape[axis], -1)
        _, _, vt = np.linalg.svd(m[bp == 0], full_matrices=False)
        return np.moveaxis(vt[0].reshape((1,) + tuple(np.delete(t.shape, axis))), 0, axis)

    T = [[None] * cols for _ in range(rows)]
    P = [[None] * cols for _ in range(rows)]
    for r in range(rows):
        for c in range(cols):
            t = np.array(z["ta"] if (r + c) % 2 == 0 else z["tb"])
            pars = [bp, bp, bp, bp]
            if r == 0:
                t, pars[3] = project(t, 3), one
            elif r == rows - 1:
                t, pars[1] = project(t, 1), one
            if c == 0:
                t, pars[0] = project(t, 0), one
            elif c == cols - 1:
                t, pars[2] = project(t, 2), one
            mx = np.max(np.abs(t))
            T[r][c] = [np.ascontiguousarray(t[..., s_]) * (3.0 / mx) for s_ in range(3)]
            P[r][c] = pars
    return F.FermionTPS(T, P, (1, 1, 0))


def doped_tj_configs(rows, cols, W, seed=0):
    """1/8 hole doping, equal numbers of up and down spins (even electron number), one shuffle per walker."""
    n = rows * cols
    holes = n // 8 + ((n - n // 8) % 2)
    ne = n - holes
    base = np.array([0] * (ne // 2) + [1] * (ne - ne // 2) + [2] * holes)
    return np.stack([np.random.default_rng(seed + w).permutation(base).reshape(rows, cols) for w in range(W)])
