"""oracle/make_golden.py -- TEST INFRASTRUCTURE.

Runs the UNMODIFIED reference (/root/reference, via oracle/ref_loader.py) and the
oracle restatement on identical seeded float64 inputs, asserts they agree, and writes the
reference's outputs as small fixtures under tests/golden/.  /root/reference does not
exist on the GPU box, so the fixtures (plus this script) are what travels.

    python -m oracle.make_golden            # from the repo root, in the build container
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import ref_loader, dsp_oracle as O, detect_oracle as D  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
DX = 2.0419046878814697   # OOI RCA channel spacing, DAS4Whales_ExampleNotebook.md:224-230
FS = 200.0


def synth(nx, ns, seed, dx=DX, fs=FS, ncalls=3):
    """Seeded noise + hyperbolic-moveout chirps (SURVEY.md 8d), float64."""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((nx, ns))
    L = min(int(0.68 * fs), ns // 4)
    t = np.arange(L) / fs
    import scipy.signal as sps
    c = sps.chirp(t, f0=28.8, f1=17.8, t1=0.68, method="hyperbolic") * np.hanning(L)
    for _ in range(ncalls):
        c0 = rng.integers(0, nx)
        t0 = rng.uniform(0, ns / fs * 0.6)
        for ch in range(nx):
            d = np.sqrt(((ch - c0) * dx) ** 2 + 500.0 ** 2) / 1500.0
            i0 = int((t0 + d) * fs)
            if i0 + L <= ns:
                x[ch, i0:i0 + L] += 3.0 * c
    return x


def close(a, b, tol=1e-12, what=""):
    a = np.asarray(a); b = np.asarray(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    den = max(np.max(np.abs(a)), 1e-300)
    err = np.max(np.abs(a - b)) / den
    assert err <= tol, f"{what}: oracle vs reference rel err {err:.3e} > {tol}"
    return err


def main():
    os.makedirs(OUT, exist_ok=True)
    dsp, detect = ref_loader.load()
    rep = {}

    # ---- masks (a1, a2) -------------------------------------------------------------
    masks = {}
    for (nx, ns, step) in [(40, 240, 1), (45, 175, 1), (38, 120, 2)]:
        sel = [0, nx * step, step]
        r = dsp.fk_filter_design((nx, ns), sel, DX, FS, 1400, 1450, 3400, 3500)
        o = O.fk_filter_design((nx, ns), sel, DX, FS, 1400, 1450, 3400, 3500)
        rep[f"fan_{nx}x{ns}"] = close(r, o, what="fk_filter_design")
        masks[f"fan_{nx}x{ns}_s{step}"] = np.ascontiguousarray(r)
    for (nx, ns) in [(40, 240), (38, 120)]:
        sel = [0, nx, 1]
        r = np.asarray(dsp.hybrid_ninf_filter_design((nx, ns), sel, DX, FS, 1350., 1450., 3300, 3450, 14., 30.))
        o = O.hybrid_ninf_filter_design((nx, ns), sel, DX, FS, 1350., 1450., 3300, 3450, 14., 30.)
        rep[f"ninf_{nx}x{ns}"] = close(r, o, what="hybrid_ninf_filter_design")
        masks[f"ninf_{nx}x{ns}"] = r
        r = np.asarray(dsp.hybrid_filter_design((nx, ns), sel, DX, FS, 1400., 1450., 15., 25.))
        o = O.hybrid_filter_design((nx, ns), sel, DX, FS, 1400., 1450., 15., 25.)
        rep[f"hyb_{nx}x{ns}"] = close(r, o, what="hybrid_filter_design")
        masks[f"hyb_{nx}x{ns}"] = r
    for (nx, ns) in [(40, 240)]:
        sel = [0, nx, 1]
        r = np.asarray(dsp.hybrid_gs_filter_design((nx, ns), sel, DX, FS, 1400., 1450., 15., 25.))
        rep[f"gs_{nx}x{ns}"] = close(r, O.hybrid_gs_filter_design((nx, ns), sel, DX, FS, 1400., 1450., 15., 25.), what="hybrid_gs")
        masks[f"gs_{nx}x{ns}"] = r
        r = np.asarray(dsp.hybrid_ninf_gs_filter_design((nx, ns), sel, DX, FS, 1400., 1450., 3400, 3500, 15., 25.))
        rep[f"ninfgs_{nx}x{ns}"] = close(r, O.hybrid_ninf_gs_filter_design((nx, ns), sel, DX, FS, 1400., 1450., 3400, 3500, 15., 25.), what="hybrid_ninf_gs")
        masks[f"ninfgs_{nx}x{ns}"] = r
    xl = synth(40, 240, seed=77)
    rl = dsp.fk_filt(xl, 1, FS, 1, DX, 1450., 3400.)
    rep["fk_filt_legacy"] = close(rl, O.fk_filt(xl, 1, FS, 1, DX, 1450., 3400.), what="legacy fk_filt")
    masks["legacy_x"], masks["legacy_y"] = xl, rl
    np.savez_compressed(os.path.join(OUT, "masks.npz"), **masks)

    # ---- f-k apply (a3-a5) ----------------------------------------------------------
    fk = {}
    for tag, nx, ns, mkey, taper in [("fan_even", 40, 240, "fan_40x240_s1", False),
                                     ("fan_odd", 45, 175, "fan_45x175_s1", True),
                                     ("fan_p19", 38, 120, "fan_38x120_s2", False),
                                     ("ninf_even", 40, 240, "ninf_40x240", False),
                                     ("hyb_even", 38, 120, "hyb_38x120", True)]:
        x = synth(nx, ns, seed=11 + nx + ns)
        m = masks[mkey]
        r = dsp.fk_filter_filt(x.copy(), m, tapering=taper)
        o = O.fk_filter_filt(x.copy(), m, tapering=taper)
        rep["fk_" + tag] = close(r, o, what="fk_filter_filt " + tag)
        # the folded-mask / half-spectrum identity the GPU path relies on (SURVEY App. A.1)
        o2 = O.fk_filter_filt_rows(x.copy(), m, rows=np.arange(nx), tapering=taper)
        rep["fkfold_" + tag] = close(r, o2, tol=1e-10, what="folded route " + tag)
        fk[tag + "_x"] = x
        fk[tag + "_y"] = r
        fk[tag + "_mask"] = np.array(mkey)
        fk[tag + "_taper"] = np.array(taper)
    # reference KAT: tests/test_dsp.py:85-88
    t5 = dsp.taper_data(np.array([[1., 2, 3, 4, 5], [1, 2, 3, 4, 5]]))
    assert np.array_equal(t5, np.array([[0., 2, 3, 4, 0], [0, 2, 3, 4, 0]]))
    fk["kat_taper"] = t5
    np.savez_compressed(os.path.join(OUT, "fk_apply.npz"), **fk)

    # ---- IIR (a6, a7) ---------------------------------------------------------------
    iir = {}
    x = synth(6, 900, seed=5)
    r = dsp.bp_filt(x, FS, 14, 30)
    rep["bp_filt"] = close(r, O.bp_filt(x, FS, 14, 30), what="bp_filt")
    iir["bp_x"], iir["bp_y"] = x, r
    import scipy.signal as sps
    sos = dsp.butterworth_filter([5, [10, 30], "bp"], FS)
    close(sos, O.butterworth_filter([5, [10, 30], "bp"], FS), what="butterworth_filter")
    iir["sos_bp5"] = sos
    iir["sos_bp5_y"] = sps.sosfiltfilt(sos, x, axis=1)
    sos2 = dsp.butterworth_filter([2, 5, "hp"], FS)
    iir["sos_hp2"] = sos2
    iir["sos_hp2_y"] = sps.sosfiltfilt(sos2, x, axis=1)
    np.savez_compressed(os.path.join(OUT, "iir.npz"), **iir)

    # ---- SNR / envelope (a13) ---------------------------------------------------------
    sn = {}
    kat_in = np.array([[1., 2, 3, 4, 5], [1, 2, 3, 4, 5]])
    kat = dsp.snr_tr_array(kat_in)
    assert np.allclose(kat[0], [-3.01029996, 3.01029996, 6.53212514, 9.03089987, 10.96910013])  # tests/test_dsp.py:136-141
    rep["snr_kat"] = close(kat, O.snr_tr_array(kat_in), what="snr KAT")
    x = synth(5, 600, seed=9)
    for env in (False, True):
        r = dsp.snr_tr_array(x, env=env)
        rep[f"snr_env{env}"] = close(r, O.snr_tr_array(x, env=env), tol=1e-10, what="snr_tr_array")
        sn[f"snr_env{int(env)}"] = r
    sn["x"], sn["kat_in"], sn["kat"] = x, kat_in, kat
    np.savez_compressed(os.path.join(OUT, "snr.npz"), **sn)

    # ---- matched filter (a9-a11, a14) -------------------------------------------------
    mf = {}
    ns = 1600
    time = np.arange(ns) / FS
    x = synth(6, ns, seed=21)
    for tag, (f0, f1, dur) in {"hf": (17.8, 28.8, 0.68), "lf": (14.7, 21.8, 0.78)}.items():
        tpl = detect.gen_template_fincall(time, FS, f0, f1, dur)
        rep["tpl_" + tag] = close(tpl, D.gen_template_fincall(time, FS, f0, f1, dur), what="template")
        r = detect.compute_cross_correlogram(x, tpl)
        rep["xc_" + tag] = close(r, D.compute_cross_correlogram(x, tpl), what="cross_correlogram")
        rep["xcdirect_" + tag] = close(r, D.compute_cross_correlogram_direct(x, tpl), tol=1e-10, what="A.3 identity")
        mf["tpl_" + tag], mf["corr_" + tag] = tpl, r
        import scipy.signal as sps
        mf["env_" + tag] = np.abs(sps.hilbert(r, axis=1))
        pk = detect.pick_times_env(r, 0.05)
        po = D.pick_times_env(r, 0.05)
        assert all(np.array_equal(a, b) for a, b in zip(pk, po))
        mf["picks_" + tag] = detect.convert_pick_times(pk)
    mf["x"] = x
    mf["lin_chirp"] = detect.gen_linear_chirp(15., 25., 1.0, FS)
    close(mf["lin_chirp"], D.gen_linear_chirp(15., 25., 1.0, FS), what="linear chirp")
    a = np.array([1., 2, 3, 4, 5]); b = np.array([2., 1, 0, -1, 2])
    mf["sx"] = detect.shift_xcorr(a, b); mf["snx"] = detect.shift_nxcorr(a, b)
    close(mf["sx"], D.shift_xcorr(a, b)); close(mf["snx"], D.shift_nxcorr(a, b))
    np.savez_compressed(os.path.join(OUT, "matched_filter.npz"), **mf)

    # ---- spectrogram correlation pieces that do not need librosa (a12) ---------------
    sc = {}
    ff = np.linspace(0, FS / 2, 81)[12:32]
    tt = np.linspace(0, 8.0, 201)
    tv, fv, ker = detect.buildkernel(27., 16., 4., 0.9, ff, tt, FS, 12., 36.)
    _, _, ker_o = D.buildkernel(27., 16., 4., 0.9, ff, tt, FS, 12., 36.)
    rep["buildkernel"] = close(ker, ker_o, what="buildkernel")
    rng = np.random.default_rng(3)
    S = np.abs(rng.standard_normal((len(ff), 201)))
    r = detect.xcorr2d(S, ker)
    rep["xcorr2d"] = close(r, D.xcorr2d(S, ker), what="xcorr2d")
    sc.update(ff=ff, tt=tt, ker=ker, S=S, xc2d=r)
    np.savez_compressed(os.path.join(OUT, "spectrocorr.npz"), **sc)

    # ---- peak picking on the raw correlogram + ties / flat tops (a14) and raw2strain (8(f) rank 2) -----------
    pkf = {}
    rng = np.random.default_rng(11)
    xq = np.round(rng.standard_normal((8, 700)) * 3.0) / 3.0            # quantised: many exact ties and plateaus
    xq[3] = 0.25; xq[4] = np.arange(700) / 700.0; xq[5, 100:140] = 5.0
    for thr in (0.0, 0.4, 2.0):
        pk = detect.pick_times(xq, thr)
        assert all(np.array_equal(a, b) for a, b in zip(pk, D.pick_times(xq, thr)))
        pkf[f"picks_thr{thr}"] = detect.convert_pick_times(pk)
    pkf["x"] = xq
    np.savez_compressed(os.path.join(OUT, "picks.npz"), **pkf)
    from oracle import data_oracle as DH
    dh = ref_loader.load_data_handle()
    raw = rng.integers(-2 ** 20, 2 ** 20, size=(12, 500)).astype(np.int32)
    meta = {"scale_factor": 4.0838e-11 * 1550.0 / 2.0419}
    ref_strain = dh.raw2strain(raw.astype(np.float64), meta)              # the reference works in place on float arrays
    rep["raw2strain"] = close(ref_strain, DH.raw2strain(raw, meta), what="raw2strain")
    np.savez_compressed(os.path.join(OUT, "raw2strain.npz"), raw=raw, scale_factor=meta["scale_factor"], strain=ref_strain)

    rep.update(make_round2())
    rep.update(make_spot())
    for k, v in rep.items():
        print(f"{k:24s} oracle-vs-reference rel err {v:.2e}")
    tot = sum(os.path.getsize(os.path.join(OUT, f)) for f in os.listdir(OUT))
    print(f"golden fixtures written to {OUT} ({tot / 1024:.0f} KiB)")


def make_round2():
    """Fixtures added in round 2: spectral views / alternate correlators (views.npz) and the Gabor image detector
    (gabor.npz), again reference outputs with the oracle restatement asserted against them."""
    import cv2
    from oracle import improcess_oracle as IO
    dsp, detect = ref_loader.load()
    imp = ref_loader.load_improcess()
    rep = {}
    vw = {}
    rng = np.random.default_rng(77)
    # dsp.get_fx (dsp.py:18-38): crop (nfft < ns), exact (nfft == ns) and zero-pad (nfft > ns)
    xfx = synth(5, 600, seed=31)
    vw["fx_x"] = xfx
    for nfft in (512, 600, 1000):
        vw[f"fx_{nfft}"] = dsp.get_fx(xfx, nfft)
        rep[f"get_fx_{nfft}"] = close(vw[f"fx_{nfft}"], O.get_fx(xfx, nfft), what="get_fx")
    # dsp.instant_freq (dsp.py:830-856) on a chirp with a smooth envelope
    tt = np.arange(1200) / FS
    import scipy.signal as sps
    ch = sps.chirp(tt, f0=12.0, f1=30.0, t1=tt[-1], method="linear") * (1.0 + 0.3 * np.sin(2 * np.pi * 0.7 * tt))
    vw["if_x"] = ch
    vw["if_y"] = dsp.instant_freq(ch, FS)
    rep["instant_freq"] = close(vw["if_y"], O.instant_freq(ch, FS), what="instant_freq")
    # detect.shift_xcorr / shift_nxcorr with unequal lengths (detect.py:96-137)
    a = rng.standard_normal(300); b = rng.standard_normal(120); c = rng.standard_normal(420)
    vw.update(sx_a=a, sx_b=b, sx_c=c, sx_ab=detect.shift_xcorr(a, b), sx_ac=detect.shift_xcorr(a, c),
              snx_ab=detect.shift_nxcorr(a, b), snx_ac=detect.shift_nxcorr(a, c))
    close(vw["sx_ab"], D.shift_xcorr(a, b)); close(vw["sx_ac"], D.shift_xcorr(a, c))
    # detect.xcorr (detect.py:605-647), nxcorr2d (:544-576), process_corr (:198-218)
    ff = np.linspace(0, FS / 2, 81)[12:32]
    tgrid = np.linspace(0, 8.0, 201)
    tv, fv, ker = detect.buildkernel(27., 16., 4., 0.9, ff, tgrid, FS, 12., 36.)
    S = np.abs(rng.standard_normal((len(ff) + 5, 201)))
    t_scale, cv = detect.xcorr(tgrid, ff, S, tv, fv, ker)
    to, co = D.xcorr(tgrid, ff, S, tv, fv, ker)
    rep["xcorr"] = close(cv, co, what="detect.xcorr"); close(t_scale, to, what="detect.xcorr t_scale")
    nx2 = detect.nxcorr2d(S[:len(ff)], ker)
    rep["nxcorr2d"] = close(nx2, D.nxcorr2d(S[:len(ff)], ker), what="nxcorr2d")
    corr1 = synth(1, 1600, seed=41)[0] * 0.1
    pc = detect.process_corr(corr1, 0.05)
    assert np.array_equal(pc, D.process_corr(corr1, 0.05))
    vw.update(xc_t=tgrid, xc_f=ff, xc_S=S, xc_tvec=tv, xc_fvec=fv, xc_ker=ker, xc_tscale=t_scale, xc_val=cv, nxc2d=nx2,
              pc_x=corr1, pc_idx=pc)
    np.savez_compressed(os.path.join(OUT, "views.npz"), **vw)

    # ---- Gabor image detector (a15): improcess.py:44-63, :98-140, :395-454; scripts/main_gabordetect.py:78-169 ----------
    gb = {}
    nx, ns, sel = 400, 3000, [0, 400, 1]
    trf = synth(nx, ns, seed=5, ncalls=4)
    image = imp.trace2image(trf)
    rep["trace2image"] = close(image, IO.trace2image(trf), what="trace2image")
    theta = imp.angle_fromspeed(1500., FS, DX, sel)
    imagebin = imp.binning(image, 1 / 10, 1 / 10)
    rep["binning"] = close(imagebin, IO.binning(image, 1 / 10, 1 / 10), what="binning")
    up, down = imp.gabor_filt_design(theta, plot=False)
    uo, do = IO.gabor_filt_design(theta)
    close(up, uo, what="gabor up"); close(down, do, what="gabor down")
    fimage = cv2.filter2D(imagebin, cv2.CV_64F, up) + cv2.filter2D(imagebin, cv2.CV_64F, down)     # main_gabordetect.py:109
    thr = float(np.percentile(fimage, 90.0))
    binary = fimage > thr
    m2 = cv2.filter2D(binary.astype(float), cv2.CV_64F, up) + cv2.filter2D(binary.astype(float), cv2.CV_64F, down)   # :135
    thr2 = float(np.percentile(m2, 85.0))
    mask = m2 > thr2
    smoothed = imp.apply_smooth_mask(imagebin, mask)
    mask_sparse = imp.binning(mask, 10, 10)                                                          # :166
    masked = imp.apply_smooth_mask(trf, mask_sparse)                                                 # :169
    mo, parts = IO.gabor_detect(trf, FS, DX, sel, 1500., 10, thr, thr2)
    rep["gabor_fimage"] = close(fimage, parts["fimage"], what="gabor fimage")
    assert np.array_equal(mask, parts["mask"]) and np.array_equal(mask_sparse, parts["mask_sparse"])
    rep["gabor_masked"] = close(masked, mo, what="gabor masked trace")
    rows = np.array([0, 57, 133, 200, 311, 399])
    gb.update(seed=5, nx=nx, ns=ns, ncalls=4, x_checksum=float(np.sum(trf)), theta=theta, up=up, image_rows=image[rows], rows=rows,
              imagebin=imagebin, fimage=fimage, thr=thr, m2=m2, thr2=thr2, mask=mask, smoothed=smoothed,
              mask_sparse_bits=np.packbits(mask_sparse), masked_rows=masked[rows])
    np.savez_compressed(os.path.join(OUT, "gabor.npz"), **gb)
    return rep


def make_spot():
    """Reference outputs on the seeded white-noise inputs of the spot checks in tests/test_oracle_golden.py (spot.npz).
    Every third row of the larger 2-D outputs is stored, which keeps the file small."""
    from oracle import improcess_oracle as IO
    dsp, detect = ref_loader.load()
    imp = ref_loader.load_improcess()
    rep = {}
    sp = {}
    nx, ns = 36, 200
    x = np.random.default_rng(5).standard_normal((nx, ns))
    sel = [0, nx, 1]
    m = dsp.fk_filter_design((nx, ns), sel, DX, FS)
    assert np.array_equal(m, O.fk_filter_design((nx, ns), sel, DX, FS))
    y = dsp.fk_filter_filt(x.copy(), m, True)
    rep["spot_fk"] = close(y, O.fk_filter_filt(x.copy(), m, True), tol=1e-13, what="fk_filter_filt")
    h = np.asarray(dsp.hybrid_ninf_filter_design((nx, ns), sel, DX, FS))
    rep["spot_ninf"] = close(h, O.hybrid_ninf_filter_design((nx, ns), sel, DX, FS), tol=1e-13, what="hybrid_ninf")
    bp = dsp.bp_filt(x, FS, 14, 30)
    rep["spot_bp"] = close(bp, O.bp_filt(x, FS, 14, 30), tol=1e-13, what="bp_filt")
    tpl = detect.gen_template_fincall(np.arange(ns) / FS, FS, 17.8, 28.8, 0.68)
    xc = detect.compute_cross_correlogram(x, tpl)
    rep["spot_xc"] = close(xc, D.compute_cross_correlogram(x, tpl), tol=1e-13, what="cross_correlogram")
    sp.update(a_x_checksum=float(np.sum(x)), a_mask=m, a_ninf=h, a_tpl=tpl, a_fk_rows=y[::3], a_bp_rows=bp[::3], a_xc_rows=xc[::3])
    x = np.random.default_rng(8).standard_normal((30, 500))
    fx = dsp.get_fx(x, 256)
    rep["spot_get_fx"] = close(fx, O.get_fx(x, 256), tol=1e-14, what="get_fx")
    img = imp.trace2image(x)
    rep["spot_trace2image"] = close(img, IO.trace2image(x), tol=1e-13, what="trace2image")
    b = imp.binning(img, 0.1, 0.1)
    rep["spot_binning"] = close(b, IO.binning(img, 0.1, 0.1), tol=1e-13, what="binning")
    up, down = imp.gabor_filt_design(40.0)
    assert np.array_equal(up, IO.gabor_filt_design(40.0)[0]) and np.array_equal(down, np.flipud(up))
    sp.update(b_x_checksum=float(np.sum(x)), b_fx_rows=fx[::3], b_img_rows=img[::3], b_bin=b, b_up=up)
    np.savez_compressed(os.path.join(OUT, "spot.npz"), **sp)
    return rep


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] in ("round2", "spot"):
        for k, v in (make_round2() if sys.argv[1] == "round2" else make_spot()).items():
            print(f"{k:24s} oracle-vs-reference rel err {v:.2e}")
    else:
        main()
