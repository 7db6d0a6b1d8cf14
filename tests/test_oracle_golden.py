"""CPU: the oracle restatement against the committed golden vectors (outputs of the
UNMODIFIED reference, tests/golden/, made by oracle/make_golden.py)."""
import numpy as np
import pytest

from oracle import dsp_oracle as O, detect_oracle as D
from conftest import rel_err

DX = 2.0419046878814697
FS = 200.0


def test_masks_match_golden(golden):
    g = golden("masks")
    for key in g.files:
        if key.startswith("legacy"):
            continue
        kind, shape = key.split("_")[0], key.split("_")[1]
        nx, ns = (int(v) for v in shape.split("x"))
        step = int(key.split("_s")[1]) if "_s" in key else 1
        sel = [0, nx * step, step]
        if kind == "fan":
            m = O.fk_filter_design((nx, ns), sel, DX, FS, 1400, 1450, 3400, 3500)
        elif kind == "ninf":
            m = O.hybrid_ninf_filter_design((nx, ns), sel, DX, FS, 1350., 1450., 3300, 3450, 14., 30.)
        elif kind == "gs":
            m = O.hybrid_gs_filter_design((nx, ns), sel, DX, FS, 1400., 1450., 15., 25.)
        elif kind == "ninfgs":
            m = O.hybrid_ninf_gs_filter_design((nx, ns), sel, DX, FS, 1400., 1450., 3400, 3500, 15., 25.)
        else:
            m = O.hybrid_filter_design((nx, ns), sel, DX, FS, 1400., 1450., 15., 25.)
        assert np.max(np.abs(m - g[key])) <= 1e-13, key
    assert rel_err(O.fk_filt(g["legacy_x"], 1, FS, 1, DX, 1450., 3400.), g["legacy_y"])[0] <= 1e-12


def test_fk_apply_matches_golden(golden):
    g, gm = golden("fk_apply"), golden("masks")
    for tag in ("fan_even", "fan_odd", "fan_p19", "ninf_even", "hyb_even"):
        x, y = g[tag + "_x"], g[tag + "_y"]
        m = gm[str(g[tag + "_mask"])]
        taper = bool(g[tag + "_taper"])
        assert rel_err(O.fk_filter_filt(x.copy(), m, tapering=taper), y)[0] <= 1e-12
        # folded half-spectrum identity the CUDA path is built on
        assert rel_err(O.fk_filter_filt_rows(x.copy(), m, np.arange(x.shape[0]), tapering=taper), y)[0] <= 1e-10


def test_reference_known_answers(golden):
    # reference tests/test_dsp.py:85-88 and :136-141
    t = O.taper_data(np.array([[1., 2, 3, 4, 5], [1, 2, 3, 4, 5]]))
    assert np.array_equal(t, golden("fk_apply")["kat_taper"])
    assert np.array_equal(t, np.array([[0., 2, 3, 4, 0], [0, 2, 3, 4, 0]]))
    s = golden("snr")
    out = O.snr_tr_array(s["kat_in"])
    assert np.allclose(out[0], [-3.01029996, 3.01029996, 6.53212514, 9.03089987, 10.96910013])
    assert rel_err(out, s["kat"])[0] <= 1e-14


def test_iir_and_snr_match_golden(golden):
    g = golden("iir")
    assert rel_err(O.bp_filt(g["bp_x"], FS, 14, 30), g["bp_y"])[0] <= 1e-12
    assert rel_err(O.sosfiltfilt(g["sos_bp5"], g["bp_x"]), g["sos_bp5_y"])[0] <= 1e-12
    assert rel_err(O.butterworth_filter([5, [10, 30], "bp"], FS), g["sos_bp5"])[0] <= 1e-14
    s = golden("snr")
    for env in (0, 1):
        a, b = O.snr_tr_array(s["x"], env=bool(env)), s[f"snr_env{env}"]
        assert np.max(np.abs(a - b)) <= 1e-9


def test_matched_filter_matches_golden(golden):
    g = golden("matched_filter")
    x = g["x"]
    time = np.arange(x.shape[1]) / FS
    for tag, (f0, f1, dur) in {"hf": (17.8, 28.8, 0.68), "lf": (14.7, 21.8, 0.78)}.items():
        tpl = D.gen_template_fincall(time, FS, f0, f1, dur)
        assert rel_err(tpl, g["tpl_" + tag])[0] <= 1e-14
        assert rel_err(D.compute_cross_correlogram(x, tpl), g["corr_" + tag])[0] <= 1e-12
        assert rel_err(D.compute_cross_correlogram_direct(x, tpl), g["corr_" + tag])[0] <= 1e-10
        assert rel_err(D.envelope(g["corr_" + tag]), g["env_" + tag])[0] <= 1e-12
        picks = D.convert_pick_times(D.pick_times_env(g["corr_" + tag], 0.05))
        assert np.array_equal(picks, g["picks_" + tag])
    assert rel_err(D.gen_linear_chirp(15., 25., 1.0, FS), g["lin_chirp"])[0] <= 1e-14
    a = np.array([1., 2, 3, 4, 5]); b = np.array([2., 1, 0, -1, 2])
    assert rel_err(D.shift_xcorr(a, b), g["sx"])[0] <= 1e-14
    assert rel_err(D.shift_nxcorr(a, b), g["snx"])[0] <= 1e-14


def test_spectrocorr_pieces_match_golden(golden):
    g = golden("spectrocorr")
    _, _, ker = D.buildkernel(27., 16., 4., 0.9, g["ff"], g["tt"], FS, 12., 36.)
    assert rel_err(ker, g["ker"])[0] <= 1e-14
    assert rel_err(D.xcorr2d(g["S"], g["ker"]), g["xc2d"])[0] <= 1e-12


def test_stft_restatement_against_scipy():
    """librosa is not installed anywhere here; pin the restated STFT (SURVEY App. A.6) against
    SciPy's independent implementation with the same framing."""
    import scipy.signal as sps
    rng = np.random.default_rng(0)
    y = rng.standard_normal(3000)
    for n_fft, hop in ((128, 25), (256, 12), (160, 8)):
        s = O.stft_librosa(y, n_fft, hop)
        _, _, z = sps.stft(y, nperseg=n_fft, noverlap=n_fft - hop, window=sps.get_window("hann", n_fft, fftbins=True),
                           boundary="zeros", padded=False, return_onesided=True, scaling="spectrum")
        z = z * sps.get_window("hann", n_fft, fftbins=True).sum()     # undo scipy's 1/sum(w) scaling
        n = min(s.shape[1], z.shape[1])
        assert n >= 1 + (len(y) - n_fft) // hop
        assert rel_err(np.abs(s[:, :n]), np.abs(z[:, :n]))[0] <= 1e-10


@pytest.mark.parametrize("n_fft,hop,b0,b1", [(160, 8, 12, 24), (160, 8, 0, 30), (160, 8, 50, 80), (128, 8, 3, 18)])
def test_sliding_dft_recursion_numerics(n_fft, hop, b0, b1):
    """The recursion behind d4w_stft_slide, restated in fp32 NumPy, against the fp64 STFT restatement: re-anchoring every
    160 frames keeps it at ~1e-6 of the spectrum's maximum, also when the band only sees the leakage of a strong
    out-of-band tone or of a DC offset (the rectangular-window values are large there, the Hann combination cancels them)."""
    rng = np.random.default_rng(n_fft + b0)
    ns = 20000
    t = np.arange(ns) / 200.0
    for y in (rng.standard_normal(ns), rng.standard_normal(ns) + 100 * np.sin(2 * np.pi * 0.7 * t), rng.standard_normal(ns) + 1e3):
        full = np.abs(O.stft_librosa(y, n_fft, hop))
        got = O.stft_sliding_band(y, n_fft, hop, b0, b1)
        assert got.shape == (b1 - b0 + 1, 1 + ns // hop)
        assert np.abs(got - full[b0:b1 + 1]).max() / full.max() <= 5e-6
    y = rng.standard_normal(3000)                                                                     # the identity itself, in fp64
    ref = np.abs(O.stft_librosa(y, n_fft, hop))
    assert np.abs(O.stft_sliding_band(y, n_fft, hop, b0, b1, dtype=np.float64) - ref[b0:b1 + 1]).max() / ref.max() <= 1e-12


def test_oracle_against_live_reference(golden):
    """Spot check on seeded white noise against the reference's outputs for the same input (tests/golden/spot.npz;
    every third row of the 2-D outputs is stored)."""
    g = golden("spot")
    rng = np.random.default_rng(5)
    nx, ns = 36, 200
    x = rng.standard_normal((nx, ns))
    assert abs(float(np.sum(x)) - float(g["a_x_checksum"])) <= 1e-9
    sel = [0, nx, 1]
    m = g["a_mask"]
    assert np.array_equal(m, O.fk_filter_design((nx, ns), sel, DX, FS))
    assert rel_err(O.fk_filter_filt(x.copy(), m, True)[::3], g["a_fk_rows"])[0] <= 1e-13
    assert np.max(np.abs(g["a_ninf"] - O.hybrid_ninf_filter_design((nx, ns), sel, DX, FS))) <= 1e-13
    assert rel_err(O.bp_filt(x, FS, 14, 30)[::3], g["a_bp_rows"])[0] <= 1e-13
    tpl = g["a_tpl"]
    assert np.array_equal(tpl, D.gen_template_fincall(np.arange(ns) / FS, FS, 17.8, 28.8, 0.68))
    assert rel_err(D.compute_cross_correlogram(x, tpl)[::3], g["a_xc_rows"])[0] <= 1e-13


def test_picks_and_raw2strain_match_golden(golden):
    """find_peaks(prominence) picks on rows full of ties / flat tops, and the loader's raw2strain."""
    from oracle import data_oracle as DH
    g = golden("picks")
    for thr in (0.0, 0.4, 2.0):
        got = D.convert_pick_times(D.pick_times(g["x"], thr))
        assert np.array_equal(got, g[f"picks_thr{thr}"])
    r = golden("raw2strain")
    out = DH.raw2strain(r["raw"], {"scale_factor": float(r["scale_factor"])})
    assert rel_err(out, r["strain"])[0] <= 1e-15


def test_round2_views_match_golden(golden):
    """dsp.get_fx / instant_freq, detect.xcorr / nxcorr2d / process_corr, unequal-length shift_xcorr (tests/golden/views.npz)."""
    g = golden("views")
    for nfft in (512, 600, 1000):
        assert rel_err(O.get_fx(g["fx_x"], nfft), g[f"fx_{nfft}"])[0] <= 1e-14
    assert rel_err(O.instant_freq(g["if_x"], FS), g["if_y"])[0] <= 1e-12
    assert rel_err(D.shift_xcorr(g["sx_a"], g["sx_b"]), g["sx_ab"])[0] <= 1e-13
    assert rel_err(D.shift_xcorr(g["sx_a"], g["sx_c"]), g["sx_ac"])[0] <= 1e-13
    assert rel_err(D.shift_nxcorr(g["sx_a"], g["sx_c"]), g["snx_ac"])[0] <= 1e-13
    ts, cv = D.xcorr(g["xc_t"], g["xc_f"], g["xc_S"], g["xc_tvec"], g["xc_fvec"], g["xc_ker"])
    assert np.array_equal(ts, g["xc_tscale"]) and rel_err(cv, g["xc_val"])[0] <= 1e-13
    nf = len(g["xc_f"])
    assert rel_err(D.nxcorr2d(g["xc_S"][:nf], g["xc_ker"]), g["nxc2d"])[0] <= 1e-12
    assert np.array_equal(D.process_corr(g["pc_x"], 0.05), g["pc_idx"])


def test_round2_gabor_oracle_matches_golden(golden):
    """The image-domain detector restated on OpenCV / torchvision (oracle/improcess_oracle.py) against the outputs of the
    unmodified reference functions (tests/golden/gabor.npz)."""
    cv2 = pytest.importorskip("cv2")
    pytest.importorskip("torchvision")
    from oracle import improcess_oracle as IO
    from oracle.make_golden import synth
    g = golden("gabor")
    trf = synth(int(g["nx"]), int(g["ns"]), seed=int(g["seed"]), ncalls=int(g["ncalls"]))
    assert abs(float(np.sum(trf)) - float(g["x_checksum"])) <= 1e-6 * abs(float(g["x_checksum"]))
    masked, parts = IO.gabor_detect(trf, FS, DX, [0, int(g["nx"]), 1], 1500., 10, float(g["thr"]), float(g["thr2"]))
    assert rel_err(parts["imagebin"], g["imagebin"])[0] <= 1e-12
    assert rel_err(parts["fimage"], g["fimage"])[0] <= 1e-12
    assert np.array_equal(parts["mask"], g["mask"])
    ms = np.unpackbits(g["mask_sparse_bits"])[: trf.size].reshape(trf.shape).astype(bool)
    assert np.array_equal(parts["mask_sparse"], ms)
    assert rel_err(masked[g["rows"]], g["masked_rows"])[0] <= 1e-13
    assert np.max(np.abs(IO.gabor_filt_design(float(g["theta"]))[0] - g["up"])) <= 1e-15


def test_torch_second_oracle_pinned_to_numpy_oracle():
    """oracle/torch_oracle.py (the float64 whole-matrix oracle of tests/test_fullsize_gpu.py) == oracle/dsp_oracle.py on the CPU."""
    import torch
    from oracle import torch_oracle as TO
    rng = np.random.default_rng(3)
    for nx, ns in ((64, 400), (100, 1200), (63, 406)):
        sel = [0, nx, 1]
        assert np.array_equal(TO.fk_filter_design((nx, ns), sel, DX, FS).numpy(), np.asarray(O.fk_filter_design((nx, ns), sel, DX, FS)))
        args = (1350., 1450., 3300, 3450, 14., 30.)
        mo = O.hybrid_ninf_filter_design((nx, ns), sel, DX, FS, *args)
        assert np.max(np.abs(TO.hybrid_ninf_filter_design((nx, ns), sel, DX, FS, *args).numpy() - mo)) <= 1e-15
        x = rng.standard_normal((nx, ns))
        y = TO.fk_filter_filt(torch.from_numpy(x), torch.from_numpy(mo)).numpy()
        assert rel_err(y, O.fk_filter_filt(x, mo))[0] <= 1e-13
        assert rel_err(O.fk_filter_filt(x, mo, workers=2), O.fk_filter_filt(x, mo))[0] <= 1e-13     # bench's threaded CPU arm


def test_round2_oracle_against_live_reference(golden):
    """Spot check of the spectral view and the image-detector helpers against the reference's outputs for the same
    seeded input (tests/golden/spot.npz; the reference's Gabor `down` kernel is flipud(up))."""
    from oracle import improcess_oracle as IO
    g = golden("spot")
    rng = np.random.default_rng(8)
    x = rng.standard_normal((30, 500))
    assert abs(float(np.sum(x)) - float(g["b_x_checksum"])) <= 1e-9
    assert rel_err(O.get_fx(x, 256)[::3], g["b_fx_rows"])[0] <= 1e-14
    image = IO.trace2image(x)
    assert rel_err(image[::3], g["b_img_rows"])[0] <= 1e-13
    assert rel_err(IO.binning(image, 0.1, 0.1), g["b_bin"])[0] <= 1e-13
    up, down = IO.gabor_filt_design(40.0)
    assert np.array_equal(up, g["b_up"]) and np.array_equal(down, np.flipud(g["b_up"]))
