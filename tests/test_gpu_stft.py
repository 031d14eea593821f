"""GPU parity: framed STFT / iSTFT kernels (through the C ABI) vs the oracle and the golden
vectors produced by the reference's own functions.  fp32 kernels vs float64 reference:
tolerance 2e-6 relative L2 on spectra, 5e-6 on reconstructed audio (stated per assert)."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from dspgolden import check  # noqa: E402
from oracle import dsp  # noqa: E402


def rel(a, b):
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


@pytest.fixture(scope="module")
def ctx():
    from deepconvsep_b200.engine import Context
    return Context(0)


def _plan(ctx, N, H, w):
    from deepconvsep_b200.engine import Stft
    return Stft(ctx, N, H, w)


def test_golden_stft_istft(ctx, golden):
    g = golden
    for ci in range(int(g["n_stft"])):
        N, H = (int(v) for v in g["stft%d_NH" % ci])
        x, w = g["stft%d_x" % ci], g["stft%d_w" % ci]
        # the reference's spectrum and inverses, recomputed by the oracle and held to what the reference stored
        Xr = dsp.stft_norm(x, window=w, hopsize=float(H), nfft=float(N))
        check(g, "stft%d_X" % ci, Xr)
        st = _plan(ctx, N, H, w)
        xd = torch.tensor(x, dtype=torch.float32, device="cuda")
        X, mag = st.forward(xd, mag_scale=0.3)
        torch.cuda.synchronize()
        T, F = Xr.shape
        assert X.shape == (T, st.ldf)
        Xg = X.cpu().numpy()[:, :F].astype(np.complex128)
        assert rel(Xg, Xr) < 2e-6, (ci, rel(Xg, Xr))
        assert np.all(X.cpu().numpy()[:, F:] == 0) and np.all(mag.cpu().numpy()[:, F:] == 0)
        mref = 0.3 * (np.abs(Xr) / np.sqrt(N))
        assert rel(mag.cpu().numpy()[:, :F].astype(np.float64), mref) < 2e-6
        # inverse of the reference spectrum vs the reference's istft
        Z = g["stft%d_Z" % ci]
        for spec, key in ((Xr, "stft%d_y" % ci), (Z, "stft%d_y2" % ci)):
            want = dsp.istft_norm(spec, window=w, analysisWindow=w, hopsize=float(H), nfft=float(N))
            check(g, key, want)
            S = torch.zeros((1, T, st.ldf), dtype=torch.complex64, device="cuda")
            S[0, :, :F] = torch.tensor(spec.astype(np.complex64), device="cuda")
            y = st.inverse(S).cpu().numpy()[0].astype(np.float64)
            assert y.shape == want.shape
            # the last N/2 samples divide by sum(w^2) -> 0 (only the vanishing tail of the last
            # frame covers them): ill-conditioned in any precision and cut by data[:L] in the
            # pipeline.  Strict on the samples the pipeline keeps, loose on the full length.
            keep = x.size
            assert rel(y[:keep], want[:keep]) < 5e-6, (ci, rel(y[:keep], want[:keep]))
            assert rel(y, want) < 1e-4, (ci, rel(y, want))
        # GPU round trip reconstructs the signal
        y = st.inverse(X.unsqueeze(0), num_out=x.size).cpu().numpy()[0]
        assert rel(y.astype(np.float64), x) < 5e-6


@pytest.mark.parametrize("N,H,wname", [(1024, 512, "hanning"), (2048, 512, "hanning"), (4096, 512, "blackmanharris"),
                                       (1024, 256, "hanning"), (512, 256, "sinebell"), (256, 128, "hanning")])
def test_polar_compute_file_and_inverse(ctx, N, H, wname):
    """transformFFT.compute_file(phase=True) / compute_inverse semantics."""
    from deepconvsep_b200.engine import get_window
    rng = np.random.default_rng(N + H)
    x = rng.standard_normal(7777) * 0.1
    w = get_window(wname, N)
    st = _plan(ctx, N, H, w)
    mag_r, ph_r = dsp.compute_file(x, phase=True, frameSize=N, hopSize=H, window=w)
    xd = torch.tensor(x, dtype=torch.float32, device="cuda")
    mag, ph = st.forward_polar(xd)
    F = N // 2 + 1
    mg, pg = mag.cpu().numpy()[:, :F].astype(np.float64), ph.cpu().numpy()[:, :F].astype(np.float64)
    assert rel(mg, mag_r) < 2e-6
    # phases compare as unit phasors weighted by magnitude (angle is ill-conditioned at |X| ~ 0)
    assert rel(mg * np.exp(1j * pg), mag_r * np.exp(1j * ph_r)) < 3e-6
    y_r = dsp.compute_inverse(mag_r * 0.5, ph_r, frameSize=N, hopSize=H, window=w)
    mt = torch.zeros((mag.shape[0], st.ldf), dtype=torch.float32, device="cuda")
    pt = torch.zeros_like(mt)
    mt[:, :F] = torch.tensor(mag_r * 0.5, dtype=torch.float32, device="cuda")
    pt[:, :F] = torch.tensor(ph_r, dtype=torch.float32, device="cuda")
    y = st.inverse_polar(mt, pt).cpu().numpy().astype(np.float64)
    assert y.shape == y_r.shape
    assert rel(y[:x.size], y_r[:x.size]) < 5e-6
    assert rel(y, y_r) < 1e-4          # includes the ill-conditioned tail (sum(w^2) -> 0)


def test_large_roundtrip_property(ctx):
    """Full-size (180 s @ 44.1 kHz) size-independent property: istft(stft(x)) == x."""
    st = _plan(ctx, 2048, 512, np.hanning)
    g = torch.Generator(device="cuda").manual_seed(5)
    x = (torch.rand(7938000, generator=g, device="cuda") - 0.5) * 0.4
    X, _ = st.forward(x, want_mag=False)
    assert X.shape[0] == 15506
    y = st.inverse(X.unsqueeze(0), num_out=x.numel())[0]
    err = (torch.linalg.vector_norm(y - x) / torch.linalg.vector_norm(x)).item()
    assert err < 5e-6, err
    # linearity of the analysis: stft(a*x) == a*stft(x) bit-exactly for a power of two
    X2, _ = st.forward(x * 0.5, want_mag=False)
    assert torch.equal(torch.view_as_real(X2), torch.view_as_real(X) * 0.5)
