"""The transforms and the window table against their mathematical definitions, evaluated in float64, at every
block size the tested setups use (256 ... 4096).  The bit-exact tests compare the kernels with an fp32
restatement of the reference's arithmetic (the oracle) that reads the same setup; a wrong trig, bit-reverse
or window table would be shared by both and pass there.  Checked on the oracle everywhere and on the CUDA
entry points on the GPU.

  mdct_forward   X[k] = 4/N * sum_n x[n] cos(2 pi/N (n + 1/2 + N/4)(k + 1/2)),   k < N/2
  mdct_backward  y[n] =       sum_k X[k] cos(2 pi/N (n + 1/2 + N/4)(k + 1/2)),   n < N
  drft_forward   unscaled real FFT in FFTPACK order [r0, r1, i1, ..., r(N/2-1), i(N/2-1), r(N/2)]
  window (W, 2)  w[i] = sin(pi/2 sin^2((i + 1/2)/(N/2) pi/2)),  i < N/2  (the Vorbis window, lib/window.c)"""
import numpy as np
import pytest

import refrec

# one setup per block size (refrec.setup: a committed fixture or a recorded setup)
SIZES = {256: ((2, 44100, 0.5), 0), 512: ((2, 44100, -0.1), 0), 1024: ((1, 16000, 0.5), 1),
         2048: ((2, 44100, 0.5), 1), 4096: ((2, 44100, -0.1), 1)}
REL = 1e-6          # max |error| over max |exact| of each row


def _inputs(N):
    rng = np.random.default_rng(N)
    x = rng.uniform(-1, 1, (12, N))
    x[0] = 0.0                              # silence
    x[1] = 1.0                              # DC
    x[2, ::2], x[2, 1::2] = 1.0, -1.0       # alternating +-1 (Nyquist)
    x[3] *= 1e-30
    x[4] = np.sin(2 * np.pi * 37.25 * np.arange(N) / N)
    y = rng.uniform(-1, 1, (12, N // 2))
    y[0] = 0.0
    y[1] = 1.0
    y[2, ::2], y[2, 1::2] = 1.0, -1.0
    y[3] *= 1e-30
    y[4] = 0.0
    y[4, N // 8] = 1.0                      # one basis function
    return x.astype(np.float32), y.astype(np.float32)


def _mdct_basis(N):
    n = np.arange(N, dtype=np.float64)
    k = np.arange(N // 2, dtype=np.float64)
    return np.cos(2 * np.pi / N * np.outer(k + 0.5, n + 0.5 + N / 4))       # [N/2][N]


def _fftpack(x):
    f = np.fft.rfft(x.astype(np.float64), axis=1)
    N = x.shape[1]
    out = np.empty((x.shape[0], N))
    out[:, 0] = f[:, 0].real
    out[:, 1:N - 1:2] = f[:, 1:N // 2].real
    out[:, 2:N - 1:2] = f[:, 1:N // 2].imag
    out[:, N - 1] = f[:, N // 2].real
    return out


def _close(got, exact, what):
    got = np.asarray(got, np.float64)
    assert got.shape == exact.shape, "%s: shape %s vs %s" % (what, got.shape, exact.shape)
    err = np.abs(got - exact).max(axis=1)
    scale = np.abs(exact).max(axis=1)
    bad = np.where(err > REL * scale)[0]
    assert not len(bad), "%s: row %d error %.3g of max %.3g" % (what, bad[0], err[bad[0]], scale[bad[0]])


def check_against_definitions(impl, W, N):
    """impl: an oracle.pyoracle.Oracle or a vorbis_b200.lib.Context (same method names) whose block size W is N"""
    assert impl.bs[W] == N
    x, y = _inputs(N)
    C = _mdct_basis(N)
    _close(impl.mdct_forward(W, x), (4.0 / N) * (x.astype(np.float64) @ C.T), "mdct_forward N=%d" % N)
    _close(impl.mdct_backward(W, y), y.astype(np.float64) @ C, "mdct_backward N=%d" % N)
    _close(impl.drft_forward(W, x), _fftpack(x), "drft_forward N=%d" % N)
    i = np.arange(N // 2, dtype=np.float64)
    win = np.sin(np.pi / 2 * np.sin((i + 0.5) / (N // 2) * np.pi / 2) ** 2)
    _close(impl.table(W, 2)[None], win[None], "window table N=%d" % N)


@pytest.mark.parametrize("N", sorted(SIZES))
def test_oracle_transforms_match_definitions(N, oracle_lib):
    args, W = SIZES[N]
    check_against_definitions(oracle_lib.Oracle(refrec.setup(*args)), W, N)


@pytest.mark.gpu
@pytest.mark.parametrize("N", sorted(SIZES))
def test_cuda_transforms_match_definitions(N, cuda_ok):
    from vorbis_b200 import lib as vlib
    args, W = SIZES[N]
    check_against_definitions(vlib.Context(refrec.setup(*args)), W, N)
