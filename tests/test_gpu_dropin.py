"""Drop-in proof: the reference's own encoder and decoder (unmodified sources, real API loop)
with lib/mapping0.c's hot callees AND lib/block.c's envelope search (the block-size decisions of
vorbis_analysis_blockout) bound to the CUDA library through the reference-signature shims
(vorbis_b200/host/vb200_ref_shim.c) must produce byte-identical packets and bit-identical decoded PCM.  Needs oracle/_ref/*.so (built in the container where /root/reference exists;
the .so files travel to the GPU box)."""
import numpy as np
import pytest

from conftest import probe_signal
from oracle import pyref

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("ch,rate,q", [(2, 44100, 0.5), (1, 44100, 0.4), (2, 44100, 0.1), (6, 48000, 0.2),
                                      (2, 44100, -0.1), (2, 96000, 0.7)])
def test_encoder_packets_identical(cuda_ok, ch, rate, q):
    if not (pyref.available() and pyref.dropin_available()):
        pytest.skip("oracle/_ref not built (needs /root/reference at build time)")
    pcm = probe_signal(ch, rate, 0.6, seed=5)
    ref = pyref.Ref(ch, rate, q)
    ref.encode_capture(pcm, fields=())
    want = ref.packets()
    got_enc = pyref.Ref(ch, rate, q, dropin=True)
    l0 = got_enc.L.vb200shim_launches()
    got_enc.encode_capture(pcm, fields=())
    got = got_enc.packets()
    assert got_enc.L.vb200shim_launches() - l0 > 100, "the CUDA path did not run"
    assert len(got) == len(want) and len(want) > 10
    for i, (a, b) in enumerate(zip(got, want)):
        assert a == b, "packet %d differs" % i
    # decode the same packets through the shimmed mdct_backward
    d_ref = ref.decode_capture(len(want) + 4, pcm.shape[1] + 8192, fields=())
    d_got = got_enc.decode_capture(len(want) + 4, pcm.shape[1] + 8192, fields=())
    assert d_ref["pcm"].shape == d_got["pcm"].shape
    assert np.array_equal(d_ref["pcm"].view(np.uint32), d_got["pcm"].view(np.uint32))
    got_enc.close()
    ref.close()


def _stock_summary(ch, rate, q, pcm):
    import ctypes as C
    L = pyref.lib()
    L.ref_stock_encode_summary.restype = C.c_long
    h, b, c = C.c_uint64(0), C.c_long(0), C.c_long(0)
    p = np.ascontiguousarray(pcm, np.float32)
    nb = L.ref_stock_encode_summary(ch, C.c_long(rate), C.c_float(q), p.ctypes.data_as(C.c_void_p), C.c_long(p.shape[1]),
                                    C.byref(h), C.byref(b), C.byref(c))
    return nb, h.value, b.value, c.value


@pytest.mark.parametrize("ch,rate,q", [(2, 44100, 0.5), (1, 44100, 0.4), (2, 44100, 0.1), (6, 48000, 0.2),
                                      (2, 44100, -0.1), (2, 96000, 0.7)])
def test_block_seam_packets_identical(cuda_ok, ch, rate, q):
    """SURVEY §8b seam 1: vorbis_analysis through vb200_mapping0_exportbundle.forward - ONE vb200_encode_dsp call per
    block (one H2D, the chain kernels, one D2H), then the reference's own floor1_encode / residue forward for the
    bits - must give byte-identical packets, with an order of magnitude fewer device round trips than the
    per-function shims."""
    if not (pyref.available() and pyref.dropin_available()):
        pytest.skip("oracle/_ref not built (needs /root/reference at build time)")
    pcm = probe_signal(ch, rate, 0.6, seed=5)
    ref = pyref.Ref(ch, rate, q)
    ref.encode_capture(pcm, fields=())
    want = ref.packets()
    enc = pyref.Ref(ch, rate, q, dropin=True)
    enc.L.ref_use_block_seam(1)
    try:
        l0 = enc.L.vb200shim_launches()
        nb = enc.L.ref_encode_capture(enc.h, np.ascontiguousarray(pcm, np.float32), pcm.shape[1], None, None)
        launches = enc.L.vb200shim_launches() - l0
    finally:
        enc.L.ref_use_block_seam(0)
    got = enc.packets()
    assert nb == len(want) and len(got) == len(want) and len(want) > 10
    for i, (a, b) in enumerate(zip(got, want)):
        assert a == b, "packet %d differs" % i
    # envelope search (2 kernels per analysed chunk) + 6 chain kernels per block; the per-function shims need > 20 per block
    assert launches <= 10 * nb, "%d launches for %d blocks" % (launches, nb)
    enc.close()
    ref.close()


@pytest.mark.parametrize("ch,rate,nominal", [(2, 44100, 128000), (1, 44100, 64000)])
def test_block_seam_managed_packets_identical(cuda_ok, ch, rate, nominal):
    """bitrate-managed encoders (vorbis_encode_init with a nominal bitrate) through the same seam: ONE
    vb200_encode_dsp_managed call per block returns all 15 curves (three masks and fits, twelve interpolated
    curves, render + couple/quantise per curve), the host writes all 15 packet blobs with the reference's own
    floor1_encode / residue forward, and lib/bitrate.c picks among them - the packets that come out must be
    byte-identical to the stock encoder's."""
    if not (pyref.available() and pyref.dropin_available()):
        pytest.skip("oracle/_ref not built (needs /root/reference at build time)")
    pcm = probe_signal(ch, rate, 0.5, seed=6)
    pcm[:, 6000:9000] = 0
    ref = pyref.Ref(ch, rate, nominal_bitrate=nominal)
    ref.encode_capture(pcm, fields=())
    want = ref.packets()
    enc = pyref.Ref(ch, rate, nominal_bitrate=nominal, dropin=True)
    enc.L.ref_use_block_seam(1)
    try:
        nb = enc.L.ref_encode_capture(enc.h, np.ascontiguousarray(pcm, np.float32), pcm.shape[1], None, None)
    finally:
        enc.L.ref_use_block_seam(0)
    got = enc.packets()
    assert nb > 0 and len(got) == len(want) and len(want) > 10
    for i, (a, b) in enumerate(zip(got, want)):
        assert a == b, "packet %d differs" % i
    assert len(set(len(p) for p in want)) > 3
    enc.close()
    ref.close()


@pytest.mark.parametrize("ch,rate,q", [(2, 44100, 0.5), (1, 22050, 0.3)])
def test_multistream_driver_packets_identical(cuda_ok, ch, rate, q):
    """vb200ms_*: 7 concurrent encoders whose ready blocks go to the device together (one vb200_encode_dsp call per
    block size and round); every stream's packets (count, bytes, hash of all bytes in order) must equal what the
    stock reference encoder produces for that stream alone."""
    import ctypes as C
    from test_plan_vs_ref import burst_signal
    if not (pyref.available() and pyref.dropin_available()):
        pytest.skip("oracle/_ref not built (needs /root/reference at build time)")
    ns, secs = 7, 0.8
    n = int(rate * secs)
    sig = [probe_signal(ch, rate, secs, seed=20 + i)[:, :n] if i % 2 == 0 else burst_signal(ch, rate, secs, 30 + i)[:, :n] for i in range(ns)]
    pcm = np.ascontiguousarray(np.stack(sig), np.float32)
    L = pyref.dropin_lib()
    L.ref_ms_encode.restype = C.c_long
    hashes = (C.c_uint64 * ns)()
    nbytes = (C.c_long * ns)()
    counts = (C.c_long * ns)()
    blocks = L.ref_ms_encode(ns, ch, C.c_long(rate), C.c_float(q), 0, pcm.ctypes.data_as(C.c_void_p), C.c_long(n), hashes, nbytes, counts)
    assert blocks > 0
    total = 0
    for i in range(ns):
        nb, h, b, c = _stock_summary(ch, rate, q, pcm[i])
        assert (counts[i], nbytes[i]) == (c, b), "stream %d: %d packets / %d bytes, stock %d / %d" % (i, counts[i], nbytes[i], c, b)
        assert hashes[i] == h, "stream %d packet bytes differ" % i
        total += nb
    assert blocks == total
