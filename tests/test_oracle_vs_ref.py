"""CPU oracle (our restatement) against the compiled reference on fresh signals, for a grid of
(channels, rate, quality): every stage, the fused Phase-A chain recorded from the real mapping0_forward,
Phase B, the ampmax chain and the decoded PCM.  Bit-exact.
What the reference computed is recorded in tests/golden/ref_records.xz by tests/golden/make_golden_ref.py
(large arrays as digests, see tests/refrec.py); the signals and random vectors are built here, from the
same seeds, for both."""
import numpy as np
import pytest

import refrec
from conftest import probe_signal
from vorbis_b200 import abi, lib as vlib

GRID = [(2, 44100, 0.5), (1, 44100, 0.4), (2, 44100, 0.1), (2, 44100, 0.3), (1, 44100, 0.2),
        (2, 48000, 0.9), (2, 32000, 0.0), (1, 22050, 0.3), (2, 44100, -0.1), (1, 44100, -0.1), (4, 44100, 0.5)]
FLOOR1_ARGS = [(2, 44100, 0.5), (6, 48000, 0.2), (2, 32000, -0.1), (1, 16000, 0.5), (2, 96000, 0.7)]
ENCODE_ARGS = [(2, 44100, 0.5), (2, 44100, 0.1), (1, 44100, 0.4), (6, 48000, 0.2), (2, 44100, -0.1), (6, 48000, -0.1),
               (8, 48000, 0.3)]
MANAGED_ARGS = [(2, 44100, 0.5), (1, 44100, 0.4), (6, 48000, 0.2), (2, 44100, -0.1)]
ENVELOPE_ARGS = [(2, 44100, 0.5), (1, 44100, 0.4), (6, 48000, 0.2), (1, 22050, 0.3), (2, 32000, 0.0), (2, 96000, 0.7),
                 (2, 44100, -0.1)]
INVERSE2_ARGS = [(2, 44100, 0.5), (6, 48000, 0.2), (1, 22050, 0.3), (2, 44100, -0.1)]
RESIDUE_ARGS = [(2, 44100, 0.5), (1, 44100, 0.4), (6, 48000, 0.2), (1, 22050, 0.3), (2, 44100, 0.1), (2, 44100, -0.1),
                (4, 44100, 0.5)]
ids = lambda g: "ch%d_%d_q%g" % g  # noqa: E731


def pair_signal(ch, rate):
    pcm = probe_signal(ch, rate, 1.2, seed=11)
    if ch == 2:
        pcm[1] = (0.7 * pcm[0] + 0.3 * pcm[1]).astype(np.float32)
    return pcm


def floor1_signal(ch, rate):
    pcm = probe_signal(ch, rate, 1.0, seed=5)
    pcm[:, :3000] = 0
    return pcm


def encode_signal(ch, rate):
    pcm = probe_signal(ch, rate, 1.0, seed=9)
    pcm[:, 5000:9000] = 0
    return pcm


def managed_signal(ch, rate):
    pcm = probe_signal(ch, rate, 0.6, seed=21)
    pcm[:, 5000:9000] = 0
    return pcm


def envelope_signal(ch, rate):
    rng = np.random.default_rng(3)
    pcm = probe_signal(ch, rate, 44100 / rate, seed=5)[:, :44100].copy()
    pcm[:, 8000:12000] *= 0.001
    pcm[:, 20000:20300] = rng.uniform(-.9, .9, (ch, 300))
    pcm[:, 30000:33000] = 0
    return pcm


def transform_inputs(bs):
    rng = np.random.default_rng(7)
    for W in (0, 1):
        N = bs[W]
        x = rng.uniform(-1, 1, (16, N)).astype(np.float32)
        y = rng.uniform(-1, 1, (16, N // 2)).astype(np.float32)
        lW = rng.integers(0, 2, 16).astype(np.int32)
        nW = rng.integers(0, 2, 16).astype(np.int32)
        yield W, x, y, lW, nW


def inverse2_inputs(ch, bs):
    rng = np.random.default_rng(4)
    for W in (0, 1):
        n, rows = bs[W] // 2, ch * 7
        posts = rng.integers(0, 140, (rows, abi.FLOOR1_STRIDE)).astype(np.int32)
        flag = rng.random(posts.shape) < 0.4
        flag[:, :2] = False
        posts[flag] |= 0x8000
        posts[3, 5] = 400
        posts[4, 0] = 999
        present = (rng.random(rows) < 0.85).astype(np.int32)
        data = (rng.standard_normal((rows, n)) * 5).astype(np.float32)
        yield W, posts, present, data


def residue_inputs(ch, bs):
    rng = np.random.default_rng(13)
    for W in (0, 1):
        n, nb = bs[W] // 2, 6
        mag = np.exp(rng.uniform(-2, 3, (nb, ch, 1))) * np.exp(-np.arange(n) / (n / 4.0))[None, None, :]
        iwork = np.rint(rng.standard_normal((nb, ch, n)) * mag).astype(np.int32)
        nonzero = (rng.random((nb, ch)) < 0.8).astype(np.int32)
        nonzero[1] = 0
        yield W, iwork, nonzero


def encoder_outputs(o, enc, W, idx):
    """Phase A, floor1 fit + render and couple/quantise of the oracle on the reference's blocks `idx` of size W
    (what mapping0_forward computes per block): the inputs each later stage of the reference was handed."""
    n = enc.bs[W] // 2
    out = o.phaseA(W, enc.blocks(W, idx), enc.desc(idx), taps=True)
    k, ch = out["mdct"].shape[:2]
    posts, nz = o.floor1_fit(W, out["logmdct"], out["logmask"])
    out["enc_posts"], ilog, nz2 = o.floor1_render(W, posts, nz)
    out["ilogmask"], out["nonzero_in"] = ilog.reshape(k, ch, n), nz2.reshape(k, ch)
    out["iwork_out"] = np.zeros((k, ch, n), np.int32)
    for bt in (0, 1):
        s = np.where(enc.case["blocktype"][idx] == bt)[0]
        if len(s):
            out["iwork_out"][s] = o.couple_quantize_normalize(W, bt, 7, out["mdct"][s], out["ilogmask"][s],
                                                              out["nonzero_in"][s])[0]
    return out


def decoded_residue(setup, W, iwork):
    """The residue the decoder reads back from the packet: the quantised residue [ch][n] with the bins outside
    the residue's coded range [begin, end) zeroed; for residue type 2 the range counts interleaved samples of
    the channels of the submap."""
    a = setup.arrays
    res = iwork.astype(np.float32)
    mux = a["chmux"][W][:len(res)]
    for c in range(len(res)):
        pre = "residue_%d_%d_" % (W, mux[c])
        pos = np.arange(res.shape[1])
        if a[pre + "type"].item() == 2:
            pos = pos * int((mux == mux[c]).sum()) + int((mux[:c] == mux[c]).sum())
        res[c, (pos < a[pre + "begin"].item()) | (pos >= a[pre + "end"].item())] = 0
    return res


@pytest.fixture(scope="module", params=GRID, ids=ids)
def pair(request, oracle_lib):
    ch, rate, q = request.param
    rec = refrec.Case("pair", ch, rate, q)
    setup = refrec.setup(ch, rate, q)
    o = oracle_lib.Oracle(setup)
    pcm = pair_signal(ch, rate)
    enc = refrec.Encoding(rec, setup, pcm)
    return rec, setup, o, enc, pcm


def test_tables(pair):
    rec, setup, o, enc, _ = pair
    for W in (0, 1):
        for which in (0, 1, 2, 3):
            rec.check(o.table(W, which), "table_%d_%d" % (W, which), "table W%d #%d" % (W, which))


def test_transforms_random(pair):
    rec, setup, o, enc, _ = pair
    for W, x, y, lW, nW in transform_inputs(enc.bs):
        rec.check(o.mdct_forward(W, x), "mdct_forward_%d" % W, "mdct_forward")
        rec.check(o.mdct_backward(W, y), "mdct_backward_%d" % W, "mdct_backward")
        rec.check(o.drft_forward(W, x), "drft_forward_%d" % W, "drft_forward")
        rec.check(o.apply_window(W, x, lW, nW), "window_%d" % W, "window")


def test_phaseA_chain_of_the_real_encoder(pair):
    rec, setup, o, enc, _ = pair
    for W in (0, 1):
        idx = enc.idx(W)
        if not len(idx):
            continue
        blocks = enc.blocks(W, idx)
        rec.check(blocks, "pcm_%d" % W, "W%d blocks" % W)
        out = o.phaseA(W, blocks, enc.desc(idx), taps=True)
        for k, g in (("mdct_raw", "mdct_raw"), ("logfft", "logfft"), ("noise", "noise"), ("tone", "tone"),
                     ("logmdct", "logmdct"), ("logmask", "logmask"), ("mdct", "mdct_m1")):
            rec.check(out[k], "%s_%d" % (g, W), "W%d %s" % (W, k))
        rec.check(out["ampmax_out"], "ampmax_out_%d" % W, "ampmax_out")
        # the driver's batched reference helper (used by bench.py's CPU legs) agrees too
        rec.check(out["logmask"], "batch_logmask_%d" % W, "ref_phaseA_batch logmask")
        rec.check(out["mdct"], "batch_mdct_%d" % W, "ref_phaseA_batch mdct")


def test_phaseB_of_the_real_encoder(pair):
    rec, setup, o, enc, _ = pair
    for W in (0, 1):
        for bt in (0, 1):
            sel = np.where((enc.W == W) & (enc.case["blocktype"] == bt))[0]
            if not len(sel):
                continue
            inp = encoder_outputs(o, enc, W, sel)
            for k, g in (("mdct", "mdct_m1"), ("ilogmask", "ilogmask"), ("nonzero_in", "nonzero_in")):
                rec.check(inp[k], "%s_%d_%d" % (g, W, bt), "Phase B input %s" % g)
            iw, nz = o.couple_quantize_normalize(W, bt, 7, inp["mdct"], inp["ilogmask"], inp["nonzero_in"])
            rec.check(iw, "iwork_out_%d_%d" % (W, bt), "iwork")
            rec.check(nz, "nonzero_out_%d_%d" % (W, bt), "nonzero")


def test_decode_of_the_real_stream(pair):
    rec, setup, o, enc, pcm = pair
    Wseq = rec["dec_W"][None, :]
    bs = enc.bs
    coef_off, pcm_off, coef_len, pcm_len = vlib.synthesis_layout(Wseq, bs, setup.channels)
    blocks = [None] * len(enc.W)
    for W in (0, 1):
        idx = enc.idx(W)
        if not len(idx):
            continue
        e = encoder_outputs(o, enc, W, idx)
        ch = setup.channels
        for j, b in enumerate(idx):
            res = o.decouple(W, decoded_residue(setup, W, e["iwork_out"][j])[None])[0]
            blocks[b] = o.floor1_inverse2(W, e["enc_posts"][j * ch:(j + 1) * ch], e["nonzero_in"][j], res)
    coef = np.concatenate([blocks[k].reshape(-1) for k in range(Wseq.shape[1])])
    rec.check(coef, "dec_coef", "the decoder's spectra")        # the input: what the reference decoder read back
    out = o.synthesis(Wseq, coef_off, coef, pcm_off, pcm_len)
    m = min(int(rec["dec_len"]), pcm_len)
    assert m > 0 and m == int(rec["dec_len"])
    rec.check(out[0][:, :m], "dec_pcm", "decoded pcm")


@pytest.mark.parametrize("args", FLOOR1_ARGS, ids=ids)
def test_floor1_vs_reference(args, oracle_lib):
    """floor1_fit / floor1_encode recorded inside the reference's own mapping0_forward, incl. silent
    blocks (NULL fit) and the 5.1 LFE submap with its own 2-post floor."""
    ch, rate, q = args
    rec = refrec.Case("floor1", ch, rate, q)
    setup = refrec.setup(ch, rate, q)
    o = oracle_lib.Oracle(setup)
    enc = refrec.Encoding(rec, setup, floor1_signal(ch, rate))
    nulls = 0
    for W in (0, 1):
        idx = enc.idx(W)
        if not len(idx):
            continue
        n = enc.bs[W] // 2
        a = o.phaseA(W, enc.blocks(W, idx), enc.desc(idx))
        rec.check(a["logmdct"], "logmdct_%d" % W, "floor1_fit input logmdct")
        rec.check(a["logmask"], "logmask_%d" % W, "floor1_fit input logmask")
        posts, nz = o.floor1_fit(W, a["logmdct"], a["logmask"])
        nulls += int((nz == 0).sum())
        rec.check(nz, "fit_nonzero_%d" % W, "fit nonzero")
        rec.check(posts, "fit_posts_%d" % W, "fit posts")
        p2, ilog, nz2 = o.floor1_render(W, posts, nz)
        rec.check(p2[nz == 1], "enc_posts_%d" % W, "floor1_encode posts")
        rec.check(ilog, "ilogmask_%d" % W, "ilogmask")
        rec.check(nz2, "nonzero_in_%d" % W, "nonzero")
    assert nulls > 0


@pytest.mark.parametrize("args", ENCODE_ARGS, ids=ids)
def test_encode_chain_vs_reference(args, oracle_lib):
    """the composed oracle chain (what vb200_encode_dsp is checked against) equals the reference's own
    functions called in mapping0_forward's order (ref_encode_dsp_batch, also bench.py's CPU arm), on the
    PCM blocks, block flags and ampmax the reference's own API loop handed to mapping0_forward"""
    ch, rate, q = args
    rec = refrec.Case("encode", ch, rate, q)
    setup = refrec.setup(ch, rate, q)
    o = oracle_lib.Oracle(setup)
    enc = refrec.Encoding(rec, setup, encode_signal(ch, rate))
    for W in (0, 1):
        idx = enc.idx(W)
        if not len(idx):
            continue
        blocks = enc.blocks(W, idx)
        rec.check(blocks, "pcm_%d" % W, "W%d blocks" % W)
        a = o.encode_dsp(W, blocks, enc.desc(idx))
        for k in ("posts", "nonzero", "iwork", "ampmax_out"):
            rec.check(a[k], "batch_%s_%d" % (k, W), k)
        rec.check(a["iwork"], "iwork_out_%d" % W, "iwork vs the API loop's capture")


@pytest.mark.parametrize("args", MANAGED_ARGS, ids=ids)
def test_managed_chain_vs_reference(args, oracle_lib):
    """bitrate-managed mode: the composed oracle (three masks, three fits, twelve interpolated curves, render +
    couple/quantise per curve; what vb200_encode_dsp_managed is checked against) equals the reference's own
    functions called in mapping0_forward's managed order (lib/mapping0.c:500-573, 596-646), incl. silent blocks
    (NULL curves) and both block sizes"""
    ch, rate, q = args
    rec = refrec.Case("managed", ch, rate, q)
    setup = refrec.setup(ch, rate, q)
    o = oracle_lib.Oracle(setup)
    enc = refrec.Encoding(rec, setup, managed_signal(ch, rate))
    nulls = 0
    for W in (0, 1):
        idx = enc.idx(W)[:10]
        if not len(idx):
            continue
        blocks = enc.blocks(W, idx)
        desc = enc.desc(idx)
        a = o.encode_dsp_managed(W, blocks, desc)
        for k in ("posts", "nonzero", "iwork", "ampmax_out"):
            rec.check(a[k], "managed_%s_%d" % (k, W), "%s W%d" % (k, W))
        mid = abi.PACKETBLOBS // 2
        assert np.array_equal(a["iwork"][mid], o.encode_dsp(W, blocks, desc)["iwork"]), "curve 7 is the un-managed chain"
        assert not np.array_equal(a["iwork"][0], a["iwork"][abi.PACKETBLOBS - 1]), "low and high rate curves differ"
        nulls += int((a["posts"].reshape(abi.PACKETBLOBS, -1, abi.FLOOR1_STRIDE)[:, :, :2] == 0).all(axis=2).sum())
    assert nulls > 0, "the probe holds silent blocks"


@pytest.mark.parametrize("args", ENVELOPE_ARGS, ids=ids)
def test_envelope_vs_reference(args, oracle_lib):
    """the reference's own _ve_envelope_search on a fresh dsp state vs the restatement: marks, filter
    states and stretch bit-identical (the stream buffer, incl. the pre-extrapolated preamble, is the
    reference's)"""
    ch, rate, q = args
    rec = refrec.Case("envelope", ch, rate, q)
    setup = refrec.setup(ch, rate, q)
    o = oracle_lib.Oracle(setup)
    stream = refrec.timeline(rec, envelope_signal(ch, rate), setup.blocksize(1) // 2)
    steps, marks = int(rec["steps"]), rec["marks"]
    ret, state = o.envelope_search(stream[None], 0, steps)
    assert np.array_equal(o.envelope_marks(ret[0])[:steps + 2], marks)
    assert np.array_equal(state[0], rec["state"])
    assert marks.sum() > 0


@pytest.mark.parametrize("args", INVERSE2_ARGS, ids=ids)
def test_floor1_inverse2_vs_reference(args, oracle_lib):
    """decode-side floor: the reference's own floor1_inverse2 (through floor1_exportbundle) vs the
    restatement, on random fit_value[] incl. unused posts (bit 15), out-of-range values (clamped,
    lib/floor1.c:1056-1064) and absent floors (row zeroed)"""
    ch, rate, q = args
    rec = refrec.Case("inverse2", ch, rate, q)
    setup = refrec.setup(ch, rate, q)
    o = oracle_lib.Oracle(setup)
    for W, posts, present, data in inverse2_inputs(ch, [setup.blocksize(0), setup.blocksize(1)]):
        rec.check(o.floor1_inverse2(W, posts, present, data), "inverse2_%d" % W, "floor1_inverse2 W=%d" % W)


@pytest.mark.parametrize("args", RESIDUE_ARGS, ids=ids)
def test_residue_classify_vs_reference(args, oracle_lib):
    """res1_class / res2_class through the reference's own _residue_P[] (per submap, as mapping0_forward
    calls them) vs the restatement; residue types 1 and 2, the 5.1 setup's two submaps and 30-sample
    partitions, silent channels and silent bundles"""
    ch, rate, q = args
    rec = refrec.Case("residue", ch, rate, q)
    setup = refrec.setup(ch, rate, q)
    o = oracle_lib.Oracle(setup)
    for W, iwork, nonzero in residue_inputs(ch, [setup.blocksize(0), setup.blocksize(1)]):
        assert o.residue_partvals(W) > 0
        a = o.residue_classify(W, iwork, nonzero)
        rec.check(a, "classes_%d" % W, "residue classes W=%d" % W)
        assert a.max() > 0 and not a[1].any()
