"""CUDA path against the CPU oracle, and against what the reference recorded, at encoder setups the five golden
configurations of tests/test_gpu_parity.py never reach:

  512/4096 blocks (every vorbisenc quality below 0 at 32-48 kHz): the generic N = 4096 transform
  instantiations, psy at n = 2048, floor 1 over 2048 bins, 64 couple/quantise chunks per row, the
  synthesis and block planner at a 4096/512 size ratio; 96 kHz and 16 kHz psy tables; the top quality;
  uncoupled 4 and 8 channel mappings (one submap, the generic couple/quantise kernel).

The setup-only tests of tests/test_gpu_parity.py run here again through this module's own `cfg` fixture
(they take the setup, the CUDA context and the oracle from it and build their own inputs); the tests below
them cover what those leave to the golden fixtures.  Bit-exact throughout."""
import numpy as np
import pytest

import refrec
from conftest import assert_bits_equal
from test_gpu_parity import (  # noqa: F401  (collected here, with this module's cfg)
    test_couple_quantize_normalize_vs_oracle_random, test_decode_dsp_one_call_vs_oracle, test_decode_int16_egress,
    test_decode_vs_oracle_random_streams, test_decouple_vs_oracle, test_encode_dsp_dev_split_half_batches,
    test_encode_dsp_int16_residue, test_encode_dsp_managed_vs_oracle, test_encode_dsp_many_chunks,
    test_encode_dsp_streams_vs_oracle, test_encode_then_decode_round_trip, test_envelope_search_streams_vs_oracle,
    test_floor1_inverse2_vs_oracle, test_floor1_vs_oracle_random, test_phaseA_adversarial_inputs,
    test_phaseA_host_path_multichunk, test_phaseA_pcm_ingest_from_stream_buffers, test_phaseA_stream_mode_device,
    test_phaseA_vs_oracle_random, test_plan_blocks_device_vs_oracle, test_psy_stages_vs_oracle_random,
    test_tables_match_oracle, test_transforms_vs_oracle_random)
from test_oracle_vs_ref import encode_signal, encoder_outputs, floor1_signal, pair_signal
from vorbis_b200 import abi, lib as vlib

pytestmark = pytest.mark.gpu

SETUPS = [(2, 44100, -0.1),     # 512/4096, coupled stereo
          (1, 44100, -0.1),     # 512/4096 mono
          (6, 48000, -0.1),     # 512/4096 5.1: two submaps, LFE floor
          (2, 32000, -0.1),     # 512/4096 at another rate
          (2, 96000, 0.7),      # 96 kHz psy tables
          (2, 48000, 0.9),      # top quality
          (1, 16000, 0.5),      # 16 kHz, 512/1024
          (4, 44100, 0.5),      # uncoupled, one submap
          (8, 48000, 0.3)]      # uncoupled, one submap
# the reference's recorded encodings of tests/test_oracle_vs_ref.py (test name -> the signal it encoded)
RECORDED = {"pair": pair_signal, "encode": encode_signal, "floor1": floor1_signal}


@pytest.fixture(scope="module", params=SETUPS, ids=lambda a: refrec.case_id(*a))
def cfg(request, oracle_lib, cuda_ok):
    """(name, setup, CUDA context, oracle, None, None): the layout of test_gpu_parity's cfg, without its golden
    encode / decode vectors (none exist for these setups)"""
    setup = refrec.setup(*request.param)
    return refrec.case_id(*request.param), setup, vlib.Context(setup), oracle_lib.Oracle(setup), None, None


def _blocks(setup, W, nb, seed):
    """nb random blocks of size W: tones over noise at random levels, silence, a quiet block, one live channel"""
    N, ch = setup.blocksize(W), setup.channels
    rng = np.random.default_rng(seed)
    t = np.arange(N)
    pcm = (rng.uniform(-1, 1, (nb, ch, N)) * 10.0 ** rng.uniform(-3, -0.5, (nb, ch, 1)) +
           0.5 * np.sin(2 * np.pi * rng.uniform(50, setup.rate / 2.5, (nb, ch, 1)) * t / setup.rate)).astype(np.float32)
    pcm[0] = 0.0
    pcm[1] *= 1e-4
    pcm[2, 1:] = 0.0
    desc = np.zeros(nb, abi.BLOCKDESC_DTYPE)
    desc["lW"] = rng.integers(0, 2, nb) if W else 0
    desc["nW"] = rng.integers(0, 2, nb) if W else 0
    desc["blocktype"] = rng.integers(0, 2, nb)
    desc["ampmax"] = rng.choice([-9999.0, -30.0, -3.0, 0.0], nb).astype(np.float32)
    return pcm, desc


@pytest.mark.parametrize("psy", ["default", "VB200_PSY_V2", "VB200_PSY_V1"])
@pytest.mark.parametrize("W", [0, 1])
def test_phaseA_psy_kernels_vs_oracle(cfg, W, psy, monkeypatch):
    """Phase A with and without taps (the taps select the psy kernel's debug instance), on the default psy
    kernel and with VB200_PSY_V2 / VB200_PSY_V1 forcing the psy2 and the generic kernel"""
    name, setup, ctx, o, _, _ = cfg
    if psy != "default":
        monkeypatch.setenv(psy, "1")
    pcm, desc = _blocks(setup, W, 40, 606 + W)
    want = o.phaseA(W, pcm, desc, taps=True)
    got = ctx.phaseA(W, pcm, desc, taps=True)
    for k in ("mdct_raw", "logfft", "noise", "tone", "logmdct", "logmask", "mdct", "ampmax_out"):
        assert_bits_equal(got[k], want[k], "%s taps %s" % (psy, k))
    got = ctx.phaseA(W, pcm, desc, taps=False)
    for k in ("mdct", "logmdct", "logmask", "ampmax_out"):
        assert_bits_equal(got[k], want[k], "%s no taps %s" % (psy, k))


@pytest.mark.parametrize("W", [0, 1])
def test_encode_dsp_classes_vs_oracle(cfg, W, monkeypatch):
    """the one-call chain handing back the residue partition classes, in chunks of 3 blocks with a ragged last one,
    against the oracle's chain followed by its residue_classify"""
    name, setup, ctx, o, _, _ = cfg
    monkeypatch.setenv("VB200_CHUNK_BLOCKS", "3")
    pcm, desc = _blocks(setup, W, 11, 919 + W)
    want = o.encode_dsp(W, pcm, desc)
    wcls = o.residue_classify(W, want["iwork"], want["nonzero"])
    assert wcls.max() > 0 and not want["nonzero"][0].any()
    got = ctx.encode_dsp(W, pcm, desc, classes=True)
    for k in ("posts", "nonzero", "iwork"):
        assert np.array_equal(got[k], want[k]), k
    assert np.array_equal(got["classes"], wcls), "classes"
    if not (setup.channels & (setup.channels - 1)):
        got = ctx.encode_dsp(W, pcm, desc, classes=True, iwork_s16=True)
        assert np.array_equal(got["classes"], wcls), "classes with the int16 residue"


def _recorded(args, setup):
    """(test name, record, timeline) of every encoding the reference recorded for setup `args`"""
    out = []
    for test, signal in RECORDED.items():
        rec = refrec.Case(test, *args)
        if "timeline" in rec:
            out.append((test, rec, refrec.timeline(rec, signal(args[0], args[1]), setup.blocksize(1) // 2)))
    assert out, "no recorded encoding for %s" % (args,)
    return out


@pytest.mark.parametrize("fmt", ["f32", "s16"])
def test_encode_streams_on_reference_timelines(cfg, fmt):
    """vb200_encode_streams (envelope search, block planning, both block sizes, the ampmax chain across sizes in one
    call) on the stream buffers the reference encoded: the block plan must be the reference's (f32), and every
    block's posts, nonzero flags and residue the oracle's composition for the same timeline; with the reference
    built, f32 residue and nonzero flags also against the reference's own encoder"""
    from oracle import pyref
    name, setup, ctx, o, _, _ = cfg
    args = next(a for a in SETUPS if refrec.case_id(*a) == name)
    ch = setup.channels
    recs = _recorded(args, setup)
    stride = (max(tl.shape[1] for _, _, tl in recs) + 3) & ~3
    tl = np.zeros((len(recs), ch, stride), np.float32)
    for i, (_, _, t) in enumerate(recs):
        tl[i, :, :t.shape[1]] = t
    pcm_len = np.array([t.shape[1] for _, _, t in recs], np.int64)
    eof = np.array([t.shape[1] - int(rec["tail"]) for _, rec, t in recs], np.int64)
    if fmt == "f32":
        got = ctx.encode_streams(tl, pcm_len, eof)
    else:
        s16 = np.clip(np.rint(tl * 32767.0), -32768, 32767).astype(np.int16)
        tl = s16.astype(np.float32) / np.float32(32768.0)
        got = ctx.encode_streams(np.ascontiguousarray(s16.transpose(0, 2, 1)), pcm_len, eof, fmt=vlib.PCM_S16_INTERLEAVED)
    sizes = set()
    for i, (test, rec, _) in enumerate(recs):
        wplan, wouts = o.encode_stream(tl[i], int(pcm_len[i]), int(eof[i]))
        k = len(wplan)
        assert got["nblocks"][i] == k, "%s: %d blocks, want %d" % (test, got["nblocks"][i], k)
        plan = got["plan"][i, :k]
        for nm in ("W", "lW", "nW", "blocktype", "pos"):
            assert np.array_equal(plan[nm], wplan[nm]), "%s plan %s" % (test, nm)
            if fmt == "f32":
                assert np.array_equal(plan[nm], rec[nm]), "%s plan %s vs reference" % (test, nm)
        cap = None
        if fmt == "f32" and pyref.available():
            r = pyref.Ref(*args)
            cap = r.encode_capture(RECORDED[test](args[0], args[1]), fields=("iwork_out",))
            r.close()
            assert cap["nblocks"] == k
        for b in range(k):
            W, slot = int(plan[b]["W"]), int(plan[b]["slot"])
            sizes.add(W)
            g, w = got[W], wouts[b]
            assert np.array_equal(g["posts"][slot], w["posts"][0]), "%s block %d posts" % (test, b)
            assert np.array_equal(g["nonzero"][slot], w["nonzero"][0]), "%s block %d nonzero" % (test, b)
            assert np.array_equal(g["iwork"][slot], w["iwork"][0]), "%s block %d residue" % (test, b)
            assert_bits_equal(g["ampmax_out"][slot:slot + 1], w["ampmax_out"], "%s block %d ampmax" % (test, b))
            if cap is not None:
                n = setup.blocksize(W) // 2
                assert np.array_equal(g["nonzero"][slot], cap["nonzero_out"][b]), "%s block %d nonzero vs reference" % (test, b)
                assert np.array_equal(g["iwork"][slot], cap["iwork_out"][b][:, :n]), "%s block %d residue vs reference" % (test, b)
    assert sizes == {0, 1}, "the streams hold blocks of both sizes"


def test_device_vs_reference_records(cfg):
    """the CUDA path on the reference's own blocks checked directly against the reference's recorded digests, not
    through the oracle: Phase A with its taps and Phase B (pair), the one-call chain (encode), floor 1 fit and
    render (floor1), whichever of them tests/golden/ref_records.xz holds for this setup"""
    name, setup, ctx, o, _, _ = cfg
    args = next(a for a in SETUPS if refrec.case_id(*a) == name)
    for test, rec, _ in _recorded(args, setup):
        enc = refrec.Encoding(rec, setup, RECORDED[test](args[0], args[1]))
        for W in (0, 1):
            idx = enc.idx(W)
            if not len(idx):
                continue
            blocks, desc = enc.blocks(W, idx), enc.desc(idx)
            rec.check(blocks, "pcm_%d" % W, "W%d blocks" % W)
            if test == "pair":
                out = ctx.phaseA(W, blocks, desc, taps=True)
                for k, g in (("mdct_raw", "mdct_raw"), ("logfft", "logfft"), ("noise", "noise"), ("tone", "tone"),
                             ("logmdct", "logmdct"), ("logmask", "logmask"), ("mdct", "mdct_m1"),
                             ("ampmax_out", "ampmax_out"), ("logmask", "batch_logmask"), ("mdct", "batch_mdct")):
                    rec.check(out[k], "%s_%d" % (g, W), "CUDA W%d %s" % (W, k))
                for bt in (0, 1):
                    sel = np.where((enc.W == W) & (rec["blocktype"] == bt))[0]
                    if not len(sel):
                        continue
                    inp = encoder_outputs(ctx, enc, W, sel)
                    for k, g in (("mdct", "mdct_m1"), ("ilogmask", "ilogmask"), ("nonzero_in", "nonzero_in")):
                        rec.check(inp[k], "%s_%d_%d" % (g, W, bt), "CUDA Phase B input %s" % g)
                    iw, nz = ctx.couple_quantize_normalize(W, bt, 7, inp["mdct"], inp["ilogmask"], inp["nonzero_in"])
                    rec.check(iw, "iwork_out_%d_%d" % (W, bt), "CUDA iwork")
                    rec.check(nz, "nonzero_out_%d_%d" % (W, bt), "CUDA nonzero")
            elif test == "encode":
                a = ctx.encode_dsp(W, blocks, desc)
                for k in ("posts", "nonzero", "iwork", "ampmax_out"):
                    rec.check(a[k], "batch_%s_%d" % (k, W), "CUDA encode_dsp " + k)
                rec.check(a["iwork"], "iwork_out_%d" % W, "CUDA iwork vs the API loop's capture")
            else:
                a = ctx.phaseA(W, blocks, desc)
                rec.check(a["logmdct"], "logmdct_%d" % W, "CUDA logmdct")
                rec.check(a["logmask"], "logmask_%d" % W, "CUDA logmask")
                posts, nz = ctx.floor1_fit(W, a["logmdct"], a["logmask"])
                rec.check(nz, "fit_nonzero_%d" % W, "CUDA fit nonzero")
                rec.check(posts, "fit_posts_%d" % W, "CUDA fit posts")
                p2, ilog, nz2 = ctx.floor1_render(W, posts, nz)
                rec.check(p2[nz == 1], "enc_posts_%d" % W, "CUDA floor1_encode posts")
                rec.check(ilog, "ilogmask_%d" % W, "CUDA ilogmask")
                rec.check(nz2, "nonzero_in_%d" % W, "CUDA nonzero")
