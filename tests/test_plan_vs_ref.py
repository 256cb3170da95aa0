"""Block planning (SURVEY §8 a15): the oracle's restatement of what vorbis_analysis_blockout decides per block
(W, lW, nW, blocktype, position) must equal the reference's own block sequence, captured while the unmodified
reference encodes a stream through its public API.  The reference's sequences are recorded in
tests/golden/ref_records.xz by tests/golden/make_golden_ref.py (see tests/refrec.py)."""
import numpy as np
import pytest

import refrec
from conftest import probe_signal
from oracle import pyoracle

GRID = [(2, 44100, .5), (1, 44100, .4), (2, 44100, .1), (1, 22050, .3), (6, 48000, .2), (2, 48000, .9), (2, 32000, 0.),
        (2, 44100, -.1)]


def burst_signal(ch, rate, secs, seed):
    rng = np.random.default_rng(seed)
    ns = int(rate * secs)
    t = np.arange(ns)
    pcm = np.stack([0.1 * rng.uniform(-1, 1, ns) + 0.4 * np.sin(2 * np.pi * (300 + 70 * c) * t / rate)
                    for c in range(ch)]).astype(np.float32)
    for _ in range(6):
        a = int(rng.integers(2000, ns - 3000))
        pcm[:, a:a + 200] *= 0.02
        pcm[:, a + 200:a + 260] = rng.uniform(-0.9, 0.9, (ch, 60))
    return pcm


def plan_signal(ch, rate, mode):
    return probe_signal(ch, rate, 1.5, 7) if mode == "probe" else burst_signal(ch, rate, 1.5, 7)


def config1_signal():
    t = np.arange(44100)
    return (0.8 * np.sin(2 * np.pi * 440.0 * t / 44100.0)).astype(np.float32)[None]


@pytest.mark.parametrize("mode", ["probe", "bursts"])
@pytest.mark.parametrize("ch,rate,q", GRID)
def test_oracle_plan_equals_reference_block_sequence(ch, rate, q, mode):
    rec = refrec.Case("plan", ch, rate, q, mode)
    setup = refrec.setup(ch, rate, q)
    tl = refrec.timeline(rec, plan_signal(ch, rate, mode), setup.blocksize(1) // 2)
    o = pyoracle.Oracle(setup)
    mark, nsteps = o.timeline_marks(tl[None])
    plan, nb = o.plan_blocks(mark, nsteps, [tl.shape[1]], [int(rec["eof"])])
    k = int(rec["nblocks"])
    assert nb[0] == k and (rec["W"] == 0).sum() >= 5           # the signals do switch block sizes
    for name in ("W", "lW", "nW", "blocktype"):
        assert np.array_equal(plan[0, :k][name], rec[name]), name
    for b in range(k):                                          # positions: the block is that slice of the timeline
        N = setup.blocksize(int(rec["W"][b]))
        p = plan[0, b]["pos"]
        rec.check(tl[:, p:p + N], "block_%d" % b, "block %d position" % b)


def test_config1_plumbing_numbers():
    """BASELINE config 1 (SURVEY §8d): 1 s mono 44.1 kHz 440 Hz sine (0.8 amplitude, float), q=0.4 through the
    reference API.  The committed driver (oracle/ref_driver.c ref_encode_capture: 1024-sample
    vorbis_analysis_wrote calls, then wrote(0); audio packets only) gives 46 blocks = 2 short + 44 long and
    1705 packet bytes.  (SURVEY §8d quotes 47 / 2+45 / 1851 from a survey-time probe whose source was not
    kept; block count and bytes depend on the write chunking - 45..46 blocks, 1615..1705 bytes for chunks
    of 256..44100 samples - so the pinned numbers are the ones this repository can reproduce.)"""
    rec = refrec.Case("plan", 1, 44100, .4, "config1")
    assert int(rec["nblocks"]) == 46
    assert int((rec["W"] == 0).sum()) == 2 and int((rec["W"] == 1).sum()) == 44
    assert int(rec["bytes"]) == 1705
    setup = refrec.setup(1, 44100, .4)
    tl = refrec.timeline(rec, config1_signal(), setup.blocksize(1) // 2)
    o = pyoracle.Oracle(setup)
    mark, nsteps = o.timeline_marks(tl[None])
    plan, nb = o.plan_blocks(mark, nsteps, [tl.shape[1]], [int(rec["eof"])])
    assert nb[0] == 46 and np.array_equal(plan[0, :46]["W"], rec["W"])
