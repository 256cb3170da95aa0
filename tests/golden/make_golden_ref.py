#!/usr/bin/env python
"""Record what the REFERENCE computes for tests/test_oracle_vs_ref.py and tests/test_plan_vs_ref.py.

Runs only where oracle/_ref/libvorbis_ref.so was built (the unmodified reference sources compiled by
oracle/Makefile).  Each case below runs the reference on exactly the inputs the test builds (the same
seeded signals, the same random vectors) and keeps what the test compares against; tests/refrec.py
describes the format.  Before writing, the rebuild (tests/refrec.py) of every recorded timeline is checked
here against the reference's own buffer.

  ref_records.xz    block plans, marks, counts, LPC coefficients and digests of the large arrays, and the
                    setups of the configurations without a setup_<cfg>.npz

usage:  python tests/golden/make_golden_ref.py
"""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
import refrec  # noqa: E402
from conftest import REF_ARGS  # noqa: E402
from oracle import pyoracle, pyref  # noqa: E402
from vorbis_b200 import abi  # noqa: E402
import test_oracle_vs_ref as T  # noqa: E402
import test_plan_vs_ref as P  # noqa: E402

CHUNK = 1024        # samples per vorbis_analysis_wrote of ref_encode_capture
REC = {}
SETUPS = {}


def lpc_from_data(x, order):
    """the reference's own vorbis_lpc_from_data on x [n] -> float32 [order]"""
    x = np.ascontiguousarray(x, np.float32)
    out = np.zeros(order, np.float32)
    pyref.lib().vorbis_lpc_from_data(x.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p),
                                     C.c_int(len(x)), C.c_int(order))
    return out


class Rec:
    def __init__(self, test, args, tag=None):
        self.case = refrec.Case.__new__(refrec.Case)
        self.case.prefix = "%s/%s%s/" % (test, refrec.case_id(*args), "" if tag is None else "_" + tag)
        self.case.r = REC
        ch, rate, q = args
        if args not in REF_ARGS.values() and refrec.case_id(*args) not in SETUPS:
            s = pyref.Ref(ch, rate, q)
            SETUPS[refrec.case_id(*args)] = s.setup().arrays
            s.close()

    def put(self, key, value):
        REC[self.case.prefix + key] = np.asarray(value)

    def dig(self, key, a):
        REC[self.case.prefix + key] = refrec.digest(a)

    def timeline(self, pcm, tl, first, eof=None):
        """LPC coefficients of the preamble (extrapolated backwards from the first `first` input samples,
        order 16, lib/block.c _preextrapolate_helper) and of the tail (order 32 from the last blocksizes[1]
        samples, lib/block.c vorbis_analysis_wrote(v,0)); checks the rebuild against `tl`"""
        ch, S = pcm.shape
        pre = tl.shape[1] - S if eof is None else eof - S
        self.put("lpc_head", np.stack([lpc_from_data(pcm[c, :first][::-1], 16) for c in range(ch)]))
        if eof is not None:
            n = min(eof, 2 * pre)
            self.put("lpc_tail", np.stack([lpc_from_data(tl[c, eof - n:eof], 32) for c in range(ch)]))
            self.put("tail", tl.shape[1] - eof)
        self.dig("timeline", tl)
        assert np.array_equal(refrec.timeline(self.case, pcm, pre).view(np.uint32), tl.view(np.uint32))

    def encoding(self, r, pcm, cap):
        """the recorded capture's plan, the timeline, the block positions in it"""
        bs1 = r.bs[1]
        self.timeline(pcm, cap["timeline"], min(pcm.shape[1], CHUNK * (bs1 // CHUNK + 1)), cap["eof"])
        k = cap["nblocks"]
        for f in ("W", "lW", "nW", "blocktype", "ampmax_in"):
            self.put(f, cap[f][:k])
        o = pyoracle.Oracle(r.setup())
        mark, nsteps = o.timeline_marks(cap["timeline"][None])
        plan, nb = o.plan_blocks(mark, nsteps, [cap["timeline"].shape[1]], [cap["eof"]])
        assert nb[0] == k
        pos = plan[0, :k]["pos"].astype(np.int64)
        for b in range(k):
            N = r.bs[cap["W"][b]]
            assert np.array_equal(cap["pcm"][b][:, :N], cap["timeline"][:, pos[b]:pos[b] + N])
        self.put("pos", pos)
        o.close()
        enc = refrec.Encoding(self.case, r.setup(), pcm)
        for W in (0, 1):
            idx = enc.idx(W)
            if len(idx):
                self.dig("pcm_%d" % W, cap["pcm"][idx][:, :, :r.bs[W]])
        return enc


def pair_cases():
    for args in T.GRID:
        ch, rate, q = args
        rc = Rec("pair", args)
        r = pyref.Ref(ch, rate, q)
        pcm = T.pair_signal(ch, rate)
        cap = r.encode_capture(pcm, timeline=True)
        rc.encoding(r, pcm, cap)
        for W in (0, 1):
            for which in (0, 1, 2, 3):
                rc.dig("table_%d_%d" % (W, which), r.table(W, which))
        for W, x, y, lW, nW in T.transform_inputs([r.bs[0], r.bs[1]]):
            rc.dig("mdct_forward_%d" % W, r.mdct_forward(W, x))
            rc.dig("mdct_backward_%d" % W, r.mdct_backward(W, y))
            rc.dig("drft_forward_%d" % W, r.drft_forward(W, x))
            rc.dig("window_%d" % W, r.apply_window(W, x, lW, nW))
        for W in (0, 1):
            idx = np.where(cap["W"] == W)[0]
            if not len(idx):
                continue
            N = r.bs[W]
            n = N // 2
            for g in ("mdct_raw", "logfft", "noise", "tone", "logmdct", "logmask", "mdct_m1"):
                rc.dig("%s_%d" % (g, W), cap[g][idx][:, :, :n])
            rc.dig("ampmax_out_%d" % W, cap["ampmax_out"][idx])
            desc = np.zeros(len(idx), abi.BLOCKDESC_DTYPE)
            for k in ("lW", "nW", "blocktype"):
                desc[k] = cap[k][idx]
            desc["ampmax"] = cap["ampmax_in"][idx]
            m, lmd, lmk, amp = r.phaseA_batch(W, cap["pcm"][idx][:, :, :N], desc)
            rc.dig("batch_logmask_%d" % W, lmk)
            rc.dig("batch_mdct_%d" % W, m)
            for bt in (0, 1):
                sel = np.where((cap["W"] == W) & (cap["blocktype"] == bt))[0]
                if not len(sel):
                    continue
                for f in ("mdct_m1", "ilogmask", "iwork_out"):
                    rc.dig("%s_%d_%d" % (f, W, bt), cap[f][sel][:, :, :n])
                for f in ("nonzero_in", "nonzero_out"):
                    rc.dig("%s_%d_%d" % (f, W, bt), cap[f][sel])
        d = r.decode_capture(cap["nblocks"] + 4, pcm.shape[1] + 8192)
        rc.put("dec_W", d["W"])
        rc.dig("dec_coef", np.concatenate([d["dec_coef"][k][:, :r.bs[d["W"][k]] // 2].reshape(-1) for k in range(len(d["W"]))]))
        rc.put("dec_len", d["pcm"].shape[1])
        rc.dig("dec_pcm", d["pcm"])
        r.close()


def floor1_cases():
    for args in T.FLOOR1_ARGS:
        ch, rate, q = args
        rc = Rec("floor1", args)
        r = pyref.Ref(ch, rate, q)
        pcm = T.floor1_signal(ch, rate)
        cap = r.encode_capture(pcm, timeline=True)
        rc.encoding(r, pcm, cap)
        for W in (0, 1):
            idx = np.where(cap["W"] == W)[0]
            if not len(idx):
                continue
            n = r.bs[W] // 2
            want = cap["fit_posts"][idx].reshape(-1, abi.FLOOR1_STRIDE).copy()
            wnz = (want[:, 0] != -1).astype(np.int32)
            want[wnz == 0] = 0
            rc.dig("logmdct_%d" % W, cap["logmdct"][idx][:, :, :n])
            rc.dig("logmask_%d" % W, cap["logmask"][idx][:, :, :n])
            rc.dig("fit_nonzero_%d" % W, wnz)
            rc.dig("fit_posts_%d" % W, want)
            rc.dig("enc_posts_%d" % W, cap["enc_posts"][idx].reshape(-1, abi.FLOOR1_STRIDE)[wnz == 1])
            rc.dig("ilogmask_%d" % W, cap["ilogmask"][idx][:, :, :n].reshape(-1, n))
            rc.dig("nonzero_in_%d" % W, cap["nonzero_in"][idx].reshape(-1))
        r.close()


def encode_cases():
    for args in T.ENCODE_ARGS:
        ch, rate, q = args
        rc = Rec("encode", args)
        r = pyref.Ref(ch, rate, q)
        pcm = T.encode_signal(ch, rate)
        cap = r.encode_capture(pcm, timeline=True)
        rc.encoding(r, pcm, cap)
        for W in (0, 1):
            idx = np.where(cap["W"] == W)[0]
            if not len(idx):
                continue
            N = r.bs[W]
            desc = np.zeros(len(idx), abi.BLOCKDESC_DTYPE)
            for k in ("lW", "nW", "blocktype"):
                desc[k] = cap[k][idx]
            desc["ampmax"] = cap["ampmax_in"][idx]
            b = r.encode_dsp_batch(W, np.ascontiguousarray(cap["pcm"][idx][:, :, :N]), desc)
            for k in ("posts", "nonzero", "iwork", "ampmax_out"):
                rc.dig("batch_%s_%d" % (k, W), b[k])
            rc.dig("iwork_out_%d" % W, cap["iwork_out"][idx][:, :, :N // 2])
        r.close()


def managed_cases():
    for args in T.MANAGED_ARGS:
        ch, rate, q = args
        rc = Rec("managed", args)
        r = pyref.Ref(ch, rate, q)
        pcm = T.managed_signal(ch, rate)
        cap = r.encode_capture(pcm, timeline=True)
        rc.encoding(r, pcm, cap)
        for W in (0, 1):
            idx = np.where(cap["W"] == W)[0][:10]
            if not len(idx):
                continue
            N = r.bs[W]
            desc = np.zeros(len(idx), abi.BLOCKDESC_DTYPE)
            for k in ("lW", "nW", "blocktype"):
                desc[k] = cap[k][idx]
            desc["ampmax"] = cap["ampmax_in"][idx]
            b = r.encode_dsp_managed_batch(W, np.ascontiguousarray(cap["pcm"][idx][:, :, :N]), desc)
            for k in ("posts", "nonzero", "iwork", "ampmax_out"):
                rc.dig("managed_%s_%d" % (k, W), b[k])
        r.close()


def envelope_cases():
    for args in T.ENVELOPE_ARGS:
        ch, rate, q = args
        rc = Rec("envelope", args)
        r = pyref.Ref(ch, rate, q)
        pcm = T.envelope_signal(ch, rate)
        marks, steps, st, stream = r.envelope_marks(pcm)
        rc.timeline(pcm, stream, pcm.shape[1])
        rc.put("marks", marks)
        rc.put("steps", steps)
        rc.put("state", st)
        r.close()


def inverse2_cases():
    for args in T.INVERSE2_ARGS:
        ch, rate, q = args
        rc = Rec("inverse2", args)
        r = pyref.Ref(ch, rate, q)
        for W, posts, present, data in T.inverse2_inputs(ch, r.bs):
            rc.dig("inverse2_%d" % W, r.floor1_inverse2(W, posts, present, data))
        r.close()


def residue_cases():
    for args in T.RESIDUE_ARGS:
        ch, rate, q = args
        rc = Rec("residue", args)
        r = pyref.Ref(ch, rate, q)
        o = pyoracle.Oracle(r.setup())
        for W, iwork, nonzero in T.residue_inputs(ch, r.bs):
            rc.dig("classes_%d" % W, r.residue_classify(W, iwork, nonzero, o.residue_partvals(W)))
        o.close()
        r.close()


def plan_cases():
    for mode in ("probe", "bursts"):
        for args in P.GRID:
            ch, rate, q = args
            rc = Rec("plan", args, mode)
            r = pyref.Ref(ch, rate, q)
            pcm = P.plan_signal(ch, rate, mode)
            cap = r.encode_capture(pcm, fields=("pcm",), timeline=True)
            rc.timeline(pcm, cap["timeline"], min(pcm.shape[1], CHUNK * (r.bs[1] // CHUNK + 1)), cap["eof"])
            k = cap["nblocks"]
            rc.put("eof", cap["eof"])
            rc.put("nblocks", k)
            for name in ("W", "lW", "nW", "blocktype"):
                rc.put(name, cap[name][:k])
            for b in range(k):
                rc.dig("block_%d" % b, cap["pcm"][b][:, :r.bs[cap["W"][b]]])
            r.close()
    args = (1, 44100, 0.4)
    rc = Rec("plan", args, "config1")
    r = pyref.Ref(*args)
    pcm = P.config1_signal()
    cap = r.encode_capture(pcm, fields=("pcm",), timeline=True)
    rc.timeline(pcm, cap["timeline"], min(pcm.shape[1], CHUNK * (r.bs[1] // CHUNK + 1)), cap["eof"])
    for name in ("eof", "nblocks", "bytes"):
        rc.put(name, cap[name])
    rc.put("W", cap["W"][:cap["nblocks"]])
    r.close()


def main():
    if not pyref.available():
        sys.exit("oracle/_ref/libvorbis_ref.so is not built")
    pyoracle.build()
    for name, args in REF_ARGS.items():      # the committed fixtures are the reference's setups
        r = pyref.Ref(*args)
        with np.load(os.path.join(HERE, "setup_%s.npz" % name)) as z:
            have = r.setup().arrays
            assert sorted(z.files) == sorted(have) and all(np.array_equal(z[k], have[k]) for k in z.files), name
        r.close()
    for f in (pair_cases, floor1_cases, encode_cases, managed_cases, envelope_cases, inverse2_cases,
              residue_cases, plan_cases):
        f()
    REC.update({"setup/%s/%s" % (c, k): v for c, a in SETUPS.items() for k, v in a.items()})
    refrec.save(refrec.RECORDS, REC)
    print("%d records, %d extra setups" % (len(REC), len(SETUPS)))


if __name__ == "__main__":
    main()
