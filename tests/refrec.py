"""What the compiled reference computed for tests/test_oracle_vs_ref.py and tests/test_plan_vs_ref.py,
recorded by tests/golden/make_golden_ref.py, so that those comparisons run without the reference.

tests/golden/ref_records.xz holds, per test case, the small results as they are (block plans, envelope
marks, counts) and every large array as a SHA-256 digest of its dtype, shape and bytes: a test computes the
array with the oracle and compares digests, which is the same bit-exact comparison.  Integer arrays are
digested as int64, since the tests compare integers by value.  The file is LZMA-compressed: one line of JSON
mapping each key to its digest or to [dtype, shape, offset] of an array in the byte pool that follows;
identical arrays are stored once.

The reference encodes from a stream buffer (the timeline): an LPC-extrapolated preamble of blocksizes[1]/2
samples, the input, and an LPC-extrapolated tail after the end of the stream.  The input is the test's own
seeded signal; the two extrapolations are rebuilt here from the reference's recorded LPC coefficients, and
the rebuilt timeline is checked against the reference's digest before anything uses it.

The file also holds the encoder setups of the configurations that have no setup_*.npz (keys setup/<case>/)."""
import hashlib
import json
import lzma
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RECORDS = os.path.join(GOLDEN, "ref_records.xz")


def case_id(ch, rate, q):
    return "ch%d_%d_q%g" % (ch, rate, q)


def digest(a):
    a = np.ascontiguousarray(a)
    if a.dtype.kind in "iub":
        a = a.astype(np.int64)
    h = hashlib.sha256(("%s%s" % (a.dtype.str, a.shape)).encode())
    h.update(a.tobytes())
    return h.hexdigest()[:24]


def save(path, records):
    """write `records` (key -> digest string or array) in the format records() reads"""
    index, pool, where = {}, bytearray(), {}
    for k, v in records.items():
        if isinstance(v, str):
            index[k] = v
            continue
        v = np.asarray(v)
        ident = (v.dtype.str, v.shape, np.ascontiguousarray(v).tobytes())
        if ident not in where:
            where[ident] = len(pool)
            pool += ident[2]
        index[k] = [v.dtype.str, list(v.shape), where[ident]]
    with lzma.open(path, "wb", preset=9 | lzma.PRESET_EXTREME) as f:
        f.write(json.dumps(index, sort_keys=True).encode() + b"\n")
        f.write(bytes(pool))


_records = None


def records():
    global _records
    if _records is None:
        with lzma.open(RECORDS) as f:
            index = json.loads(f.readline())
            pool = f.read()
        _records = {}
        for k, v in index.items():
            if not isinstance(v, str):
                dt, shape, off = np.dtype(v[0]), tuple(v[1]), v[2]
                v = np.frombuffer(pool, dt, int(np.prod(shape)), off).reshape(shape).copy()
            _records[k] = v
    return _records


class Case:
    """The recorded results of one test case: `case[key]` is a stored array, `case.check(got, key)` asserts
    that `got` is bit-identical to the reference's array recorded under `key`."""

    def __init__(self, test, ch, rate, q, tag=None):
        self.prefix = "%s/%s%s/" % (test, case_id(ch, rate, q), "" if tag is None else "_" + tag)
        self.r = records()

    def __getitem__(self, key):
        return self.r[self.prefix + key]

    def __contains__(self, key):
        return self.prefix + key in self.r

    def check(self, got, key, what=None):
        assert digest(got) == str(self[key]), "%s differs from the reference's (%s%s)" % (what or key, self.prefix, key)


def setup(ch, rate, q):
    from conftest import GOLDEN as FIXTURES, REF_ARGS
    from vorbis_b200 import abi
    for name, args in REF_ARGS.items():
        if args == (ch, rate, q):
            return abi.SetupHolder.load(os.path.join(FIXTURES, "setup_%s.npz" % name))
    pre = "setup/%s/" % case_id(ch, rate, q)
    return abi.SetupHolder({k[len(pre):]: v for k, v in records().items() if k.startswith(pre)})


def lpc_predict(coeff, prime, n):
    """n samples per row of the all-pole predictor `coeff` [rows][m] run on from `prime` [rows][m] (the m
    samples before the first predicted one), in float32 and in the reference's summation order:
    y[i] = -sum_j x[i-m+j] * coeff[m-1-j], j ascending."""
    rows, m = coeff.shape
    work = np.zeros((rows, m + n), np.float32)
    work[:, :m] = prime
    c = np.ascontiguousarray(coeff[:, ::-1], np.float32)
    for i in range(n):
        y = np.zeros(rows, np.float32)
        for j in range(m):
            y -= work[:, i + j] * c[:, j]
        work[:, i + m] = y
    return work[:, m:]


def timeline(case, pcm, preamble):
    """The reference's stream buffer for input `pcm` [ch][S]: `preamble` samples extrapolated backwards
    from the start of the input (case["lpc_head"]), the input, and case["tail"] samples extrapolated on
    from its end (case["lpc_tail"]; none if the case has no tail).  Checked against case["timeline"]."""
    head_lpc = case["lpc_head"]
    m = head_lpc.shape[1]
    parts = [lpc_predict(head_lpc, pcm[:, :m][:, ::-1], preamble)[:, ::-1], pcm]
    if "lpc_tail" in case:
        tail_lpc = case["lpc_tail"]
        parts.append(lpc_predict(tail_lpc, pcm[:, -tail_lpc.shape[1]:], int(case["tail"])))
    tl = np.ascontiguousarray(np.concatenate(parts, axis=1), np.float32)
    case.check(tl, "timeline", "the rebuilt stream buffer")
    return tl


class Encoding:
    """The blocks the reference's encoder cut from the timeline of `pcm` (case["W"], ["lW"], ["nW"],
    ["blocktype"], ["pos"]) and the ampmax each of them was handed (case["ampmax_in"])."""

    def __init__(self, case, setup, pcm):
        self.case, self.bs = case, [setup.blocksize(0), setup.blocksize(1)]
        self.tl = timeline(case, pcm, self.bs[1] // 2)
        self.W = case["W"]

    def idx(self, W):
        return np.where(self.W == W)[0]

    def blocks(self, W, idx):
        N = self.bs[W]
        return np.ascontiguousarray(np.stack([self.tl[:, p:p + N] for p in self.case["pos"][idx]]))

    def desc(self, idx):
        from vorbis_b200 import abi
        d = np.zeros(len(idx), abi.BLOCKDESC_DTYPE)
        for k in ("lW", "nW", "blocktype"):
            d[k] = self.case[k][idx]
        d["ampmax"] = self.case["ampmax_in"][idx]
        return d
