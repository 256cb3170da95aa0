#!/usr/bin/env python
"""bench.py — per-block encode DSP of mapping0_forward (window + MDCT + FFT + noise/tone masks + mix
+ floor1 fit/render + couple/quantise/normalise) throughput.

  python bench.py --gpus N --steps K --warmup W          our CUDA path (default N=1)
  python bench.py --impl reference ...                   the reference's CPU code on the host cores

Workload (BASELINE.json configs[2]): 44.1 kHz stereo, vorbis_encode_init_vbr q=0.5, 100 000
long blocks (N=2048 samples -> 1024 spectral lines per channel: the "N=1024" of the metric;
SURVEY.md §8d) per GPU per step, synthetic PCM, independent blocks with ampmax given per block
(drop-in semantics).  One step = one pass of the hot path over that batch: ONE vb200_encode_dsp_dev
call = six kernels (transform, ampmax, psy, floor1_fit, floor1_render, couple_quantize_normalize).
`e2e` is the same chain through vb200_encode_dsp with pinned HOST buffers: int16 interleaved stream
PCM in (blocks cut on the device, hop N/2), floor posts + quantised residue (int16) out.  The reference arm
and cpu_baseline run the same chain with the reference's own functions.

One JSON line on stdout (rank 0).  See DESIGN.md "Measurement" for the byte accounting.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLD = os.path.join(ROOT, "tests", "golden")
METRIC = "stereo_blocks_per_sec_mdct_psy"
UNIT = "blocks/s"
W_LONG = 1


def workload_name(nblocks, N, ch):
    return ("mapping0_forward per-block DSP (window+MDCT+FFT+noise/tone mask+mix, floor1 fit+render, "
            "couple/quantise/normalise), 44.1kHz stereo q=0.5, "
            "%d long blocks x %d ch x N=%d samples (n=%d lines/ch)" % (nblocks, ch, N, N // 2))


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def count(self):
        return len(self.lines)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------
def synth_pcm_torch(torch, nblocks, ch, N, rate, device, seed):
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    t = torch.arange(N, device=device, dtype=torch.float32)
    pcm = torch.rand((nblocks, ch, N), generator=g, device=device, dtype=torch.float32)
    pcm.mul_(0.5).sub_(0.25)                                     # 0.25*uniform(-1,1)
    f = 440.0 + 110.0 * torch.arange(ch, device=device, dtype=torch.float32).view(1, ch, 1)
    ph = torch.rand((nblocks, 1, 1), generator=g, device=device) * 6.2831853
    pcm.add_(0.5 * torch.sin(2 * np.pi * f * t.view(1, 1, N) / rate + ph))
    return pcm


def make_desc(nblocks):
    from vorbis_b200 import abi
    d = np.zeros(nblocks, abi.BLOCKDESC_DTYPE)
    d["lW"] = 1; d["nW"] = 1; d["blocktype"] = 1          # steady-state long blocks (psy look 3)
    d["ampmax"] = -6.0
    return d


def usable_cpus():
    """CPUs this process may really run on: the affinity mask, capped by the cgroup CPU quota
    (a container can show 128 CPUs in its mask and own a fraction of them)."""
    try:
        cpus = sorted(os.sched_getaffinity(0))
    except AttributeError:
        cpus = list(range(os.cpu_count() or 1))
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            f = open(path).read().split()
            if path.endswith("cpu.max"):
                if f[0] != "max":
                    quota = float(f[0]) / float(f[1])
            else:
                q = float(f[0])
                if q > 0:
                    quota = q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            break
        except Exception:
            continue
    n = len(cpus)
    if quota is not None:
        n = max(1, min(n, int(quota)))
    return cpus[:n], {"affinity": len(cpus), "cgroup_quota": quota, "os_cpu_count": os.cpu_count()}


def bind_to_gpu_numa_node(torch, local):
    """Run this rank (and first-touch its pinned buffers) on the NUMA node its GPU hangs off: the H2D/D2H DMA of
    the end-to-end path then stays on one socket.  Returns a short description for the JSON line."""
    try:
        pr = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read())
        if node < 0:
            return {"gpu": bdf, "numa_node": None}
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = set(os.sched_getaffinity(0))
        use = sorted(cpus & allowed)
        if use:
            os.sched_setaffinity(0, use)
        return {"gpu": bdf, "numa_node": node, "cpus_bound": len(use)}
    except Exception as e:  # binding is an optimisation, never a reason to fail
        return {"error": repr(e)}


def cpu_worker_main(argv):
    """`bench.py --cpu-worker cpu blocks reps seed`: ONE process pinned to ONE cpu running the reference
    chain (oracle/_ref when built, else the oracle port) on its own synthetic blocks.  Protocol on
    stdin/stdout: prints "ready", waits for a line, runs `reps` passes, prints the elapsed seconds."""
    cpu, nb, reps, seed = int(argv[0]), int(argv[1]), int(argv[2]), int(argv[3])
    try:
        os.sched_setaffinity(0, {cpu})
    except Exception:
        pass
    from vorbis_b200 import abi
    from oracle import pyref
    setup = abi.SetupHolder.load(os.path.join(GOLD, "setup_44k_stereo_q5.npz"))
    N, ch = setup.blocksize(W_LONG), setup.channels
    rng = np.random.default_rng(seed)
    t = np.arange(N, dtype=np.float32)
    pcm = (0.25 * rng.uniform(-1, 1, (nb, ch, N)) +
           0.5 * np.sin(2 * np.pi * (440 + 110 * np.arange(ch)).reshape(1, ch, 1) * t / 44100.0
                        + rng.uniform(0, 6.28, (nb, 1, 1)))).astype(np.float32)
    desc = make_desc(nb)
    if pyref.available():
        kind = "reference"
        inst = pyref.Ref(ch, 44100, 0.5)
        run = lambda: inst.encode_dsp_batch(W_LONG, pcm, desc)
    else:
        kind = "port"
        from oracle import pyoracle
        inst = pyoracle.Oracle(setup)
        run = lambda: inst.encode_dsp(W_LONG, pcm, desc)
    run()                                              # page in / warm caches
    sys.stdout.write("ready %s\n" % kind); sys.stdout.flush()
    while True:
        line = sys.stdin.readline()
        if not line or line.startswith("quit"):
            return
        t0 = time.perf_counter()
        for _ in range(reps):
            run()
        sys.stdout.write("%.6f\n" % (time.perf_counter() - t0)); sys.stdout.flush()


class CpuPool:
    """One pinned worker PROCESS per cpu (the reference library is single threaded; blocks of different
    streams are independent - BASELINE.md section 3).  step() releases all workers at once and returns the
    wall time until the slowest one has finished."""

    def __init__(self, cpus, blocks_per_core, reps=1):
        self.cpus, self.nb, self.reps = list(cpus), blocks_per_core, reps
        self.procs = [subprocess.Popen([sys.executable, os.path.abspath(__file__), "--cpu-worker", str(c),
                                        str(blocks_per_core), str(reps), str(7000 + i)],
                                       stdin=subprocess.PIPE, stdout=subprocess.PIPE, text=True, cwd=ROOT)
                      for i, c in enumerate(self.cpus)]
        self.kind = None
        for p in self.procs:
            ln = p.stdout.readline().split()
            if not ln or ln[0] != "ready":
                raise RuntimeError("cpu worker failed to start")
            self.kind = ln[1]

    def step(self):
        t0 = time.perf_counter()
        for p in self.procs:
            p.stdin.write("go\n"); p.stdin.flush()
        per = [float(p.stdout.readline()) for p in self.procs]
        return time.perf_counter() - t0, per

    def blocks_per_step(self):
        return self.nb * self.reps * len(self.procs)

    def close(self):
        for p in self.procs:
            try:
                p.stdin.write("quit\n"); p.stdin.flush(); p.stdin.close()
            except Exception:
                pass
        for p in self.procs:
            try:
                p.wait(timeout=10)
            except Exception:
                p.kill()


def cpu_reference_rates(blocks_per_core, steps, warmup, single_core=True, cpus_info=None):
    """(all-core dict, 1-core dict or None).  Every step is a bounded sample: blocks_per_core long stereo
    blocks on every usable cpu."""
    cpus, info = cpus_info if cpus_info else usable_cpus()
    pool = CpuPool(cpus, blocks_per_core)
    try:
        for _ in range(warmup):
            pool.step()
        walls = [pool.step()[0] for _ in range(steps)]
    finally:
        pool.close()
    nb = pool.blocks_per_step()
    rate = nb * len(walls) / sum(walls)
    allc = {"value": rate, "unit": UNIT, "cores": len(cpus), "kind": pool.kind,
            "blocks_per_s_per_core": rate / len(cpus), "cpu_info": info, "ms_per_step": 1e3 * sum(walls) / len(walls),
            "sample": "%d long stereo blocks per step = %d on each of %d pinned single-threaded processes"
                      % (nb, blocks_per_core, len(cpus))}
    one = None
    if single_core:
        p1 = CpuPool(cpus[:1], blocks_per_core)
        try:
            p1.step()
            w = [p1.step()[0] for _ in range(max(2, min(steps, 3)))]
        finally:
            p1.close()
        one = {"value": blocks_per_core * len(w) / sum(w), "unit": UNIT, "cores": 1, "kind": p1.kind,
               "sample": "%d long stereo blocks per step on one pinned process" % blocks_per_core}
    return allc, one


# ------------------------------------------------------------------------------------------
def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from vorbis_b200 import abi
    setup = abi.SetupHolder.load(os.path.join(GOLD, "setup_44k_stereo_q5.npz"))
    N, ch = setup.blocksize(W_LONG), setup.channels
    allc, one = cpu_reference_rates(args.ref_blocks_per_core, args.steps, args.warmup)
    value = allc["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": allc["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.blocks, N, ch), "blocks_per_gpu": args.blocks,
                   "l2": "n/a (CPU)", "sharding": "independent blocks per rank, no collective",
                   "note": "each step is a bounded sample of the workload: " + allc["sample"]},
        "cpu_baseline": allc, "cpu_baseline_1core": one,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def extra_configs(torch, lib, abi, device, peak):
    """BASELINE configs[1] (batched mdct_forward N=1024 x 65536) and configs[3] (decode: IMDCT +
    overlap-add, mixed 256/2048 blocks), device resident, CUDA events.  Informational."""
    out = {}
    dev = torch.device("cuda", device)
    stream = torch.cuda.current_stream().cuda_stream

    def timed(fn, reps=5):
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    # config 2: mdct_init(1024), 65536 vectors uniform(-1,1)
    s22 = abi.SetupHolder.load(os.path.join(GOLD, "setup_22k_mono_q3.npz"))
    c22 = lib.Context(s22, device=device)
    N = s22.blocksize(1)
    nv = 65536
    g = torch.Generator(device=dev); g.manual_seed(12345)
    x = torch.rand((nv, N), generator=g, device=dev) * 2 - 1
    y = torch.empty((nv, N // 2), device=dev)
    ms = timed(lambda: c22.mdct_forward_dev(1, nv, x.data_ptr(), y.data_ptr(), stream))
    out["mdct_forward_N1024_x65536"] = {"ms": ms, "transforms_per_s": nv / ms * 1e3,
                                         "algorithmic_GBps": 6 * N * nv / ms / 1e6,
                                         "frac_of_hbm_peak": 6 * N * nv / ms / 1e6 / peak}
    c22.close()
    # config 4: decode, 4096 stereo streams x 33 blocks, one run of 8 short blocks per 24 long
    s44 = abi.SetupHolder.load(os.path.join(GOLD, "setup_44k_stereo_q5.npz"))
    c44 = lib.Context(s44, device=device)
    bs = [s44.blocksize(0), s44.blocksize(1)]
    ns, nblk = 4096, 33
    Wrow = np.ones(nblk, np.int32); Wrow[12:20] = 0
    Wseq = np.tile(Wrow, (ns, 1))
    coef_off, pcm_off, coef_len, pcm_len = lib.synthesis_layout(Wseq, bs, s44.channels)
    coef = (torch.rand(coef_len, generator=g, device=dev) * 2 - 1) * 1e-2
    pcm = torch.zeros((ns, s44.channels, pcm_len), device=dev)
    dW = torch.from_numpy(Wseq).to(dev); dco = torch.from_numpy(coef_off).to(dev); dpo = torch.from_numpy(pcm_off).to(dev)
    ms = timed(lambda: c44.synthesis_dev(ns, nblk, dW.data_ptr(), dco.data_ptr(), coef.data_ptr(), dpo.data_ptr(),
                                         pcm.data_ptr(), pcm_len, stream))
    byts = 4 * (coef_len + ns * s44.channels * pcm_len)
    out["decode_4096streams_x33blocks_mixed"] = {"ms": ms, "stereo_blocks_per_s": ns * nblk / ms * 1e3,
                                                  "algorithmic_GBps": byts / ms / 1e6,
                                                  "frac_of_hbm_peak": byts / ms / 1e6 / peak}
    # SURVEY §8 f3: the whole decode DSP in one call (de-couple + floor multiply + IMDCT + overlap-add, int16 out)
    posts = torch.randint(0, 120, (ns * nblk * s44.channels, abi.FLOOR1_STRIDE), generator=g, device=dev, dtype=torch.int32)
    present = torch.ones(ns * nblk * s44.channels, dtype=torch.int32, device=dev)
    pcm16 = torch.zeros((ns, pcm_len, s44.channels), dtype=torch.int16, device=dev)
    res0 = coef.clone()

    def dec():
        coef.copy_(res0)                              # the chain works in place on the residue
        c44.L.vb200_decode_dsp_dev(c44.h, ns, nblk, dW.data_ptr(), dco.data_ptr(), coef.data_ptr(), posts.data_ptr(),
                                   present.data_ptr(), dpo.data_ptr(), pcm16.data_ptr(), 1, pcm_len, stream)
    ms_d = timed(dec) - timed(lambda: coef.copy_(res0))
    out["decode_dsp_4096streams_x33blocks_mixed_s16"] = {"ms": ms_d, "stereo_blocks_per_s": ns * nblk / ms_d * 1e3}
    # SURVEY §8 f2: envelope / block-switch detector, 1000 stereo streams x 800 steps (= 50 long blocks each), int16 PCM
    nse, steps = 1000, 800
    stride_e = 64 * (steps - 1) + 128
    pe = torch.randint(-8000, 8000, (nse, stride_e, s44.channels), generator=g, device=dev, dtype=torch.int16)
    st_e = torch.zeros((nse, abi.ve_state_words(s44.channels)), dtype=torch.int32, device=dev)
    ret_e = torch.zeros((nse, steps), dtype=torch.uint8, device=dev)
    ms_e = timed(lambda: c44.envelope_search_dev(nse, pe.data_ptr(), lib.PCM_S16_INTERLEAVED, stride_e, 0, steps,
                                                 st_e.data_ptr(), ret_e.data_ptr(), stream=stream))
    out["envelope_search_1000streams_x800steps_s16"] = {"ms": ms_e, "long_block_equivalents_per_s": nse * steps / 16 / ms_e * 1e3}
    # bitrate-managed mode (SURVEY §8 a12): all 15 rate curves of every block, device resident
    nbm, Nm, chm = 4000, bs[1], s44.channels
    nm = Nm // 2
    pm = synth_pcm_torch(torch, nbm, chm, Nm, 44100, dev, 77)
    dm = torch.from_numpy(make_desc(nbm).view(np.uint8)).to(dev)
    rows_m = nbm * chm
    NBm = abi.PACKETBLOBS
    posts_m = torch.empty((NBm, rows_m, abi.FLOOR1_STRIDE), dtype=torch.int32, device=dev)
    nz_m = torch.empty((NBm, rows_m), dtype=torch.int32, device=dev)
    iw_m = torch.empty((NBm, rows_m, nm), dtype=torch.int32, device=dev)
    amp_m = torch.empty(nbm, dtype=torch.float32, device=dev)
    iom = abi.EncodeIO()
    iom.pcm, iom.pcm_fmt, iom.desc, iom.independent = pm.data_ptr(), 0, dm.data_ptr(), 1
    iom.posts, iom.nonzero, iom.iwork, iom.ampmax_out = posts_m.data_ptr(), nz_m.data_ptr(), iw_m.data_ptr(), amp_m.data_ptr()
    Lm = lib.load()

    def run_managed():
        rc = Lm.vb200_encode_dsp_managed_dev(c44.h, 1, nbm, 1, C.byref(iom), stream)
        if rc:
            raise RuntimeError("vb200_encode_dsp_managed_dev failed: %d" % rc)
    try:
        ms_m = timed(run_managed, reps=3)
        out["managed_mode_4000_long_stereo_15curves"] = {"ms": ms_m, "stereo_blocks_per_s": nbm / ms_m * 1e3,
                                                         "curves_per_s": nbm * NBm / ms_m * 1e3}
    except Exception as e:                                   # informational leg: never take the headline down
        out["managed_mode_4000_long_stereo_15curves"] = {"error": str(e)}
    del posts_m, nz_m, iw_m, pm
    # Phase A alone through vb200_analysis_phaseA with float host buffers (the round-1 e2e figure, kept for
    # continuity: 16 KB in + 24.6 KB out per block instead of 4 KB + 8.4 KB for the one-call chain)
    nb, N, chn = 20000, bs[1], s44.channels
    n = N // 2
    hp = synth_pcm_torch(torch, nb, chn, N, 44100, dev, 99).cpu().pin_memory()
    outs = [torch.empty((nb, chn, n), dtype=torch.float32).pin_memory() for _ in range(3)]
    hamp = torch.empty(nb, dtype=torch.float32).pin_memory()
    hdesc = make_desc(nb)
    hio = abi.PhaseAIO()
    hio.pcm, hio.desc = hp.data_ptr(), hdesc.ctypes.data
    hio.mdct, hio.logmdct, hio.logmask = (o.data_ptr() for o in outs)
    hio.ampmax_out = hamp.data_ptr()
    L = lib.load()
    for _ in range(2):
        L.vb200_analysis_phaseA(c44.h, 1, nb, C.byref(hio))
    t0 = time.perf_counter()
    for _ in range(3):
        L.vb200_analysis_phaseA(c44.h, 1, nb, C.byref(hio))
    dt = (time.perf_counter() - t0) / 3
    out["phaseA_only_f32_host_buffers_20000_long_stereo"] = {"stereo_blocks_per_s": nb / dt,
                                                             "h2d_bytes": int(hp.numel() * 4), "d2h_bytes": int(3 * outs[0].numel() * 4)}
    c44.close()
    return out


def synth_stream_s16(torch, ns, stride, ch, rate, device, seed):
    """[streams][stride][ch] int16: the same noise+sine mix as synth_pcm_torch, as a contiguous stream"""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    t = torch.arange(stride, device=device, dtype=torch.float32).view(1, stride, 1)
    x = torch.rand((ns, stride, ch), generator=g, device=device, dtype=torch.float32)
    x.mul_(0.5).sub_(0.25)
    f = 440.0 + 110.0 * torch.arange(ch, device=device, dtype=torch.float32).view(1, 1, ch)
    ph = torch.rand((ns, 1, 1), generator=g, device=device) * 6.2831853
    x.add_(0.5 * torch.sin(2 * np.pi * f * t / rate + ph))
    return (x * 32767.0).round_().clamp_(-32768, 32767).to(torch.int16)


def verify_against_oracle(setup, W, pcm_blocks, desc_np, got, streams=None, what=""):
    """bit-exact check of a sample of what was just timed against the CPU oracle (outside any timed region);
    raises on the first difference so that no throughput is ever printed for wrong output"""
    from oracle import pyoracle
    want = pyoracle.Oracle(setup).encode_dsp(W, pcm_blocks, desc_np, streams=streams)
    for k in ("posts", "nonzero", "iwork"):
        w = want[k]
        if k == "iwork" and got[k].dtype == np.int16:
            w = np.clip(w, -32768, 32767).astype(np.int16)
        if not np.array_equal(got[k].reshape(w.shape), w):
            bad = int((got[k].reshape(w.shape) != w).sum())
            raise RuntimeError("%s: CUDA output differs from the oracle in `%s` (%d of %d values)" % (what, k, bad, w.size))
    return int(pcm_blocks.shape[0])


def synth_timelines_s16(torch, lo, hi, stride, ch, rate, device):
    """int16 interleaved timelines [streams][stride][ch] of streams lo..hi-1 of the job: the config-3 noise+sine
    mix with a few level drops followed by bursts per stream, so that the encoder really switches block sizes.
    The tone frequencies, phases and transient positions are functions of the stream id; the noise generator is
    seeded by the slice start, so the shards of different N are statistically identical, not bit-identical
    (the total block count of the job moves by < 0.1 %)."""
    ns = hi - lo
    g = torch.Generator(device=device)
    g.manual_seed(777000 + lo)
    t = torch.arange(stride, device=device, dtype=torch.float32).view(1, stride, 1)
    x = torch.rand((ns, stride, ch), generator=g, device=device, dtype=torch.float32).mul_(0.5).sub_(0.25)
    sid = torch.arange(lo, hi, device=device, dtype=torch.float32).view(ns, 1, 1)
    f = 440.0 + 110.0 * torch.arange(ch, device=device, dtype=torch.float32).view(1, 1, ch) + (sid % 97.0)
    x.add_(0.5 * torch.sin(2 * np.pi * f * t / rate + sid))
    # transients: every ~12000 samples a 300-sample drop to 1 % followed by a 100-sample burst (position by stream id)
    pos = (torch.arange(stride, device=device).view(1, stride) + (torch.arange(lo, hi, device=device).view(ns, 1) * 1237) % 12000) % 12000
    gain = torch.where(pos < 300, 0.01, 1.0).unsqueeze(-1)
    x.mul_(gain)
    burst = ((pos >= 300) & (pos < 400)).unsqueeze(-1)
    x = torch.where(burst, torch.rand((ns, stride, ch), generator=g, device=device) * 1.8 - 0.9, x)
    return (x * 32767.0).round_().clamp_(-32768, 32767).to(torch.int16)


def streams_leg(torch, dist, ctx, abi, lib, setup, dev, world, rank, total_streams, blocks_per_stream, sptr):
    """BASELINE configs[4]: `total_streams` independent streams as ONE job, split over the ranks with
    shard.stream_slice (STRONG scaling: total work fixed), each rank running vb200_encode_streams_dev on its
    slice: envelope search, block planning, both block sizes, ampmax chain across sizes.  Timed on the device
    (CUDA events), max over ranks.  Two streams per rank are verified block by block against the oracle."""
    from vorbis_b200 import shard
    ch, rate = setup.channels, setup.rate
    bs0, bs1 = setup.blocksize(0), setup.blocksize(1)
    lo, hi = shard.stream_slice(total_streams, world, rank)
    ns = hi - lo
    stride = ((blocks_per_stream + 2) * (bs1 // 2) + 3) & ~3
    pcm = synth_timelines_s16(torch, lo, hi, stride, ch, rate, dev)
    max_blocks = stride // (bs0 // 2) + 8
    cap = [ns * (stride // (bs0 // 2) + 8) // 4 + 64, ns * (stride // (bs1 // 2) + 8)]
    plen = torch.full((ns,), stride, dtype=torch.int64, device=dev)
    plan = torch.zeros((ns, max_blocks, 6), dtype=torch.int32, device=dev)
    nblk = torch.zeros(ns, dtype=torch.int32, device=dev)
    io = abi.StreamsIO()
    io.pcm, io.pcm_fmt, io.max_blocks, io.stream_stride = pcm.data_ptr(), lib.PCM_S16_INTERLEAVED, max_blocks, stride
    io.pcm_len, io.eof, io.plan, io.nblocks = plen.data_ptr(), None, plan.data_ptr(), nblk.data_ptr()
    outs = []
    for w, bsz in ((0, bs0), (1, bs1)):
        io.cap[w] = cap[w]
        o = {"posts": torch.empty((cap[w], ch, abi.FLOOR1_STRIDE), dtype=torch.int32, device=dev),
             "nonzero": torch.empty((cap[w], ch), dtype=torch.int32, device=dev),
             "iwork": torch.empty((cap[w], ch, bsz // 2), dtype=torch.int32, device=dev),
             "ampmax_out": torch.empty(cap[w], dtype=torch.float32, device=dev)}
        io.posts[w], io.nonzero[w], io.iwork[w], io.ampmax_out[w] = (o[k].data_ptr() for k in ("posts", "nonzero", "iwork", "ampmax_out"))
        outs.append(o)

    def step():
        rc = ctx.L.vb200_encode_streams_dev(ctx.h, ns, 7, C.byref(io), sptr)
        if rc:
            raise RuntimeError("vb200_encode_streams_dev failed: %d %s" % (rc, ctx.L.vb200_last_error()))
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 3
    e0.record()
    for _ in range(reps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    counts = [int(io.count[0]), int(io.count[1])]
    # verify two streams of this rank's slice block by block (outside the timed region)
    from oracle import pyoracle
    orc = pyoracle.Oracle(setup)
    hplan = plan.cpu().numpy().view(abi.STREAM_BLOCK_DTYPE).reshape(ns, max_blocks)
    hn = nblk.cpu().numpy()
    verified = 0
    for s_ in sorted(set([0, ns - 1])):
        tl = (pcm[s_].cpu().numpy().T.astype(np.float32) / np.float32(32768.0))
        wplan, wouts = orc.encode_stream(tl, stride, 0)
        if hn[s_] != len(wplan):
            raise RuntimeError("streams leg: stream %d has %d blocks, oracle %d" % (lo + s_, hn[s_], len(wplan)))
        for k, wb in enumerate(wplan):
            gb = hplan[s_, k]
            for nm in ("pos", "W", "lW", "nW", "blocktype"):
                if gb[nm] != wb[nm]:
                    raise RuntimeError("streams leg: plan differs from the oracle (stream %d block %d %s)" % (lo + s_, k, nm))
            o = outs[int(gb["W"])]
            sl = int(gb["slot"])
            for nm in ("posts", "nonzero", "iwork"):
                if not np.array_equal(o[nm][sl].cpu().numpy(), wouts[k][nm][0]):
                    raise RuntimeError("streams leg: %s differs from the oracle (stream %d block %d)" % (nm, lo + s_, k))
            verified += 1
    t = torch.tensor([ms, float(counts[0]), float(counts[1]), float(verified)], device=dev, dtype=torch.float64)
    tmax = t.clone()
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    blocks = float(t[1] + t[2])
    return {"streams": total_streams, "blocks": int(blocks), "short_blocks": int(t[1]), "long_blocks": int(t[2]),
            "ms_max_over_ranks": float(tmax[0]), "blocks_per_s": blocks / (float(tmax[0]) * 1e-3),
            "streams_per_rank": ns, "scaling": "strong (fixed job, shard.stream_slice)",
            "verified_blocks_vs_oracle": int(t[3]),
            "call": "vb200_encode_streams_dev: int16 timelines resident, envelope search + block plan + both block sizes + "
                    "ampmax chain across sizes; posts/nonzero/int32 residue out (device)"}


KERNELS = ["k_phaseA_transform", "k_ampmax", "k_phaseA_psy", "k_floor1_fit", "k_floor1_render", "k_cqn"]
DUMP_BLOCKS = 2048


def dump_outputs(torch, path, outs, nb, prefix=""):
    """Write what a step returned, for comparing two builds output for output: every output array on the same
    seeded sample of DUMP_BLOCKS blocks (with the same --blocks, the same blocks in every run), as float64 (exact
    for the int32 and float32 outputs), and the sampled block indices (block_index.npy); about 36 MB for stereo."""
    os.makedirs(path, exist_ok=True)
    sel = np.sort(np.random.default_rng(1234).choice(nb, size=min(DUMP_BLOCKS, nb), replace=False))
    tsel = torch.from_numpy(sel).to(next(iter(outs.values())).device)
    np.save(os.path.join(path, prefix + "block_index.npy"), sel.astype(np.float64))
    for name, t in outs.items():
        np.save(os.path.join(path, prefix + name + ".npy"), t[tsel].cpu().numpy().astype(np.float64))


def run_ours(args):
    import torch
    from vorbis_b200 import abi, lib
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    cpus_info = usable_cpus()                    # before the NUMA binding below narrows this process' affinity
    numa = bind_to_gpu_numa_node(torch, local)
    setup = abi.SetupHolder.load(os.path.join(GOLD, "setup_44k_stereo_q5.npz"))
    ctx = lib.Context(setup, device=local)       # raises if the CUDA library is missing
    N, ch = setup.blocksize(W_LONG), setup.channels
    n = N // 2
    nb = args.blocks
    stream = torch.cuda.current_stream()
    sptr = stream.cuda_stream

    # every rank owns its own shard of independent blocks (weak scaling: nb per GPU, no collective)
    pcm = synth_pcm_torch(torch, nb, ch, N, setup.rate, dev, seed=1000 + rank)
    desc_np = make_desc(nb)
    desc = torch.from_numpy(desc_np.view(np.uint8).reshape(nb, 16).copy()).to(dev)
    posts = torch.empty((nb, ch, abi.FLOOR1_STRIDE), device=dev, dtype=torch.int32)
    nonzero = torch.empty((nb, ch), device=dev, dtype=torch.int32)
    iwork = torch.empty((nb, ch, n), device=dev, dtype=torch.int32)
    amp = torch.empty(nb, device=dev, dtype=torch.float32)
    io = abi.EncodeIO()
    io.pcm, io.pcm_fmt, io.desc, io.independent = pcm.data_ptr(), 0, desc.data_ptr(), 1
    io.posts, io.nonzero, io.iwork, io.ampmax_out = posts.data_ptr(), nonzero.data_ptr(), iwork.data_ptr(), amp.data_ptr()

    def step():
        ctx.encode_dsp_dev(W_LONG, nb, 1, io, blobno=7, stream=sptr)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                  # nvidia-smi needs ~0.1 s before its first line: start it ahead of the warm-up
    for _ in range(args.warmup):
        step()
    barrier()
    if rank == 0:
        sampler.lines.clear()            # keep only samples taken from here on (timed region + same-load tail)
    l0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    launches = ctx.launch_count() - l0
    if args.dump_outputs:                # the last timed step's outputs, before anything else runs the chain again
        dump_outputs(torch, args.dump_outputs, {"posts": posts, "nonzero": nonzero, "iwork": iwork, "ampmax_out": amp},
                     nb, "" if world == 1 else "rank%d_" % rank)
    if rank == 0:
        # the timed region is ~0.1 s: keep the same load running (untimed) until a few clock samples exist
        t_end = time.time() + 2.0
        while sampler.count() < 4 and time.time() < t_end:
            step()
            torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    barrier()
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * nb * args.steps / (ms_max * 1e-3)

    # per-kernel durations (CUDA events on the launching stream, inside the library) for the roofline
    ctx.set_profiling(True)
    kms = np.zeros(6)
    reps = max(3, args.steps)
    for _ in range(reps):
        step()
        torch.cuda.synchronize()
        kms += np.array(ctx.encode_dsp_kernel_ms())
    kms /= reps
    ctx.set_profiling(False)

    # ---- the timed output must be the right output: 256 random blocks of the last step vs the oracle
    vr = np.random.default_rng(4242 + rank)
    sel = np.sort(vr.choice(nb, size=min(256, nb), replace=False))
    tsel = torch.from_numpy(sel).to(dev)
    got = {"posts": posts[tsel].cpu().numpy(), "nonzero": nonzero[tsel].cpu().numpy(), "iwork": iwork[tsel].cpu().numpy()}
    verified = verify_against_oracle(setup, W_LONG, pcm[tsel].cpu().numpy(), desc_np[sel], got, what="resident step")

    # ---- end to end through the host-buffer C-ABI call: int16 stream PCM in (pinned), posts + residue out.
    # Every rank runs it on its own shard at the same time (streams are independent: no collective).
    bps = args.e2e_blocks_per_stream
    ns_e = max(1, min(nb, args.e2e_blocks) // bps)
    nb_e = ns_e * bps
    hop = N // 2
    stride = (bps - 1) * hop + N
    s16 = synth_stream_s16(torch, ns_e, stride, ch, setup.rate, dev, seed=2000 + rank)
    hp = torch.empty((ns_e, stride, ch), dtype=torch.int16).pin_memory()
    hp.copy_(s16)
    del s16
    hdesc = make_desc(nb_e)
    h_posts = torch.empty((nb_e, ch, abi.FLOOR1_STRIDE), dtype=torch.int32).pin_memory()
    h_nz = torch.empty((nb_e, ch), dtype=torch.int32).pin_memory()
    h_iw = torch.empty((nb_e, ch, n), dtype=torch.int16).pin_memory()      # VB200_IWORK_S16: saturated, counted
    h_ovf = torch.empty(nb_e, dtype=torch.int32).pin_memory()
    h_amp = torch.empty(nb_e, dtype=torch.float32).pin_memory()
    hio = abi.EncodeIO()
    hio.pcm, hio.pcm_fmt, hio.hop, hio.stream_stride = hp.data_ptr(), lib.PCM_S16_INTERLEAVED, hop, stride
    hio.desc, hio.independent = hdesc.ctypes.data, 0
    hio.iwork_fmt, hio.overflow = lib.IWORK_S16, h_ovf.data_ptr()
    hio.posts, hio.nonzero, hio.iwork, hio.ampmax_out = h_posts.data_ptr(), h_nz.data_ptr(), h_iw.data_ptr(), h_amp.data_ptr()
    L = lib.load()

    def e2e_step():
        rc = L.vb200_encode_dsp(ctx.h, W_LONG, ns_e, bps, 7, C.byref(hio))
        if rc:
            raise RuntimeError("vb200_encode_dsp failed: %d" % rc)
    for _ in range(2):
        e2e_step()
    barrier()
    l1 = ctx.launch_count()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    e2e_launches = ctx.launch_count() - l1
    td = torch.tensor([dt], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(td, op=dist.ReduceOp.MAX)
    dt_max = float(td.item())
    h2d = int(hp.numel() * 2 + hdesc.nbytes)
    d2h = int((h_posts.numel() + h_nz.numel() + h_amp.numel() + h_ovf.numel()) * 4 + h_iw.numel() * 2)
    if int(h_ovf.sum()) != 0:
        raise RuntimeError("int16 residue overflowed on the bench signal")
    # verify whole streams (the ampmax chain runs along a stream): 6 random streams = 300 blocks
    ssel = np.sort(vr.choice(ns_e, size=min(6, ns_e), replace=False))
    hp_np = hp.numpy()
    blk = np.stack([(hp_np[s_, k * hop:k * hop + N, :].T.astype(np.float32) / np.float32(32768.0))
                    for s_ in ssel for k in range(bps)])
    bsel = np.concatenate([np.arange(s_ * bps, (s_ + 1) * bps) for s_ in ssel])
    got_e = {"posts": h_posts.numpy()[bsel], "nonzero": h_nz.numpy()[bsel], "iwork": h_iw.numpy()[bsel]}
    verified_e2e = verify_against_oracle(setup, W_LONG, blk, hdesc[bsel], got_e, streams=(len(ssel), bps), what="e2e step")
    e2e = {"value": world * nb_e * args.steps / dt_max, "unit": UNIT,
           "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h * world,
           "blocks_per_step": nb_e * world, "gpu_launches": int(e2e_launches), "numa": numa,
           "verified_blocks_vs_oracle": verified_e2e,
           "call": "vb200_encode_dsp: %d streams x %d blocks per GPU, int16 interleaved stream PCM in (hop N/2, "
                   "blocks cut on the device), posts+nonzero+quantised residue (int16, overflow-counted) out; pinned host memory; "
                   "chunks of 8192 blocks (ramped at both ends) over four buffer sets, one copy stream per direction + two compute streams; wall clock, max over ranks" % (ns_e, bps)}

    # ---- BASELINE configs[4]: a fixed job of independent streams with real block switching, split over the ranks
    streams_res = None
    if args.streams > 0:
        import torch.distributed as dist2
        try:
            streams_res = streams_leg(torch, dist2 if world > 1 else None, ctx, abi, lib, setup, dev, world, rank,
                                      args.streams, args.stream_blocks, sptr)
        except Exception as e:
            streams_res = {"error": repr(e)}

    line = None
    if rank == 0:
        peak, peak_src = load_peaks()
        # algorithmic bytes per (block,channel) row (DESIGN.md §4): transform reads 4N, writes mdct 2N + logfft 2N;
        # psy reads mdct 2N + logfft 2N, writes mdct' + logmdct + logmask 6N; floor1_fit reads logmdct + logmask 4N;
        # render writes ilogmask 2N; cqn reads mdct' 2N + ilogmask 2N, writes residue 2N
        alg = [8 * N, 0, 10 * N, 4 * N, 2 * N, 6 * N]
        dom = int(np.argmax(kms))
        achieved = alg[dom] * ch * nb / (kms[dom] * 1e-3) / 1e9
        # DRAM traffic of the dominant kernel from the committed ncu --set full capture (bytes per
        # (block,channel) row, profiles/summary.json), scaled to this launch
        traffic = None
        try:
            summ = json.load(open(os.path.join(ROOT, "profiles", "summary.json")))
            per_row = summ["kernels"][KERNELS[dom]]["dram_bytes_per_row"]
            traffic = per_row * ch * nb
        except Exception:
            pass
        # the dominant kernel is issue bound (DRAM < 10 %): executed warp-instructions per row (ncu, profiles/summary.json)
        # x rows of this launch / (live duration x SMs x SM clock) = IPC, against the 4 issue slots per cycle of an SM
        issue = None
        try:
            ipr = summ["kernels"][KERNELS[dom]]["warp_instructions_per_row"]
            sms = torch.cuda.get_device_properties(local).multi_processor_count
            mhz = (clocks or {}).get("sm_mhz") or (clocks or {}).get("sm_max_mhz") or 1965.0
            ipc = ipr * ch * nb / (kms[dom] * 1e-3 * sms * mhz * 1e6)
            issue = {"warp_instructions_per_row": ipr, "ipc": ipc, "peak_ipc": 4.0, "frac": ipc / 4.0, "sms": sms, "sm_mhz": mhz,
                     "source": "ncu instruction count (profiles/summary.json) x rows / (live CUDA-event duration x SMs x clock)"}
        except Exception:
            pass
        roof = {"bound": "hbm", "kernel": KERNELS[dom], "achieved": achieved, "peak": peak, "unit": "GB/s", "issue": issue,
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "kernel_ms": {k: float(v) for k, v in zip(KERNELS, kms)},
                "kernel_algorithmic_GBps": {k: (float(a * ch * nb / (v * 1e-3) / 1e9) if v > 0 else None)
                                            for k, a, v in zip(KERNELS, alg, kms)},
                "phaseA_only_blocks_per_s": float(nb / (kms[:3].sum() * 1e-3))}

        # ---- CPU baseline on a bounded sample of the same workload (same chain, reference functions)
        cpu, cpu1 = cpu_reference_rates(args.ref_blocks_per_core, 2, 1, cpus_info=cpus_info)

        extra = None
        if not args.no_extra:
            try:
                extra = extra_configs(torch, lib, abi, local, peak)
            except Exception as e:  # the headline line must still be printed
                extra = {"error": repr(e)}
        if streams_res is not None:
            extra = dict(extra or {})
            extra["streams_%d_mixed_blocks" % args.streams] = streams_res

        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(nb, N, ch), "blocks_per_gpu": nb,
                       "l2": "inputs+intermediates+outputs per step (%.1f GB) exceed the 126 MB L2" % (30 * N * ch * nb / 1e9),
                       "sharding": "independent blocks per rank, no collective"},
            "verified_blocks_vs_oracle": verified, "roofline": roof, "cpu_baseline": cpu, "cpu_baseline_1core": cpu1, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            "extra": extra,
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--blocks", type=int, default=100000, help="stereo blocks per GPU per step")
    ap.add_argument("--e2e-blocks", type=int, default=100000, help="stereo blocks per GPU per e2e step (same workload as the resident step)")
    ap.add_argument("--e2e-blocks-per-stream", type=int, default=50)
    ap.add_argument("--no-extra", action="store_true", help="skip the informational configs 2/4")
    ap.add_argument("--streams", type=int, default=10000, help="configs[4]: streams of the fixed mixed-block job (0 = skip)")
    ap.add_argument("--stream-blocks", type=int, default=50, help="long-block lengths per stream of that job")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a fixed sample of the last timed step's outputs "
                    "(posts, nonzero, iwork, ampmax_out) to DIR/<name>.npy")
    ap.add_argument("--ref-blocks-per-core", type=int, default=2048,
                    help="CPU arms: long stereo blocks per pinned process per step (about 0.4 s of work)")
    if len(sys.argv) > 1 and sys.argv[1] == "--cpu-worker":
        return cpu_worker_main(sys.argv[2:])
    args = ap.parse_args()
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
