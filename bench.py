#!/usr/bin/env python3
"""bench.py -- throughput of the B200 log-parsing engine on BASELINE.json's configs.

  python bench.py --gpus N --steps K --warmup W [--config c1|c2|c3|c4|c5]   (N>1: launched by torch.distributed.run)
  python bench.py --impl reference ...           (the reference-side CPU arm: oracle restatement on all host cores)

Default config = c2, BASELINE.json's headline: ProcessorParseRegexNative, nginx access-log regex with 10 capture groups
(docs/cn/plugins/processor/native/processor-parse-regex-native.md:49), 4 Mi lines x 256 B per GPU.  Weak scaling: every
rank parses its own shard, no collective on the data path.  One "step" = one pass of the hot path over the whole batch.

  value      input MB/s (1 MB = 1e6 B of log bytes, separators included) with the batch resident in HBM.  Timing: after
             a warm-up that keeps the device busy for the 1.2 s the clock sampler needs and ends with W >= 3 steps
             back to back between two CUDA events, the timed region holds exactly K steps (--steps; by default sized
             from the step time of those W with a 10 % margin, so that it lasts >= 1 s), split into up to 20 chunks
             of >= 10 ms, each between two CUDA events on the engine's stream.  One more warm-up step is queued right
             ahead of the region, which sits between barrier + synchronize on both sides.
             ms_per_step = MEDIAN over the chunks of chunk time / its steps (min also reported), value = sum of the
             shard bytes / max over ranks of that time.
  e2e        the same metric through the reference-facing C-ABI call of the path with HOST buffers (pinned arena in,
             result tables out), H2D and D2H inside the timed region -- what the engine contributes to a pipeline.
  e2e_plugin (c2) one level up: ProcessorInstance::Process(std::vector<PipelineEventGroup>&) of the B200-backed
             ProcessorParseRegexNative over event groups of <= 512 KB whose arenas are pinned SourceBuffers, with the
             wall time of its phases (gather / engine call / per-event epilogue).  At this boundary the reference's
             event-object model (one heap LogEvent per line, one AddLog per capture) costs more than the parsing
             itself on either arm; cpu_baseline is measured at the same boundary with the same model.
  roofline   achieved = algorithmic bytes of SURVEY.md section 8(d) per step / median device time of one step.

  --dump-outputs DIR writes the result tables of the last timed step (rank 0) as DIR/<name>.npy, see dump_outputs();
  c5 calls the engine once per sub-batch of 1 Mi lines into the same tables, so only its last call's tables are written.
  The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

UNIT = "MB/s"
GROUP_BYTES = 512 * 1024  # LogFileReader.cpp:97: the reader hands the processors groups of at most 512 KB
REGION_S = 1.0  # timed region without --steps: at least this long
CHUNK_MS = 10.0  # timed steps between two CUDA events: at least this long (an event costs ~2 us on a B200)
MAX_CHUNKS = 20
DUMP_BYTES = 64 * 10 ** 6  # --dump-outputs: all files together
DUMP_SEED = 20261017  # --dump-outputs: the row sample of tables larger than DUMP_BYTES


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default: enough for a region of >= %g s, sized from the warm-up's step time; "
                         "the reference arm: 30)" % REGION_S)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=["c1", "c2", "c3", "c4", "c5"])
    ap.add_argument("--lines", type=int, default=0, help="lines (c3: records) per GPU; default: the BASELINE size")
    ap.add_argument("--e2e", default="auto", choices=["auto", "plugin", "abi", "none"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result tables of the last timed step as DIR/<name>.npy (float64; c5: only "
                         "those of the step's last engine call, up to %d lines)" % C5.SUB)
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


# ------------------------------------------------------------------------------------------------ host placement
def pin_to_gpu_numa(local_rank):
    """Binds this process (and therefore its pinned allocations and host threads) to the NUMA node its GPU hangs off."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = getattr(torch.cuda.get_device_properties(local_rank), "pci_domain_id", 0)
        dev = torch.cuda.get_device_properties(local_rank).pci_device_id
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (dom, bus, dev)
        with open(path) as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "cpus": len(allowed)}
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (profiling recipe's clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        self.t_start = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=timestamp," + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def mark_region(self):
        self.t_start = time.time()

    def stop(self):
        t_end = time.time()
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons, all_sm = [], [], set(), []
        import datetime
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 10:
                continue
            try:
                s, m = float(c[2]), float(c[3])
            except ValueError:
                continue
            try:
                ts = datetime.datetime.strptime(c[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except ValueError:
                ts = None
            all_sm.append(s)
            if ts is not None and self.t_start is not None and not (self.t_start - 0.05 <= ts <= t_end + 0.05):
                continue
            sm.append(s)
            mx.append(m)
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[6:10]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                   "samples": len(sm), "samples_total": len(all_sm)}
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        return out


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def pinned_array(pins, src, dtype):
    """numpy view of a pinned allocation (lc_host_alloc); src = an array to copy in, or a byte count."""
    import loongcollector_b200 as lc
    L = lc.lib()
    nbytes = int(src.nbytes) if isinstance(src, np.ndarray) else int(src)
    p = L.lc_host_alloc(max(nbytes, 16))
    if not p:
        raise RuntimeError("lc_host_alloc failed")
    pins.append(p)
    arr = np.ctypeslib.as_array(ctypes.cast(p, ctypes.POINTER(ctypes.c_uint8)), shape=(max(nbytes, 1),))[:nbytes].view(dtype)
    if isinstance(src, np.ndarray):
        arr[:] = np.ascontiguousarray(src).view(dtype).reshape(-1)
    return arr


def profile_traffic(config):
    """dram bytes per launch of the config's dominant kernel from the committed ncu summary (stamped with the git
    hash of the kernel source it was captured on; None when the source has changed since)."""
    p = os.path.join(ROOT, "profiles", "summary.json")
    try:
        with open(p) as f:
            ent = json.load(f).get(config)
        if not ent:
            return None, None
        import hashlib
        h = hashlib.sha256()
        for name in ent.get("sources", []):
            with open(os.path.join(ROOT, name), "rb") as f:
                h.update(f.read())
        stale = ent.get("sources_sha16") != h.hexdigest()[:16]
        return ent.get("dram_bytes_per_step"), {"kernel": ent.get("kernel"), "capture": ent.get("capture"),
                                                "stale": stale}
    except Exception:
        return None, None


def job_throughput(bytes_local, ms_local, world, device="cpu"):
    """Whole-job MB/s under weak scaling: every rank parses its own shard, the job finishes when the slowest
    rank does -> sum of the shard bytes / max over ranks of the step time.  Uses the default process group
    (NCCL on GPUs, gloo in the CPU tests); no data-path collective, just this 2-number reduction."""
    import torch
    t = torch.tensor([float(ms_local)], dtype=torch.float64, device=device)
    b = torch.tensor([float(bytes_local)], dtype=torch.float64, device=device)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(b, op=dist.ReduceOp.SUM)
    ms = float(t.item())
    return float(b.item()) / (ms * 1e-3) / 1e6, ms


def gather_rank_stats(vals, world, device="cpu"):
    """[[v0, v1, ...] per rank] of a short float list (per-rank min / median / max of the step time)."""
    import torch
    t = torch.tensor([float(v) for v in vals], dtype=torch.float64, device=device)
    if world > 1:
        import torch.distributed as dist
        out = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(out, t)
        return [[float(x) for x in o.tolist()] for o in out]
    return [[float(x) for x in t.tolist()]]


def shard_seed(rank):
    """Shards are independent event groups: rank r generates (and owns) its own lines."""
    return 20260922 + rank


def make_workload(n_lines, seed):
    from loongcollector_b200 import synth
    return synth.nginx_lines(n_lines, seed=seed, line_bytes=256)


def _vp(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def dump_outputs(cfg, out_dir):
    """Writes the tables the timed path returned in its last step (cfg.outputs(): name -> array) as out_dir/<name>.npy
    in float64, which holds every u8 / u32 value exactly.  If the tables with the most rows would take the files past
    DUMP_BYTES, each of them keeps the same DUMP_SEED-seeded sample of rows, whose row numbers go to rows.npy."""
    outs = {k: np.asarray(a) for k, a in cfg.outputs().items()}
    n = max(a.shape[0] for a in outs.values())
    per_row = sum(a.size // n for a in outs.values() if a.shape[0] == n)
    fixed = sum(a.size for a in outs.values() if a.shape[0] != n)
    m = min(n, (DUMP_BYTES // 8 - 1024 - fixed) // (per_row + 1))  # 1024 values of room for the .npy headers
    if m < n:
        rows = np.sort(np.random.default_rng(DUMP_SEED).choice(n, m, replace=False))
        outs = {k: a[rows] if a.shape[0] == n else a for k, a in outs.items()}
        outs["rows"] = rows
    os.makedirs(out_dir, exist_ok=True)
    for k, a in outs.items():
        np.save(os.path.join(out_dir, k + ".npy"), a.astype(np.float64))


# ------------------------------------------------------------------------------------------------ CPU arms (oracle)
def cpu_threads_run(work, threads):
    t0 = time.perf_counter()
    if threads == 1:
        work(0)
    else:
        ts = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
    return time.perf_counter() - t0


def cpu_regex_parse(pattern, nkeys, buf, off, ln, threads):
    """Flat CPU path (oracle restatement, PCRE2 interpretive, one matcher per thread -- mirrors mReg[threadNo],
    ProcessorParseRegexNative.cpp:64-67).  Returns (seconds, status, cap_off, cap_len)."""
    from oracle import oracle as orc
    rx = orc.Regex(pattern)
    L = orc.lib()
    n, G = off.size, rx.ngroups
    status = np.zeros(n, np.uint8)
    co = np.zeros((n, G), np.uint32)
    cl = np.zeros((n, G), np.uint32)
    bounds = np.linspace(0, n, threads + 1).astype(np.int64)
    matchers = [rx.new_matcher() for _ in range(threads)]

    def work(t):
        a, b = int(bounds[t]), int(bounds[t + 1])
        if b > a:
            L.orc_regex_parse_batch(matchers[t], _vp(buf), _vp(off[a:b]), _vp(ln[a:b]), b - a, nkeys,
                                    _vp(status[a:b]), _vp(co[a:b]), _vp(cl[a:b]))

    dt = cpu_threads_run(work, threads)
    for m in matchers:
        L.orc_matcher_free(m)
    return dt, status, co, cl


_PLUGIN_LIB = None


def oracle_plugin_lib():
    global _PLUGIN_LIB
    if _PLUGIN_LIB is None:
        so = os.path.join(ROOT, "oracle", "liblc_oracle_plugin.so")
        if not os.path.exists(so):
            subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "-s"])
        L = ctypes.CDLL(so)
        L.orc_bench_plugin.argtypes = [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                       ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                                       ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p)]
        L.orc_string_free.argtypes = [ctypes.c_void_p]
        _PLUGIN_LIB = L
    return _PLUGIN_LIB


STAT_NAMES = ("groups", "in_events", "out_events", "live_contents", "checksum", "arena_bytes", "ctr_in_events",
              "ctr_out_events", "ctr_in_bytes", "ctr_out_bytes", "ctr_process_ns", "ctr_process_ms", "gather_ns",
              "engine_ns", "epilogue_ns", "spare")


def regex_plugin_config():
    from loongcollector_b200 import synth
    return json.dumps({"SourceKey": "content", "Regex": synth.NGINX_PATTERN, "Keys": synth.NGINX_KEYS}).encode()


def cpu_plugin_regex(buf, off, ln, threads, reps):
    """CPU reference arm at the plugin boundary (oracle/ref_plugin.cpp): Process(group) per <= 512 KB group on `threads`
    ProcessorRunner-like threads, PCRE2 regex_match + AddLog per capture on the same event model as the GPU arm."""
    L = oracle_plugin_lib()
    secs = np.zeros(reps, np.float64)
    stats = np.zeros(12, np.uint64)
    err = ctypes.c_void_p()
    rc = L.orc_bench_plugin(regex_plugin_config(), _vp(buf), _vp(off), _vp(ln), off.size, GROUP_BYTES, threads, reps,
                            _vp(secs), _vp(stats), ctypes.byref(err))
    if rc != 0:
        raise RuntimeError(ctypes.string_at(err.value).decode() if err.value else "orc_bench_plugin failed")
    return secs, dict(zip(STAT_NAMES, (int(x) for x in stats)))


def expected_plugin_stats(buf, st, co, cl, keys):
    """What the plugin run must leave behind, derived from the flat result tables: matching lines keep the 10 parsed
    fields (source key deleted), the others are erased (no Keeping* flag)."""
    ok = st == 0
    n_ok = int(ok.sum())
    klen = np.array([len(k) for k in keys], np.uint64)
    c_len = cl[ok].astype(np.uint64)
    first = buf[np.minimum(co[ok].astype(np.int64), buf.size - 1)].astype(np.uint64) * (c_len > 0)
    checksum = int((klen[None, :] * np.uint64(131) + c_len * np.uint64(31) + first).sum(dtype=np.uint64))
    return {"out_events": n_ok, "live_contents": n_ok * len(keys), "checksum": checksum}


# ------------------------------------------------------------------------------------------------ config definitions
class Config:
    """One BASELINE.json config: data, the device-resident step, algorithmic bytes, the host-buffer step, CPU legs."""
    name = ""
    metric = "regex_parsed_log_MBps"
    dominant = ""

    def __init__(self, args, rank, world, eng, dev):
        self.args, self.rank, self.world, self.eng, self.dev = args, rank, world, eng, dev

    def dput(self, a, dtype=None):
        import torch
        t = torch.from_numpy(np.ascontiguousarray(a))
        return t.to(self.dev, non_blocking=False)


class C2(Config):
    name = "c2"
    dominant = "regex_tdfa_staged_kernel"

    def workload(self):
        return "C2: ProcessorParseRegexNative nginx 10-group regex, %d lines x 256 B per GPU" % self.n

    def setup_host(self):
        self.n = self.args.lines or 4 * 1024 * 1024
        self.buf, self.off, self.ln = make_workload(self.n, shard_seed(self.rank))
        self.in_bytes = int(self.buf.size)
        self.units = self.n

    def setup(self):
        import torch
        import loongcollector_b200 as lc
        from loongcollector_b200 import synth
        self.setup_host()
        self.rx = lc.Regex(synth.NGINX_PATTERN)
        self.G, self.nkeys = self.rx.ngroups, len(synth.NGINX_KEYS)
        self.alg_bytes = int(self.ln.astype(np.int64).sum()) + self.n * (8 + 8 * self.G + 1)
        n, G = self.n, self.G
        self.d_buf = torch.empty(self.buf.size + 16, dtype=torch.uint8, device=self.dev)
        self.d_buf[:self.buf.size].copy_(torch.from_numpy(self.buf))
        self.d_off = self.dput(self.off.view(np.int32))
        self.d_len = self.dput(self.ln.view(np.int32))
        self.d_status = torch.empty(n, dtype=torch.uint8, device=self.dev)
        self.d_co = torch.empty(n * G, dtype=torch.int32, device=self.dev)
        self.d_cl = torch.empty(n * G, dtype=torch.int32, device=self.dev)
        self.extra = {"regex_tables": self.rx.info}

    def step(self):
        self.eng.regex_parse_dev(self.rx, self.d_buf.data_ptr(), self.in_bytes, self.d_off.data_ptr(),
                                 self.d_len.data_ptr(), self.n, self.nkeys, self.d_status.data_ptr(),
                                 self.d_co.data_ptr(), self.d_cl.data_ptr())

    def results(self):
        n, G = self.n, self.G
        return (self.d_status.cpu().numpy(), self.d_co.cpu().numpy().view(np.uint32).reshape(n, G),
                self.d_cl.cpu().numpy().view(np.uint32).reshape(n, G))

    def outputs(self):
        return dict(zip(("status", "cap_off", "cap_len"), self.results()))

    def check(self):
        """every row of a bounded prefix against the CPU oracle (rank 0)"""
        from loongcollector_b200 import synth
        st, co, cl = self.results()
        ns = min(self.n, 131072)
        dt, est, eco, ecl = cpu_regex_parse(synth.NGINX_PATTERN, self.nkeys, self.buf, self.off[:ns], self.ln[:ns], 1)
        assert np.array_equal(est, st[:ns]) and np.array_equal(eco, co[:ns]) and np.array_equal(ecl, cl[:ns]), \
            "GPU result differs from the CPU oracle on the sample"
        return {"matched_lines_fraction": float((st == 0).mean()),
                "cpu_1thread": {"value": ns * 256 / dt / 1e6, "unit": UNIT, "cores": 1, "kind": "port",
                                "sample": "%d lines x 256 B, flat oracle (PCRE2 10.42 interpretive), 1 thread" % ns}}

    # ---- end to end
    def e2e_abi_setup(self):
        import loongcollector_b200 as lc
        L = lc.lib()
        self._pins = []

        def pinned(src, dtype):
            nbytes = int(src.nbytes) if isinstance(src, np.ndarray) else int(src)
            p = L.lc_host_alloc(max(nbytes, 16))
            if not p:
                raise RuntimeError("lc_host_alloc failed")
            self._pins.append(p)
            arr = np.ctypeslib.as_array(ctypes.cast(p, ctypes.POINTER(ctypes.c_uint8)), shape=(nbytes,)).view(dtype)
            if isinstance(src, np.ndarray):
                arr[:] = src.view(dtype).reshape(-1)
            return arr

        n, G = self.n, self.G
        self.h_buf = pinned(self.buf, np.uint8)
        self.h_off = pinned(self.off, np.uint32)
        self.h_len = pinned(self.ln, np.uint32)
        self.h_status = pinned(n, np.uint8)
        self.h_co = pinned(n * G * 4, np.uint32)
        self.h_cl = pinned(n * G * 4, np.uint32)
        self.e2e_h2d = int(self.in_bytes + 8 * n)
        self.e2e_d2h = int(n * (1 + 8 * G))

    def e2e_abi_step(self):
        import loongcollector_b200 as lc
        L = lc.lib()
        rc = L.lc_regex_parse(self.eng._h, self.rx._h, _vp(self.h_buf), self.in_bytes, _vp(self.h_off),
                              _vp(self.h_len), self.n, self.nkeys, _vp(self.h_status), _vp(self.h_co), _vp(self.h_cl))
        if rc != 0:
            raise RuntimeError(L.lc_last_error().decode())

    def e2e_abi_check(self, st):
        assert np.array_equal(self.h_status, st), "host-API result differs from device-API result"

    def e2e_abi_free(self):
        import loongcollector_b200 as lc
        for p in self._pins:
            lc.lib().lc_host_free(p)

    def e2e_plugin(self, reps, mode=1):
        """ProcessorInstance::Process through the host layer (pinned SourceBuffer arenas, <= 512 KB groups)."""
        import loongcollector_b200 as lc
        L = lc.lib()
        L.lc_host_use_pinned_arenas.argtypes = [ctypes.c_int]
        L.lc_host_bench_plugin.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_void_p, ctypes.c_void_p,
                                           ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int,
                                           ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                           ctypes.POINTER(ctypes.c_void_p)]
        L.lc_host_string_free.argtypes = [ctypes.c_void_p]
        L.lc_host_use_pinned_arenas(1)
        os.environ.setdefault("LC_B200_DEVICE", str(self.dev.index))
        secs = np.zeros(reps, np.float64)
        stats = np.zeros(16, np.uint64)
        err = ctypes.c_void_p()
        rc = L.lc_host_bench_plugin(b"processor_parse_regex_native", regex_plugin_config(), _vp(self.buf),
                                    _vp(self.off), _vp(self.ln), self.n, GROUP_BYTES, mode, reps, _vp(secs),
                                    _vp(stats), ctypes.byref(err))
        if rc != 0:
            raise RuntimeError(ctypes.string_at(err.value).decode() if err.value else "lc_host_bench_plugin failed")
        return secs, dict(zip(STAT_NAMES, (int(x) for x in stats)))

    # ---- CPU legs
    def cpu_baseline(self):
        """all host cores on a bounded sample, at both boundaries: the flat path (what `e2e` is compared with) and
        the plugin call (what `e2e_plugin` is compared with)"""
        from loongcollector_b200 import synth
        cores = len(os.sched_getaffinity(0)) or 1
        ns = min(self.n, 1 << 20)
        ts = [cpu_regex_parse(synth.NGINX_PATTERN, self.nkeys, self.buf, self.off[:ns], self.ln[:ns], cores)[0]
              for _ in range(3)]
        secs, stats = cpu_plugin_regex(self.buf, self.off[:ns], self.ln[:ns], cores, 3)
        dt = float(np.median(secs))
        return {"value": ns * 256 / float(np.median(ts)) / 1e6, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": "%d lines x 256 B, flat oracle (PCRE2 10.42 interpretive regex_match, one matcher per "
                          "thread) on %d threads; median of 3" % (ns, cores),
                "plugin": {"value": ns * 256 / dt / 1e6, "unit": UNIT,
                           "sample": "the same lines in %d groups of <= 512 KB, Process(group) on %d threads: "
                                     "regex_match + AddLog per capture on the event model "
                                     "(oracle/ref_plugin.cpp); median of 3" % (stats["groups"], cores)}}


class C1(Config):
    name = "c1"
    metric = "split_log_MBps"
    dominant = "split_mask_kernel + split_scan_kernel + split_emit_kernel"

    def workload(self):
        return "C1: ProcessorSplitLogStringNative newline split, %d lines x 512 B per GPU" % self.n

    def setup_host(self):
        from loongcollector_b200 import synth
        self.n = self.args.lines or (1 << 20)
        self.buf, self.off, self.ln = synth.newline_lines(self.n, 512, seed=shard_seed(self.rank))
        self.in_bytes = int(self.buf.size)
        self.units = self.n

    def setup(self):
        import torch
        self.setup_host()
        self.alg_bytes = self.in_bytes + 8 * self.n
        self.d_buf = self.dput(self.buf)
        self.d_off = torch.empty(self.n + 16, dtype=torch.int32, device=self.dev)
        self.d_len = torch.empty(self.n + 16, dtype=torch.int32, device=self.dev)
        self.extra = {}

    def step(self):
        self.got = self.eng.split_lines_dev(self.d_buf.data_ptr(), self.in_bytes, 10, self.d_off.data_ptr(),
                                            self.d_len.data_ptr(), self.n + 16)

    def outputs(self):
        return {"line_count": np.array([self.got]), "line_off": self.d_off[:self.got].cpu().numpy().view(np.uint32),
                "line_len": self.d_len[:self.got].cpu().numpy().view(np.uint32)}

    def check(self):
        from oracle import oracle as orc
        assert self.got == self.n
        assert np.array_equal(self.d_off[:self.n].cpu().numpy().view(np.uint32), self.off)
        assert np.array_equal(self.d_len[:self.n].cpu().numpy().view(np.uint32), self.ln)
        ns = min(self.n, 1 << 18)
        t0 = time.perf_counter()
        o, l = orc.split_lines(self.buf[:ns * 512])
        dt = time.perf_counter() - t0
        assert np.array_equal(o, self.off[:ns]) and np.array_equal(l, self.ln[:ns])
        return {"cpu_1thread": {"value": ns * 512 / dt / 1e6, "unit": UNIT, "cores": 1, "kind": "port",
                                "sample": "%d lines x 512 B, flat oracle split, 1 thread" % ns}}

    def e2e_abi_setup(self):
        import loongcollector_b200 as lc
        L = lc.lib()
        self._p = [L.lc_host_alloc(self.in_bytes + 16), L.lc_host_alloc((self.n + 16) * 4),
                   L.lc_host_alloc((self.n + 16) * 4)]
        self.h_buf = np.ctypeslib.as_array(ctypes.cast(self._p[0], ctypes.POINTER(ctypes.c_uint8)),
                                           shape=(self.in_bytes,))
        self.h_buf[:] = self.buf
        self.e2e_h2d = self.in_bytes
        self.e2e_d2h = 8 * self.n

    def e2e_abi_step(self):
        import loongcollector_b200 as lc
        L = lc.lib()
        n = ctypes.c_uint64(0)
        rc = L.lc_split_lines(self.eng._h, self._p[0], self.in_bytes, 10, self._p[1], self._p[2], self.n + 16,
                              ctypes.byref(n))
        if rc != 0 or n.value != self.n:
            raise RuntimeError(L.lc_last_error().decode())

    def e2e_abi_check(self, st):
        pass

    def e2e_abi_free(self):
        import loongcollector_b200 as lc
        for p in self._p:
            lc.lib().lc_host_free(p)

    def cpu_baseline(self):
        from oracle import oracle as orc
        cores = len(os.sched_getaffinity(0)) or 1
        ns = min(self.n, 1 << 20)
        per = ns // cores
        if per == 0:
            cores, per = 1, ns
        L = orc.lib()
        offs = [np.zeros(per + 8, np.uint32) for _ in range(cores)]
        lens = [np.zeros(per + 8, np.uint32) for _ in range(cores)]

        def work(t):
            for _ in range(8):
                L.orc_split_lines(_vp(self.buf[t * per * 512:]), per * 512, 10, _vp(offs[t]), _vp(lens[t]), per + 8)

        dt = cpu_threads_run(work, cores)
        return {"value": 8 * cores * per * 512 / dt / 1e6, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": "%d lines x 512 B per thread x 8 passes, flat oracle split on %d threads" % (per, cores)}


class C3(Config):
    name = "c3"
    metric = "multiline_split_log_MBps"
    dominant = "split_mask_kernel + split_scan_kernel + split_emit_kernel + ml_pass_kernel<1..3> + ml_tile_scan_kernel"

    def workload(self):
        return "C3: ProcessorSplitMultilineLogStringNative Java stack traces, start pattern, %d records (%.0f B avg, " \
               "%d lines) per GPU" % (self.nrec, self.in_bytes / self.nrec, self.nlines)

    def setup_host(self):
        from loongcollector_b200 import synth
        self.nrec = self.args.lines or (1 << 20)
        self.buf, self.nlines, _ = synth.java_stack_records(self.nrec, seed=shard_seed(self.rank))
        self.in_bytes = int(self.buf.size)
        self.units = self.nlines

    def setup(self):
        import torch
        import loongcollector_b200 as lc
        from loongcollector_b200 import synth
        self.setup_host()
        self.alg_bytes = self.in_bytes + 8 * self.nrec + self.nlines
        self.start = lc.Regex(synth.JAVA_START_PATTERN)
        self.d_buf = self.dput(self.buf)
        self.cap = self.nrec + 1024
        self.o = torch.empty(self.cap, dtype=torch.int32, device=self.dev)
        self.l = torch.empty(self.cap, dtype=torch.int32, device=self.dev)
        self.f = torch.empty(self.cap, dtype=torch.uint8, device=self.dev)
        self.extra = {}

    def step(self):
        self.got, self.ctr = self.eng.multiline_split_dev(self.d_buf.data_ptr(), self.in_bytes, self.start, None, None,
                                                          False, self.o.data_ptr(), self.l.data_ptr(),
                                                          self.f.data_ptr(), self.cap)

    def outputs(self):
        return {"record_count": np.array([self.got]), "counters": np.array([int(x) for x in self.ctr]),
                "record_off": self.o[:self.got].cpu().numpy().view(np.uint32),
                "record_len": self.l[:self.got].cpu().numpy().view(np.uint32),
                "record_flags": self.f[:self.got].cpu().numpy()}

    def check(self):
        from loongcollector_b200 import synth
        from oracle import oracle as orc
        assert self.got == self.nrec and [int(x) for x in self.ctr] == [self.nrec, self.nlines, 0]
        ns = min(self.in_bytes, 64 << 20)
        cut = int(np.nonzero(self.buf[:ns] == 10)[0][-1]) + 1
        t0 = time.perf_counter()
        eo, el, ef, ectr = orc.multiline_split(self.buf[:cut], orc.Regex(synth.JAVA_START_PATTERN), None, None, False)
        dt = time.perf_counter() - t0
        g_off = self.o[:len(eo) - 1].cpu().numpy().view(np.uint32)
        g_len = self.l[:len(eo) - 1].cpu().numpy().view(np.uint32)
        assert np.array_equal(g_off, eo[:-1]) and np.array_equal(g_len, el[:-1])
        return {"cpu_1thread": {"value": cut / dt / 1e6, "unit": UNIT, "cores": 1, "kind": "port",
                                "sample": "%d bytes, flat oracle multiline split (PCRE2 probes), 1 thread" % cut}}

    def e2e_abi_setup(self):
        import loongcollector_b200 as lc
        L = lc.lib()
        self._p = [L.lc_host_alloc(self.in_bytes + 16), L.lc_host_alloc(self.cap * 4), L.lc_host_alloc(self.cap * 4),
                   L.lc_host_alloc(self.cap)]
        h = np.ctypeslib.as_array(ctypes.cast(self._p[0], ctypes.POINTER(ctypes.c_uint8)), shape=(self.in_bytes,))
        h[:] = self.buf
        self.e2e_h2d = self.in_bytes
        self.e2e_d2h = 9 * self.nrec

    def e2e_abi_step(self):
        import loongcollector_b200 as lc
        L = lc.lib()
        n = ctypes.c_uint64(0)
        ctr = np.zeros(3, np.uint64)
        rc = L.lc_multiline_split(self.eng._h, self._p[0], self.in_bytes, self.start._h, None, None, 0, self._p[1],
                                  self._p[2], self._p[3], self.cap, ctypes.byref(n), _vp(ctr))
        if rc != 0 or n.value != self.nrec:
            raise RuntimeError(L.lc_last_error().decode())

    def e2e_abi_check(self, st):
        pass

    def e2e_abi_free(self):
        import loongcollector_b200 as lc
        for p in self._p:
            lc.lib().lc_host_free(p)

    def cpu_baseline(self):
        from loongcollector_b200 import synth
        from oracle import oracle as orc
        cores = len(os.sched_getaffinity(0)) or 1
        per = min(self.in_bytes // cores, 8 << 20)
        cuts = []
        for t in range(cores):
            a = t * per
            seg = self.buf[a:a + per]
            nl = np.nonzero(seg == 10)[0]
            cuts.append((a, int(nl[-1]) + 1 if nl.size else per))
        rxs = [orc.Regex(synth.JAVA_START_PATTERN) for _ in range(cores)]

        def work(t):
            a, ln = cuts[t]
            orc.multiline_split(self.buf[a:a + ln], rxs[t], None, None, False)

        dt = cpu_threads_run(work, cores)
        tot = sum(c[1] for c in cuts)
        return {"value": tot / dt / 1e6, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": "%d bytes per thread on %d threads, flat oracle multiline split (PCRE2 probes)" % (per, cores)}


class C4(Config):
    name = "c4"
    metric = "delimiter_regex_chain_log_MBps"
    dominant = "delim_tiled_kernel + regex_tdfa_staged_kernel"
    MF = 11

    def workload(self):
        return "C4: ProcessorParseDelimiterNative -> ProcessorParseRegexNative (column 3) chain, %d CSV lines " \
               "(%.0f B avg) per GPU" % (self.n, self.in_bytes / self.n)

    def setup_host(self):
        from loongcollector_b200 import synth
        self.n = self.args.lines or (8 << 20)
        self.buf, self.off, self.ln = synth.csv_lines(self.n, seed=shard_seed(self.rank))
        self.in_bytes = int(self.buf.size)
        self.units = self.n
        self.G = 2  # CSV_URL_PATTERN has two groups

    def setup(self):
        import torch
        import loongcollector_b200 as lc
        from loongcollector_b200 import synth
        self.setup_host()
        n, MF = self.n, self.MF
        self.rx = lc.Regex(synth.CSV_URL_PATTERN)
        assert self.rx.ngroups == self.G
        self.d_buf = self.dput(self.buf)
        self.d_off = self.dput(self.off.view(np.int32))
        self.d_len = self.dput(self.ln.view(np.int32))
        self.st = torch.empty(n, dtype=torch.uint8, device=self.dev)
        self.nf = torch.empty(n, dtype=torch.int32, device=self.dev)
        self.fo = torch.empty(n * MF, dtype=torch.int32, device=self.dev)
        self.fl = torch.empty(n * MF, dtype=torch.int32, device=self.dev)
        self.fd = torch.empty(n * MF, dtype=torch.int32, device=self.dev)
        self.to = torch.empty(n, dtype=torch.int32, device=self.dev)
        self.tl = torch.empty(n, dtype=torch.int32, device=self.dev)
        self.rs = torch.empty(n, dtype=torch.uint8, device=self.dev)
        self.rco = torch.empty(n * self.G, dtype=torch.int32, device=self.dev)
        self.rcl = torch.empty(n * self.G, dtype=torch.int32, device=self.dev)
        self.extra = {}
        self.alg_bytes = None  # needs the column-3 byte count: filled by check()

    def step(self):
        n, MF = self.n, self.MF
        # the delimiter stage also leaves column 3 as a dense (off, len) table: the regex stage's event table
        self.eng.delim_parse_dev(self.d_buf.data_ptr(), self.in_bytes, self.d_off.data_ptr(), self.d_len.data_ptr(), n,
                                 b",", ord('"'), 10, True, True, MF, self.st.data_ptr(), self.nf.data_ptr(),
                                 self.fo.data_ptr(), self.fl.data_ptr(), self.fd.data_ptr(), 3, self.to.data_ptr(),
                                 self.tl.data_ptr())
        self.eng.regex_parse_dev(self.rx, self.d_buf.data_ptr(), self.in_bytes, self.to.data_ptr(), self.tl.data_ptr(),
                                 n, self.G, self.rs.data_ptr(), self.rco.data_ptr(), self.rcl.data_ptr())

    def outputs(self):
        """the tables lc_delim_regex_chain returns"""
        n, MF, G = self.n, self.MF, self.G

        def u32(t, w):
            return t.view(n, w).cpu().numpy().view(np.uint32)
        return {"status": self.st.cpu().numpy(), "nfields": self.nf.cpu().numpy().view(np.uint32),
                "field_off": u32(self.fo, MF), "field_len": u32(self.fl, MF), "field_dq": u32(self.fd, MF),
                "re_status": self.rs.cpu().numpy(), "cap_off": u32(self.rco, G), "cap_len": u32(self.rcl, G)}

    def finish_setup(self):
        n, MF = self.n, self.MF
        col3 = int(self.fl.view(n, MF)[:, 3].sum(dtype=__import__("torch").int64).item())
        nfields = int(self.nf.sum(dtype=__import__("torch").int64).item())
        # SURVEY 8(d): delimiter B_in + N (8 + 8 F + 1) with F = the columns actually parsed, then the regex stage over
        # column 3: its bytes + N (8 + 8 G + 1)
        self.alg_bytes = self.in_bytes + n * 9 + 8 * nfields + col3 + n * (8 + 8 * self.G + 1)

    def check(self):
        from loongcollector_b200 import synth
        from oracle import oracle as orc
        n, MF, G = self.n, self.MF, self.G
        ns = min(n, 1 << 17)
        t0 = time.perf_counter()
        est, enf, efo, efl, efd = orc.delim_parse_batch(self.buf, self.off[:ns], self.ln[:ns], b",", ord('"'), 10,
                                                        True, True, MF)
        rst, rco_e, rcl_e = orc.regex_parse_batch(orc.Regex(synth.CSV_URL_PATTERN), self.buf, efo[:, 3].copy(),
                                                  efl[:, 3].copy(), G)
        dt = time.perf_counter() - t0
        assert np.array_equal(self.st[:ns].cpu().numpy(), est)
        assert np.array_equal(self.fo.view(n, MF)[:ns].cpu().numpy().view(np.uint32), efo)
        assert np.array_equal(self.fl.view(n, MF)[:ns].cpu().numpy().view(np.uint32), efl)
        assert np.array_equal(self.fd.view(n, MF)[:ns].cpu().numpy().view(np.uint32), efd)
        assert np.array_equal(self.rs[:ns].cpu().numpy(), rst)
        assert np.array_equal(self.rco.view(n, G)[:ns].cpu().numpy().view(np.uint32), rco_e)
        assert np.array_equal(self.rcl.view(n, G)[:ns].cpu().numpy().view(np.uint32), rcl_e)
        by = int(self.ln[:ns].astype(np.int64).sum() + ns)
        return {"cpu_1thread": {"value": by / dt / 1e6, "unit": UNIT, "cores": 1, "kind": "port",
                                "sample": "%d CSV lines, flat oracle delimiter FSM + PCRE2 on column 3, 1 thread" % ns}}

    def e2e_abi_setup(self):
        # lc_delim_regex_chain: pinned host buffers in, both stages' tables out; inside the library the arena goes up once,
        # in chunks of whole lines through three streams (upload / the two stages / tables back)
        n, MF, G = self.n, self.MF, self.G
        self._pins = []
        self.hin = {k: pinned_array(self._pins, a, a.dtype)
                    for k, a in (("buf", self.buf), ("off", self.off), ("ln", self.ln))}
        self.h = {k: pinned_array(self._pins, s_ * np.dtype(d).itemsize, d)
                  for k, s_, d in (("st", n, np.uint8), ("nf", n, np.uint32), ("fo", n * MF, np.uint32),
                                   ("fl", n * MF, np.uint32), ("fd", n * MF, np.uint32), ("rs", n, np.uint8),
                                   ("rco", n * G, np.uint32), ("rcl", n * G, np.uint32))}
        self.e2e_h2d = int(self.in_bytes + 8 * n)
        self.e2e_d2h = int(n * (5 + 12 * MF) + n * (1 + 8 * G))

    def e2e_abi_step(self):
        import loongcollector_b200 as lc
        L = lc.lib()
        h, n, MF = self.h, self.n, self.MF
        sep = np.frombuffer(b",", np.uint8)
        rc = L.lc_delim_regex_chain(self.eng._h, _vp(self.hin["buf"]), self.in_bytes, _vp(self.hin["off"]),
                                    _vp(self.hin["ln"]), n, _vp(sep), 1, ord('"'), 10, 1, 1, MF, _vp(h["st"]),
                                    _vp(h["nf"]), _vp(h["fo"]), _vp(h["fl"]), _vp(h["fd"]), 3, self.rx._h, self.G,
                                    _vp(h["rs"]), _vp(h["rco"]), _vp(h["rcl"]))
        if rc != 0:
            raise RuntimeError(L.lc_last_error().decode())

    def e2e_abi_check(self, st):
        assert np.array_equal(self.h["rs"], self.rs.cpu().numpy())
        assert np.array_equal(self.h["fo"], self.fo.cpu().numpy().view(np.uint32))
        assert np.array_equal(self.h["rcl"], self.rcl.cpu().numpy().view(np.uint32))

    def e2e_abi_free(self):
        import loongcollector_b200 as lc
        self.hin = self.h = None
        for p_ in self._pins:
            lc.lib().lc_host_free(p_)

    def cpu_baseline(self):
        from loongcollector_b200 import synth
        from oracle import oracle as orc
        cores = len(os.sched_getaffinity(0)) or 1
        per = max(1, min(self.n // cores, 32768))
        rxs = [orc.Regex(synth.CSV_URL_PATTERN) for _ in range(cores)]

        def work(t):
            a = t * per
            est, enf, efo, efl, efd = orc.delim_parse_batch(self.buf, self.off[a:a + per], self.ln[a:a + per], b",",
                                                            ord('"'), 10, True, True, self.MF)
            orc.regex_parse_batch(rxs[t], self.buf, efo[:, 3].copy(), efl[:, 3].copy(), self.G)

        dt = cpu_threads_run(work, cores)
        by = int(self.ln[:per * cores].astype(np.int64).sum() + per * cores)
        return {"value": by / dt / 1e6, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": "%d CSV lines per thread on %d threads, flat oracle delimiter FSM + PCRE2 on column 3" %
                          (per, cores)}


class C5(Config):
    name = "c5"
    metric = "multi_pattern_regex_parsed_log_MBps"
    dominant = "regex_tdfa_multi_kernel"
    SUB = 1 << 20  # lines per engine call (one call stays below the 4 GiB arena limit)

    def workload(self):
        return "C5: nginx + apache multi-pattern regex (both patterns offered to every line in one grid), line length " \
               "Zipf(1.1) clipped to [120, 8191] B (%.0f B avg), %d lines per GPU as %d calls of %d lines" % \
               (self.in_bytes / self.n, self.n, self.nsub, self.sub)

    def setup_host(self):
        from loongcollector_b200 import synth
        self.n = self.args.lines or (8 << 20)
        self.sub = min(self.SUB, self.n)
        self.nsub = (self.n + self.sub - 1) // self.sub
        self.n = self.sub * self.nsub
        self.pool, self.kinds = synth.zipf_mixed_pool(1 << 20, seed=shard_seed(self.rank))
        self.nkeys = [10, 11]
        self.units = self.n

    def setup(self):
        import torch
        import loongcollector_b200 as lc
        from loongcollector_b200 import synth
        self.setup_host()
        pool, kinds = self.pool, self.kinds
        plen = np.array([len(p) for p in pool], np.int64)  # with '\n'
        W = int(plen.max())
        mat = np.zeros((len(pool), W), np.uint8)
        for k, p in enumerate(pool):
            mat[k, :len(p)] = np.frombuffer(p, np.uint8)
        d_mat = self.dput(mat)
        d_plen = self.dput(plen)
        self.rxs = [lc.Regex(synth.NGINX_PATTERN), lc.Regex(synth.APACHE_PATTERN)]
        self.nkeys = [10, 11]
        self.GP = 11
        self.subs = []
        g = torch.Generator(device=self.dev)
        total_bytes = 0
        self.alg_bytes = 0
        col = torch.arange(W, device=self.dev)[None, :]
        for s in range(self.nsub):
            g.manual_seed(shard_seed(self.rank) * 1000 + s)
            idx = torch.randint(0, len(pool), (self.sub,), generator=g, device=self.dev)
            lens = d_plen[idx]
            off = torch.cumsum(lens, 0) - lens
            nbytes = int(lens.sum().item())
            d_buf = torch.empty(nbytes + 16, dtype=torch.uint8, device=self.dev)
            at = 0
            CH = 1 << 16
            for a in range(0, self.sub, CH):
                ii = idx[a:a + CH]
                rows = d_mat[ii]
                m = col < lens[a:a + CH, None]
                cnt = int(lens[a:a + CH].sum().item())
                torch.masked_select(rows, m, out=d_buf[at:at + cnt])
                at += cnt
            self.subs.append({"buf": d_buf, "bytes": nbytes, "off": off.to(torch.int32), "idx": idx,
                              "len": (lens - 1).to(torch.int32)})
            total_bytes += nbytes
            napache = int(torch.from_numpy(kinds).to(self.dev)[idx].sum().item())
            self.alg_bytes += int((lens - 1).sum().item()) + (self.sub - napache) * 89 + napache * 97
        self.in_bytes = total_bytes
        self.units = self.n
        self.d_wh = torch.empty(self.sub, dtype=torch.uint8, device=self.dev)
        self.d_st = torch.empty(self.sub, dtype=torch.uint8, device=self.dev)
        self.d_co = torch.empty(self.sub * self.GP, dtype=torch.int32, device=self.dev)
        self.d_cl = torch.empty(self.sub * self.GP, dtype=torch.int32, device=self.dev)
        self.extra = {"sub_batches": self.nsub}

    def run_sub(self, s):
        b = self.subs[s]
        self.eng.regex_parse_multi_dev(self.rxs, self.nkeys, b["buf"].data_ptr(), b["bytes"], b["off"].data_ptr(),
                                       b["len"].data_ptr(), self.sub, None, self.d_wh.data_ptr(), self.d_st.data_ptr(),
                                       self.GP, self.d_co.data_ptr(), self.d_cl.data_ptr())

    def step(self):
        for s in range(self.nsub):
            self.run_sub(s)

    def outputs(self):
        """the tables of the step's last call (the calls share them)"""
        return {"which": self.d_wh.cpu().numpy(), "status": self.d_st.cpu().numpy(),
                "cap_off": self.d_co.cpu().numpy().view(np.uint32).reshape(self.sub, self.GP),
                "cap_len": self.d_cl.cpu().numpy().view(np.uint32).reshape(self.sub, self.GP)}

    def check(self):
        """every row of the LAST sub-batch against the oracle: per-pattern PCRE2 results on the pool lines, merged
        first-match-wins and expanded through the sampling index"""
        from loongcollector_b200 import synth
        from oracle import oracle as orc
        pool = self.pool
        plen = np.array([len(p) - 1 for p in pool], np.uint32)
        poff = np.zeros(len(pool), np.uint32)
        poff[1:] = np.cumsum(plen[:-1].astype(np.int64) + 1).astype(np.uint32)
        pbuf = np.frombuffer(b"".join(pool), np.uint8)
        t0 = time.perf_counter()
        per = [orc.regex_parse_batch(orc.Regex(p), pbuf, poff, plen, k)
               for p, k in zip((synth.NGINX_PATTERN, synth.APACHE_PATTERN), self.nkeys)]
        dt = time.perf_counter() - t0
        b = self.subs[-1]
        idx = b["idx"].cpu().numpy()
        off = b["off"].cpu().numpy().view(np.uint32)
        which = np.full(len(pool), 0xFF, np.uint8)
        st = np.ones(len(pool), np.uint8)
        co = np.zeros((len(pool), self.GP), np.int64)
        cl = np.zeros((len(pool), self.GP), np.uint32)
        for p, (pst, pco, pcl) in enumerate(per):
            take = (which == 0xFF) & (pst != 1)
            which[take] = p
            st[take] = pst[take]
            okr = take & (pst == 0)
            g = pco.shape[1]
            co[okr, :g] = pco[okr].astype(np.int64) - poff[okr, None].astype(np.int64)
            cl[okr, :g] = pcl[okr]
        valid = np.zeros((len(pool), self.GP), bool)
        for p, (pst, pco, pcl) in enumerate(per):
            valid[(which == p) & (st == 0), :pco.shape[1]] = True
        e_co = ((co[idx] + off[:, None].astype(np.int64)) * valid[idx]).astype(np.uint32)
        assert np.array_equal(self.d_wh.cpu().numpy(), which[idx])
        assert np.array_equal(self.d_st.cpu().numpy(), st[idx])
        assert np.array_equal(self.d_co.cpu().numpy().view(np.uint32).reshape(self.sub, self.GP), e_co)
        assert np.array_equal(self.d_cl.cpu().numpy().view(np.uint32).reshape(self.sub, self.GP), cl[idx])
        return {"cpu_1thread": {"value": pbuf.size / dt / 1e6, "unit": UNIT, "cores": 1, "kind": "port",
                                "sample": "%d pool lines (%d bytes), both patterns tried per line, flat oracle "
                                          "(PCRE2 interpretive), 1 thread" % (len(pool), pbuf.size)}}

    def e2e_abi_setup(self):
        b = self.subs[0]
        self._pins = []
        self.hb = pinned_array(self._pins, b["buf"][:b["bytes"]].cpu().numpy(), np.uint8)
        self.ho = pinned_array(self._pins, b["off"].cpu().numpy().view(np.uint32), np.uint32)
        self.hl = pinned_array(self._pins, b["len"].cpu().numpy().view(np.uint32), np.uint32)
        n = self.sub
        self.h = {"wh": pinned_array(self._pins, n, np.uint8), "st": pinned_array(self._pins, n, np.uint8),
                  "co": pinned_array(self._pins, n * self.GP * 4, np.uint32),
                  "cl": pinned_array(self._pins, n * self.GP * 4, np.uint32)}
        self._multi = self.eng._multi_handles(self.rxs, self.nkeys)
        self.e2e_h2d = int(b["bytes"] + 8 * n)
        self.e2e_d2h = int(n * (2 + 8 * self.GP))
        self.e2e_bytes = int(b["bytes"])

    def e2e_abi_step(self):
        import loongcollector_b200 as lc
        L = lc.lib()
        arr, nk = self._multi
        rc = L.lc_regex_parse_multi(self.eng._h, arr, len(self.rxs), _vp(nk), _vp(self.hb), self.hb.size, _vp(self.ho),
                                    _vp(self.hl), self.sub, None, _vp(self.h["wh"]), _vp(self.h["st"]), self.GP,
                                    _vp(self.h["co"]), _vp(self.h["cl"]))
        if rc != 0:
            raise RuntimeError(L.lc_last_error().decode())

    def e2e_abi_check(self, st):
        pass

    def e2e_abi_free(self):
        pass

    def cpu_baseline(self):
        from loongcollector_b200 import synth
        from oracle import oracle as orc
        cores = len(os.sched_getaffinity(0)) or 1
        pool = self.pool
        plen = np.array([len(p) - 1 for p in pool], np.uint32)
        poff = np.zeros(len(pool), np.uint32)
        poff[1:] = np.cumsum(plen[:-1].astype(np.int64) + 1).astype(np.uint32)
        pbuf = np.frombuffer(b"".join(pool), np.uint8)
        per = max(1, len(pool) // cores)
        rxs = [(orc.Regex(synth.NGINX_PATTERN), orc.Regex(synth.APACHE_PATTERN)) for _ in range(cores)]

        def work(t):
            a = (t * per) % max(1, len(pool) - per)
            for _ in range(4):
                st, _, _ = orc.regex_parse_batch(rxs[t][0], pbuf, poff[a:a + per], plen[a:a + per], 10)
                rest = st == 1  # first-match-wins: only lines the first pattern rejected see the second
                orc.regex_parse_batch(rxs[t][1], pbuf, poff[a:a + per][rest].copy(), plen[a:a + per][rest].copy(), 11)

        dt = cpu_threads_run(work, cores)
        by = 4 * cores * int(plen[:per].astype(np.int64).sum() + per)
        return {"value": by / dt / 1e6, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": "%d pool lines per thread x 4 passes on %d threads, flat oracle: nginx pattern, then the "
                          "apache pattern on the lines it rejected" % (per, cores)}


CONFIGS = {"c1": C1, "c2": C2, "c3": C3, "c4": C4, "c5": C5}


# ------------------------------------------------------------------------------------------------ reference arm
def run_reference(args):
    """The reference's own CPU path on all host cores, same config / metric / unit as the GPU arm.  c2: the flat oracle
    (PCRE2 regex_match per line; boost.regex is not installable here, kind = "port") over the SAME 4 Mi lines per step
    as the GPU arm -- the boundary `e2e` is measured at -- plus, as `plugin`, the plugin-level CPU arm
    (oracle/ref_plugin.cpp) that `e2e_plugin` compares with.  Other configs: the flat oracle on a bounded sample."""
    rank, local_rank, world = dist_env()
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0)) or 1
    if args.config == "c2":
        from loongcollector_b200 import synth
        n = args.lines or 4 * 1024 * 1024
        buf, off, ln = make_workload(n, shard_seed(0))
        reps = args.steps or 30
        for _ in range(min(args.warmup, 2)):
            cpu_regex_parse(synth.NGINX_PATTERN, len(synth.NGINX_KEYS), buf, off, ln, cores)
        ts = np.array([cpu_regex_parse(synth.NGINX_PATTERN, len(synth.NGINX_KEYS), buf, off, ln, cores)[0]
                       for _ in range(reps)])
        dt = float(np.median(ts))
        in_bytes = int(buf.size)
        v = in_bytes / dt / 1e6
        sample = "%d lines x 256 B per step (the GPU arm's whole batch), flat oracle on %d threads: PCRE2 10.42 " \
                 "interpretive regex_match + capture table per line, one matcher per thread " \
                 "(oracle/lc_oracle.c restates ProcessorParseRegexNative.cpp:186-253)" % (n, cores)
        line = {"workload": "C2: ProcessorParseRegexNative nginx 10-group regex, %d lines x 256 B per GPU" % n,
                "lines_per_gpu": n, "line_bytes": 256}
        units = n
        metric = C2.metric
        psecs, pstats = cpu_plugin_regex(buf, off, ln, cores, 3)
        extra = {"seconds_min": float(ts.min()), "seconds_max": float(ts.max()),
                 "plugin": {"value": in_bytes / float(np.median(psecs)) / 1e6, "unit": UNIT,
                            "sample": "the same lines in %d groups of <= 512 KB, Process(group) on %d threads "
                                      "(oracle/ref_plugin.cpp); median of 3" % (pstats["groups"], cores),
                            "plugin_stats": pstats}}
    else:
        # the flat oracle on all host cores, one bounded sample of the config's workload per step
        cfg = CONFIGS[args.config](args, 0, 1, None, None)
        cfg.setup_host()
        for _ in range(min(args.warmup, 1)):
            cfg.cpu_baseline()
        res = [cfg.cpu_baseline() for _ in range(args.steps or 30)]
        vals = np.array([r["value"] for r in res])
        v = float(np.median(vals))
        sample = res[0]["sample"]
        reps = len(res)
        dt = 0.0
        cfg.in_bytes = getattr(cfg, "in_bytes", 0)
        line = {"workload": "%s (bounded sample per step: %s)" % (args.config.upper(), sample)}
        units = 0
        metric = cfg.metric
        extra = {"value_min": float(vals.min()), "value_max": float(vals.max())}
    print(json.dumps({
        "impl": "reference", "metric": metric, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": reps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": line,
        "lines_per_s": (units / dt) if dt else None,
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, **extra,
    }))


# ------------------------------------------------------------------------------------------------ GPU arm
def run_ours(args):
    import torch
    import loongcollector_b200 as lc

    rank, local_rank, world = dist_env()
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    placement = pin_to_gpu_numa(local_rank)
    eng = lc.Engine(local_rank)
    stream = torch.cuda.ExternalStream(eng.stream, device=dev)
    cfg = CONFIGS[args.config](args, rank, world, eng, dev)
    cfg.setup()
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    W = max(args.warmup, 3)
    sampler = ClockSampler(local_rank)
    sampler.start()  # >= 1 s before the timed region: the first samples of nvidia-smi -lms are slow to arrive
    t_sampler = time.time()
    # ---- warm-up: the device kept busy until the sampler has run for 1.2 s, then W steps back to back between two
    # CUDA events, whose time per step sizes the default K and the chunks
    warm = 0
    w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        while time.time() - t_sampler < 1.2:
            cfg.step()
            torch.cuda.synchronize()
            warm += 1
        w0.record(stream)
        for _ in range(W):
            cfg.step()
        w1.record(stream)
    torch.cuda.synchronize()
    warm += W
    step_ms = w0.elapsed_time(w1) / W
    # the warm-up's steps run up to a few % slower than the region's: sized for 10 % more than REGION_S
    K = args.steps or int(np.ceil(1.1 * REGION_S * 1e3 / step_ms))
    if world > 1 and not args.steps:  # the same K everywhere
        t = torch.tensor([K], dtype=torch.int64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        K = int(t.item())
    # the K steps in chunks of >= CHUNK_MS between CUDA events, for a median / min / max over the chunks
    n_chunks = max(1, min(MAX_CHUNKS, K, int(K * step_ms // CHUNK_MS)))
    bounds = [K * i // n_chunks for i in range(n_chunks + 1)]
    ev = [torch.cuda.Event(enable_timing=True) for _ in bounds]
    barrier()
    sampler.mark_region()
    with torch.cuda.stream(stream):
        cfg.step()  # one more warm-up step, queued right ahead: the region starts on a busy device
        warm += 1
        launches0 = eng.launches
        ev[0].record(stream)
        for i in range(n_chunks):
            for _ in range(bounds[i + 1] - bounds[i]):
                cfg.step()
            ev[i + 1].record(stream)
    barrier()
    clocks = sampler.stop()
    launches_total = eng.launches - launches0
    per_step = np.array([a.elapsed_time(b) for a, b in zip(ev[:-1], ev[1:])]) / np.diff(bounds)
    med, mn, mx = float(np.median(per_step)), float(per_step.min()), float(per_step.max())
    if hasattr(cfg, "finish_setup"):
        cfg.finish_setup()
    if rank == 0 and args.dump_outputs:
        dump_outputs(cfg, args.dump_outputs)
    value, ms_per_step = job_throughput(cfg.in_bytes, med, world, dev)
    value_best, _ = job_throughput(cfg.in_bytes, mn, world, dev)
    per_rank = gather_rank_stats([mn, med, mx], world, dev)
    total_units = cfg.units * world

    checks = {}
    if rank == 0:
        checks = cfg.check()
    st = cfg.results()[0] if hasattr(cfg, "results") else None

    # ---- end to end with host buffers
    e2e = None
    e2e_plugin = None
    mode = "none" if args.no_e2e else args.e2e
    if mode == "auto":
        mode = "plugin" if args.config == "c2" else "abi"
    if mode in ("plugin", "abi"):
        import torch
        torch.cuda.synchronize()
        cfg.e2e_abi_setup()
        cfg.e2e_abi_step()
        barrier()
        reps = max(3, min(K, 7))
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            cfg.e2e_abi_step()
            ts.append(time.perf_counter() - t0)
        barrier()
        cfg.e2e_abi_check(st)
        e_bytes = getattr(cfg, "e2e_bytes", cfg.in_bytes)
        v, ms = job_throughput(e_bytes, float(np.median(ts)) * 1e3, world, dev)
        e2e = {"value": v, "unit": UNIT, "h2d_bytes_per_step": cfg.e2e_h2d, "d2h_bytes_per_step": cfg.e2e_d2h,
               "ms_per_step": ms, "steps": reps,
               "api": "host-pointer C-ABI call(s) of the path (include/lc_b200.h), one pinned arena per step",
               "per_rank_ms": gather_rank_stats([min(ts) * 1e3, float(np.median(ts)) * 1e3, max(ts) * 1e3],
                                                world, dev)}
        cfg.e2e_abi_free()
    if mode == "plugin" and hasattr(cfg, "e2e_plugin"):
        from loongcollector_b200 import synth
        barrier()
        reps = max(3, min(K, 5))
        secs, stats = cfg.e2e_plugin(reps + 1, mode=1)
        secs = secs[1:]  # the first repetition warms the thread's engine, its workspace and the pinned tables
        barrier()
        sts, co, cl = cfg.results()
        want = expected_plugin_stats(cfg.buf, sts, co, cl, synth.NGINX_KEYS)
        for k, v_ in want.items():
            assert stats[k] == v_, "plugin result differs from the device-API result: %s %d != %d" % (k, stats[k], v_)
        v, ms = job_throughput(cfg.in_bytes, float(np.median(secs)) * 1e3, world, dev)
        nrep = reps + 1
        e2e_plugin = {"value": v, "unit": UNIT, "h2d_bytes_per_step": int(stats["arena_bytes"] + 8 * cfg.n),
                      "d2h_bytes_per_step": int(cfg.n * (1 + 8 * cfg.G)), "ms_per_step": ms, "steps": reps,
                      "api": "ProcessorInstance::Process(std::vector<PipelineEventGroup>&) of the B200-backed "
                             "ProcessorParseRegexNative, %d groups of <= %d KB (pinned SourceBuffer arenas), "
                             "LC_B200_HOST_THREADS=%s" % (stats["groups"], GROUP_BYTES // 1024,
                                                          os.environ.get("LC_B200_HOST_THREADS", "default")),
                      "phase_ms_per_step": {"gather": stats["gather_ns"] / nrep / 1e6,
                                            "engine_call": stats["engine_ns"] / nrep / 1e6,
                                            "epilogue_overlapped_with_engine": stats["epilogue_ns"] / nrep / 1e6,
                                            "process_total": stats["ctr_process_ns"] / nrep / 1e6},
                      "per_rank_ms": gather_rank_stats([float(secs.min()) * 1e3, float(np.median(secs)) * 1e3,
                                                        float(secs.max()) * 1e3], world, dev),
                      "plugin_stats": stats}
        # the same plugin, one group per Process call (what a single ProcessorRunner thread does today)
        if rank == 0 and world == 1:
            ns = min(cfg.n, 1 << 19)
            sub = C2(args, rank, world, eng, dev)
            sub.n, sub.buf, sub.off, sub.ln = ns, cfg.buf, cfg.off[:ns], cfg.ln[:ns]
            s1, st1 = sub.e2e_plugin(3, mode=0)
            e2e_plugin["per_group_calls"] = {"value": ns * 256 / float(np.median(s1[1:])) / 1e6, "unit": UNIT,
                                             "sample": "%d lines, %d Process(group) calls, 1 thread" %
                                                       (ns, st1["groups"])}

    # ---- CPU baseline (rank 0, N == 1 only): all host cores on a bounded sample
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cfg.cpu_baseline()

    peak, peak_src = hbm_peak()
    achieved = cfg.alg_bytes / (ms_per_step * 1e-3) / 1e9
    traffic, traffic_src = profile_traffic(args.config)
    if rank == 0:
        out = {
            "metric": cfg.metric, "value": value, "unit": UNIT, "n_gpus": world, "steps": K,
            "warmup": warm, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": cfg.workload(), "units_per_gpu": cfg.units, "bytes_per_gpu": cfg.in_bytes,
                       "l2": "inputs (%.0f MB per GPU) larger than L2, no flush" % (cfg.in_bytes / 1e6),
                       **cfg.extra},
            "timing": {"statistic": "median over chunks of the K steps of (CUDA-event time of the chunk / its steps), "
                                    "max over ranks",
                       "chunks": n_chunks, "timed_region_s": float((per_step * np.diff(bounds)).sum() / 1e3),
                       "ms_per_step_min": mn, "ms_per_step_max": mx, "value_at_min": value_best,
                       "per_rank_ms_per_step_min_med_max": per_rank},
            "lines_per_s": total_units / (ms_per_step * 1e-3),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "algorithmic_bytes_per_step": cfg.alg_bytes, "kernel": cfg.dominant,
                         "kernel_ms": ms_per_step},
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches_total),
            "gpu_launches_per_step": launches_total / float(K), "clocks": clocks, "host_placement": placement,
        }
        if e2e_plugin is not None:
            out["e2e_plugin"] = e2e_plugin
        out.update(checks)
        print(json.dumps(out))
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
