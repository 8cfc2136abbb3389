#!/usr/bin/env python
"""bench.py — Mbp decoded per second, one JSON line on rank 0.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--windows M] [--config 2|3] [--impl reference] [--dump-outputs DIR]

Default (--config 2): BASELINE.json configs[1], synthetic 50 kb human-composition windows, --species=human ab initio.
A "step" is one pass of the whole hot path (prep -> sweep -> backtrace -> pack) over the rank's batch of windows.  `value` is
timed with CUDA events on the library's launch stream with the inputs already in HBM over K steps; `e2e` is the same metric through
the public call (augb200_decode_batch) from host buffers, with the host->device copy of the windows and the device->host copy of the
paths inside the timed region, also over K steps.  The job is world x M windows; no data-path collective; one NCCL gather of the final
path arrays ends each e2e step.  After a first measurement the windows are re-dealt in proportion to each rank's measured sweep rate (the same
kernel runs up to 17 % slower on some GPUs of a node, SCALE_r01.json), `config.windows_per_gpu` lists the counts.
The paths produced in the timed regions are checked against the reference's digests (tests/golden/ref_config2_digests.json):
`verified` = number of windows compared, a mismatch aborts the run.
`--dump-outputs DIR` writes the paths of the last device-resident step as float64 .npy files (dump_paths), so that two builds run
with the same arguments can be compared output for output.

--config 3: BASELINE.json configs[2], examples/chr2L in 157 windows of 200 kb, --species=fly defaults (UTR + softmasking +
sample=100), windows sharded over the ranks; the same line layout.  The default run carries it under `secondary`.

`--impl reference` times the reference's own CPU implementation (oracle/_ref/augustus, the unmodified AUGUSTUS binary built by
oracle/Makefile) on the box's host cores on a bounded sample of the same windows.  The core count is what the process may really
use (affinity mask, cgroup quota) and is calibrated against a single-process run (`cpu_baseline.single_process_mbp_s`,
`effective_cores`): round 1 reported 128 cores on a box whose 128 pinned processes shared far fewer.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WINDOW_LEN = 50000
DEFAULT_WINDOWS = 10000
METRIC = "Mbp decoded/sec"
# SURVEY.md §8d: dense column-banded figure, 0.25 + S*(8+8+4) [+ S*16 with the forward matrix]
ALG_BYTES = {"vit47": 0.25 + 47 * 20, "vit71": 0.25 + 71 * 20, "fwd47": 0.25 + 47 * 36, "fwd71": 0.25 + 71 * 36}
VERIFY_PER_RANK = 64


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


# --------------------------------------------------------------------------------------------- host cores
def usable_cores():
    """CPUs this process may really run on: the affinity mask, capped by the cgroup CPU quota (os.cpu_count() ignores both)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    quota = None
    try:                                                # cgroup v2
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(p)
    except Exception:
        try:                                            # cgroup v1
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    if quota:
        n = max(1, min(n, int(quota + 0.5)))
    return n


def cpu_list():
    try:
        return sorted(os.sched_getaffinity(0))
    except AttributeError:
        return list(range(os.cpu_count() or 1))


# --------------------------------------------------------------------------------------------- reference arm
def ref_binary():
    exe = os.path.join(ROOT, "oracle", "_ref", "augustus")
    cfg = os.path.join(ROOT, "oracle", "_ref", "config")
    return (exe, cfg) if os.path.exists(exe) and os.path.isdir(cfg) else (None, None)


def run_reference_sample(n_windows, procs, start_index=0, extra_args=(), window_len=None, seqs=None, base_args=("--species=human", "--softmasking=0"),
                         one_per_process=False):
    """Decode n_windows synthetic windows (or the given sequences) with the unmodified reference, `procs` processes at a time, each
    pinned to one of the CPUs of the affinity mask.  Returns (Mbp/s, seconds)."""
    from augustus_b200 import synth
    exe, cfg = ref_binary()
    if exe is None:
        raise RuntimeError("oracle/_ref/augustus is missing (run __graft_entry__.build() in the build container)")
    env = dict(os.environ, AUGUSTUS_CONFIG_PATH=cfg)
    wlen = window_len or WINDOW_LEN
    cpus = cpu_list()
    if seqs is not None:
        n_windows = len(seqs)
    with tempfile.TemporaryDirectory() as td:
        files = []
        nfile = n_windows if one_per_process else procs
        per = [[] for _ in range(nfile)]
        for i in range(n_windows):
            per[i % nfile].append(start_index + i)
        for c, idxs in enumerate(per):
            if not idxs:
                continue
            fa = os.path.join(td, "c%d.fa" % c)
            synth.write_fasta(fa, [seqs[i - start_index] if seqs is not None else synth.window(i, wlen) for i in idxs], ["w%d" % i for i in idxs])
            files.append(fa)
        mbp = (sum(len(s) for s in seqs) if seqs is not None else n_windows * wlen) / 1e6
        t0 = time.perf_counter()
        if one_per_process and len(files) > procs:      # more windows than processes: a pool of `procs` running processes
            import concurrent.futures as cf

            def one(a):
                c, fa = a
                return subprocess.run([exe] + list(base_args) + list(extra_args) + [fa], env=env, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL).returncode
            with cf.ThreadPoolExecutor(procs) as ex:
                if any(ex.map(one, enumerate(files))):
                    raise RuntimeError("reference process failed")
            dt = time.perf_counter() - t0
            return mbp / dt, dt
        running = []
        for c, fa in enumerate(files):
            cmd = [exe] + list(base_args) + list(extra_args) + [fa]
            if os.path.exists("/usr/bin/taskset"):
                cmd = ["taskset", "-c", str(cpus[c % len(cpus)])] + cmd
            running.append(subprocess.Popen(cmd, env=env, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL))
        for p in running:
            if p.wait() != 0:
                raise RuntimeError("reference process failed")
        dt = time.perf_counter() - t0
    return mbp / dt, dt


_single = {}


def single_process_rate(extra_args=(), window_len=None, base_args=("--species=human", "--softmasking=0"), seq=None):
    """Mbp/s of ONE reference process on one window while the box is otherwise idle (calibration of the full-box number)."""
    key = (tuple(extra_args), window_len, tuple(base_args), None if seq is None else len(seq))
    if key not in _single:
        _single[key] = run_reference_sample(1, 1, start_index=7, extra_args=extra_args, window_len=window_len, base_args=base_args,
                                            seqs=None if seq is None else [seq])[0]
    return _single[key]


def calibrated_reference(n_per_proc=2, start_index=0, **kw):
    """The reference on the whole box, calibrated.  One process per usable core; if the per-core rate of that run is below half of a
    lone process (the "cores" are not really there: SMT siblings, an oversubscribed host, a quota the cgroup files do not show), the
    run is repeated with as many processes as the first run was worth and the better total counts.  Returns the cpu_baseline dict."""
    cores = usable_cores()
    r1 = single_process_rate(**kw)
    v, dt = run_reference_sample(cores * n_per_proc, cores, start_index, **kw)
    info = {"value": v, "unit": "Mbp/s", "cores": cores, "kind": "reference", "single_process_mbp_s": r1, "per_core_mbp_s": v / cores,
            "effective_cores": v / r1, "os_cpu_count": os.cpu_count(),
            "sample": "%d windows, one unmodified augustus process per usable core (%d), %.1f s wall" % (cores * n_per_proc, cores, dt)}
    if v / cores < 0.5 * r1 and cores > 1:
        eff = max(1, int(v / r1 + 0.5))
        v2, dt2 = run_reference_sample(eff * n_per_proc, eff, start_index, **kw)
        info["starved"] = ("full-box per-core rate %.4f Mbp/s is below half of a lone process (%.4f): the box gives this job about %.0f cores' worth "
                           "of CPU, not %d; second run with %d processes: %.3f Mbp/s" % (v / cores, r1, v / r1, cores, eff, v2))
        if v2 > v:
            info.update({"value": v2, "cores": eff, "per_core_mbp_s": v2 / eff, "effective_cores": v2 / r1,
                         "sample": "%d windows, %d processes (%.1f s wall; the %d-process run was slower per core, see `starved`)" % (eff * n_per_proc, eff, dt2, cores)})
    return info


def chr2l_windows(window=200000, step=150000):
    """BASELINE.json configs[2]: examples/chr2L cut into 200 kb windows stepping 150 kb (SURVEY.md 8d: 157 windows).  The FASTA is
    reference DATA copied to oracle/_ref/data/ by oracle/Makefile (it travels with the built checker; never read from /root/reference)."""
    import gzip
    path = os.path.join(ROOT, "oracle", "_ref", "data", "chr2L.sm.fa.gz")
    if not os.path.exists(path):
        return None
    seq = "".join(l.strip() for l in gzip.open(path, "rt") if not l.startswith(">"))
    out = []
    a = 0
    while True:
        out.append(seq[a:a + window])
        if a + window >= len(seq):
            break
        a += step
    return out


def reference_arm(args, rank, world):
    if rank != 0:
        return
    exe, _ = ref_binary()
    if exe is None:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/augustus not built"}))
        return
    cores = usable_cores()
    if args.config == 3:
        w3 = chr2l_windows()
        sub = w3[: max(1, min(len(w3), cores))]
        tot_t = 0.0
        for _ in range(max(1, min(args.steps, 1))):
            v, dt = run_reference_sample(0, cores, seqs=sub, base_args=("--species=fly",), one_per_process=True)
            tot_t += dt
        r1 = None
        line = {"metric": METRIC, "unit": "Mbp/s", "n_gpus": args.gpus, "steps": 1, "warmup": 0, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f64 (LLDouble)", "data": "examples/chr2L (reference data)", "impl": "reference", "value": v, "ms_per_step": 1e3 * tot_t,
                "config": {"workload": "examples/chr2L in 200 kb windows, --species=fly defaults (BASELINE.json configs[2])", "windows_per_step": len(sub)},
                "cpu_baseline": {"value": v, "unit": "Mbp/s", "cores": min(cores, len(sub)), "kind": "reference",
                                 "sample": "%d of the 157 windows, one augustus --species=fly process per window, %.1f s wall" % (len(sub), tot_t)},
                "e2e": {"value": v, "unit": "Mbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return
    per_step = cores * 2
    base = {"metric": METRIC, "unit": "Mbp/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64 (LLDouble)", "data": "synthetic",
            "impl": "reference",
            "config": {"workload": "synthetic 50 kb human-composition windows, --species=human ab initio (BASELINE.json configs[1])",
                       "window_len": WINDOW_LEN, "windows_per_step": per_step}}
    r1 = single_process_rate()
    for w in range(min(args.warmup, 1)):
        run_reference_sample(cores, cores, 0)
    tot_t, tot_w = 0.0, 0
    for s in range(args.steps):
        _, dt = run_reference_sample(per_step, cores, s * per_step)
        tot_t += dt
        tot_w += per_step
    v = tot_w * WINDOW_LEN / 1e6 / tot_t
    cb = {"value": v, "unit": "Mbp/s", "cores": cores, "kind": "reference", "single_process_mbp_s": r1, "per_core_mbp_s": v / cores,
          "effective_cores": v / r1, "os_cpu_count": os.cpu_count(),
          "sample": "%d windows x 50 kb per step, one unmodified augustus process per usable core (%d)" % (per_step, cores)}
    if v / cores < 0.5 * r1:
        cb["starved"] = "per-core rate %.4f Mbp/s < half of a lone process (%.4f): this box gives the job about %.0f cores' worth of CPU" % (v / cores, r1, v / r1)
    base.update({"value": v, "ms_per_step": 1e3 * tot_t / args.steps, "cpu_baseline": cb,
                 "e2e": {"value": v, "unit": "Mbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
    print(json.dumps(base))


# --------------------------------------------------------------------------------------------- checking the timed outputs
def path_digest(states):
    return hashlib.sha1(json.dumps([[int(v) for v in s] for s in states], separators=(",", ":")).encode()).hexdigest()


def load_digests():
    try:
        return json.load(open(os.path.join(ROOT, "tests", "golden", "ref_config2_digests.json")))["windows"]
    except Exception:
        return {}


def verify_paths(tuples_of, my_idx, digests, limit=VERIFY_PER_RANK):
    """Compare this rank's paths with the reference digests: tuples_of(k) = condensed path of the rank's k-th window."""
    n = 0
    for k, g in enumerate(my_idx):
        ref = digests.get(str(g))
        if ref is None:
            continue
        st = tuples_of(k)
        if path_digest(st) != ref["sha1"]:
            raise SystemExit("bench: window %d decoded in the timed region differs from the reference's path" % g)
        n += 1
        if n >= limit:
            break
    return n


def raw_tuples(raw, k):
    n_st, status, logp, offset, pb, pe, pt, ptr = raw
    o, n = int(offset[k]), int(n_st[k])
    return [(int(pt[o + i]), int(pb[o + i]), int(pe[o + i]), int(ptr[o + i])) for i in range(n)]


DUMP_BYTES = 63_000_000         # array data of --dump-outputs: with the .npy headers under 64 MB
DUMP_SEED = 20261017


def dump_paths(out_dir, window_ids, paths, budget=DUMP_BYTES, prefix=""):
    """Write what a caller of the timed path receives, one float64 .npy per field: per window its global index (`window`), `status`,
    `log_prob` and state count (`n_states`), and the condensed states of those windows concatenated in window order (`type`, `begin`,
    `end`, `truncated`).  When all windows do not fit in `budget` bytes, windows are taken in a fixed seeded order while they fit and
    written in index order; `window` says which."""
    import numpy as np
    cost = np.array([8 * (4 + 4 * len(p.states)) for p in paths], dtype=np.int64)       # 4 per-window values + 4 per state
    keep = np.arange(len(paths))
    if cost.sum() > budget:
        order = np.random.default_rng(DUMP_SEED).permutation(len(paths))
        keep = np.sort(order[:int(np.argmin(np.cumsum(cost[order]) <= budget))])
    sel = [paths[k] for k in keep]
    rows = np.array([(s.type, s.begin, s.end, s.truncated) for p in sel for s in p.states], dtype=np.float64).reshape(-1, 4)
    arrays = {"window": np.asarray(window_ids, dtype=np.float64)[keep], "status": [p.status for p in sel],
              "log_prob": [p.log_prob for p in sel], "n_states": [len(p.states) for p in sel],
              "type": rows[:, 0], "begin": rows[:, 1], "end": rows[:, 2], "truncated": rows[:, 3]}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), np.asarray(a, dtype=np.float64))


def deal_windows(world, M, rates):
    """Window indices per rank: block-cyclic (window g -> rank g mod world), then the slower ranks hand their last windows to the
    faster ones so that the counts are proportional to the measured sweep rates.  Deterministic, the same on every rank."""
    base = [list(range(r, world * M, world)) for r in range(world)]
    if world == 1 or not rates or min(rates) <= 0:
        return base
    tot = world * M
    want = [int(tot * x / sum(rates)) for x in rates]
    for i in range(tot - sum(want)):
        want[i % world] += 1
    if max(abs(w - M) for w in want) * 50 < M:            # within 2 %: leave it
        return base
    pool = []
    for r in range(world):
        if want[r] < M:
            pool += base[r][want[r]:]
            base[r] = base[r][:want[r]]
    for r in range(world):
        if want[r] > M:
            k = want[r] - M
            base[r] += pool[:k]
            pool = pool[k:]
    return base


def dropin_leg(n_chr2l):
    """What a user of the drop-in sees: wall clock of oracle/_ref/augustus_b200 (the reference's front end with its three DP entry points
    bound to libaugb200.so, host/augshim.cc) against oracle/_ref/augustus for the same command lines, GFF compared line by line.
    config 1 = examples/example.fa --species=human; then the first n chr2L windows with --species=fly defaults (UTR, softmasking,
    sample=100), one process per window as scripts/createAugustusJoblist.pl runs a genome: the reference's processes side by side on
    the host cores, the drop-in's one after the other on the GPU."""
    from augustus_b200 import synth
    refdir = os.path.join(ROOT, "oracle", "_ref")
    ref, drop, cfg = os.path.join(refdir, "augustus"), os.path.join(refdir, "augustus_b200"), os.path.join(refdir, "config")
    if not (os.path.exists(ref) and os.path.exists(drop)):
        return {"unavailable": "oracle/_ref/augustus or augustus_b200 not built"}
    env = dict(os.environ, AUGUSTUS_CONFIG_PATH=cfg)

    def run(exe, args):
        t0 = time.perf_counter()
        r = subprocess.run([exe] + args, env=env, capture_output=True, text=True)
        dt = time.perf_counter() - t0
        lines = r.stdout.splitlines()
        if "# command line:" in lines:
            lines = lines[: lines.index("# command line:")]
        return dt, r.returncode, lines
    out = {}
    ex = os.path.join(ROOT, "tests", "golden", "example.fa")
    tr, rc1, g1 = run(ref, ["--species=human", "--softmasking=0", ex])
    run(drop, ["--species=human", "--softmasking=0", ex])                    # (first start of the binary on this box: page-in)
    td_, rc2, g2 = run(drop, ["--species=human", "--softmasking=0", ex])
    out["config1_example_fa"] = {"reference_s": tr, "dropin_s": td_, "gff_identical": rc1 == 0 and rc2 == 0 and g1 == g2, "gff_lines": len(g1),
                                 "note": "11.8 kb in two sequences: the drop-in's time is CUDA start-up"}
    w3 = chr2l_windows()
    if w3 is None or n_chr2l <= 0:
        return out
    pick = w3[1:1 + n_chr2l]
    with tempfile.TemporaryDirectory() as td:
        files = []
        for i, s in enumerate(pick):
            fa = os.path.join(td, "w%d.fa" % i); synth.write_fasta(fa, [s], ["chr2L_w%d" % (i + 1)]); files.append(fa)
        import concurrent.futures as cf
        t0 = time.perf_counter()
        with cf.ThreadPoolExecutor(min(len(files), usable_cores())) as exq:
            refs = list(exq.map(lambda fa: run(ref, ["--species=fly", fa]), files))
        ref_wall = time.perf_counter() - t0
        t0 = time.perf_counter()
        drops = [run(drop, ["--species=fly", fa]) for fa in files]
        drop_wall = time.perf_counter() - t0
    same = all(a[1] == 0 and b[1] == 0 and a[2] == b[2] for a, b in zip(refs, drops))
    mbp = sum(len(s) for s in pick) / 1e6
    out["chr2L_fly_defaults"] = {"windows": len(pick), "gff_identical": same, "gff_lines": sum(len(a[2]) for a in refs),
                                 "reference_s_per_window": sum(a[0] for a in refs) / len(refs), "dropin_s_per_window": sum(b[0] for b in drops) / len(drops),
                                 "reference_wall_s": ref_wall, "reference_processes_side_by_side": min(len(files), usable_cores()), "dropin_wall_s": drop_wall,
                                 "reference_mbp_s": mbp / ref_wall, "dropin_mbp_s": mbp / drop_wall,
                                 "note": "one process per 200 kb window; per window the drop-in pays process + CUDA start-up, the blob export and a GPU that holds ONE warp's work; "
                                         "the batched C ABI (config3_chr2L) decodes all 157 windows in the time of one"}
    return out


# --------------------------------------------------------------------------------------------- our arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--windows", type=int, default=DEFAULT_WINDOWS, help="windows per GPU per step (default: BASELINE.json config 2)")
    ap.add_argument("--config", type=int, default=2, choices=[2, 3], help="2: synthetic 50 kb windows (default); 3: examples/chr2L, fly defaults")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the config 3 / 4 / 5 side measurements")
    ap.add_argument("--dropin-windows", type=int, default=2, help="chr2L windows of the drop-in end-to-end leg (0 = skip the leg)")
    ap.add_argument("--assume-rates", default="", help="testing only: comma-separated per-rank sweep rates to deal by instead of the measured ones")
    ap.add_argument("--no-balance", action="store_true", help="keep the block-cyclic deal (do not re-deal by measured sweep rate)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the paths of the last timed step (config 2) as DIR/<name>.npy, float64, "
                                                          "at most 64 MB in all; with several GPUs each rank's files carry a rank<r>_ prefix")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.config != 2 or args.impl != "b200"):
        ap.error("--dump-outputs writes the paths of the config-2 timed steps of --impl b200")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return
    args.warmup = max(args.warmup, 3)

    import numpy as np
    import torch
    import torch.distributed as dist
    from augustus_b200 import Decoder, synth
    from tests import util

    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    props = torch.cuda.get_device_properties(local)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(vals):
        t = torch.tensor(vals, dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]

    def allsum(vals):
        t = torch.tensor(vals, dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [float(x) for x in t.tolist()]

    def per_rank(v):
        t = torch.zeros(world, dtype=torch.float64, device="cuda"); t[rank] = v
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [float(x) for x in t.tolist()]

    # ---------------------------------------------------------------- config 3: chr2L, fly defaults, windows sharded over the ranks
    def config3():
        w3 = chr2l_windows()
        if w3 is None:
            raise RuntimeError("oracle/_ref/data/chr2L.sm.fa.gz not present")
        mine = list(range(rank, len(w3), world))
        w3b = [w3[i].encode() for i in mine]
        dec3 = Decoder(util.blob_bytes("fly_softmask_utr"), local)
        dec3.decode_batch_sampling_raw(w3b, 100)          # untimed warm-up at full size: pinned and device buffers reach their final size
        barrier(); t0 = time.perf_counter()
        vit3, samp3 = dec3.decode_batch_sampling_raw(w3b, 100)
        torch.cuda.synchronize(); dt_mine = time.perf_counter() - t0
        assert not vit3[1].any() and not samp3[1].any()
        if world > 1:
            shard_ = __import__("augustus_b200.shard", fromlist=["x"])
            shard_.gather_to_rank0(shard_.pack_paths(*vit3), device="cuda")        # the one gather of the final gene-structure arrays
        barrier(); dt3 = time.perf_counter() - t0
        dt3 = allmax([dt3])[0]
        sweep3 = per_rank(dec3.last_sweep_ms)
        # the reference's digests of these windows (tests/golden/ref_chr2L_digests.json: its Viterbi path and its 99 sampled paths)
        nver = 0
        try:
            gold = json.load(open(os.path.join(ROOT, "tests", "golden", "ref_chr2L_digests.json")))["windows"]
        except (OSError, KeyError):
            gold = {}

        def rows(raw, i):
            n, status, logp, offset, b, e, t, tr = raw
            o, k = int(offset[i]), int(n[i])
            return np.stack([t[o:o + k].astype("<i4"), b[o:o + k].astype("<i4"), e[o:o + k].astype("<i4"), tr[o:o + k].astype("<i4")], axis=1)
        for k, g in enumerate(mine):
            r = gold.get(str(g))
            if r is None:
                continue
            ok = hashlib.sha1(np.ascontiguousarray(rows(vit3, k)).tobytes()).hexdigest() == r["viterbi_sha1"]
            h = hashlib.sha1()
            for q in range(99):
                x = rows(samp3, k * 99 + q)
                h.update(np.asarray([len(x)], dtype="<i4").tobytes()); h.update(np.ascontiguousarray(x).tobytes())
            ok &= h.hexdigest() == r["samples_sha1"]
            if not ok:
                raise SystemExit("bench: chr2L window %d (Viterbi path or sampled paths) differs from the reference" % g)
            nver += 1
        nver = int(allsum([nver])[0])
        mbp3 = sum(len(w) for w in w3) / 1e6
        tot_states = int(allsum([int(vit3[0].sum())])[0]); tot_samp = int(allsum([len(samp3[0])])[0])
        dec3.close()
        peak, how = peaks()
        kms = max(sweep3)
        ach = ALG_BYTES["fwd71"] * sum(len(w3[i]) for i in range(0, len(w3), world)) / (sweep3[0] / 1e3) / 1e9 if sweep3[0] > 0 else 0.0
        return {"workload": "examples/chr2L (23.5 Mbp, soft-masked) in %d windows of 200 kb stepping 150 kb, --species=fly defaults (UTR on = 71 states, softmasking on, "
                            "sample=100: Viterbi + forward + 99 sampled paths per window), windows dealt round-robin to %d GPU(s), e2e from host buffers through "
                            "augb200_decode_batch_sampling (+ one NCCL gather of the Viterbi paths)" % (len(w3), world),
                "value": mbp3 / dt3, "unit": "Mbp/s", "windows": len(w3), "seconds": dt3, "per_rank_kernel_ms": [round(x, 1) for x in sweep3],
                "path_states": tot_states, "sampled_paths": tot_samp, "verified": nver,
                "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None, "kernel": "k_sweep_sample_utr",
                             "peak_source": how, "note": "2556 B/base (dense S = 71 with the forward matrix) x rank 0's bases / its fused fill + sampling kernel time; "
                             "one warp per window: %d windows keep %d of %d warp slots busy, the time is the latency of one window" % (len(w3), len(w3), 148 * 16 * world)},
                "kernel_ms_max": kms}

    def config3_cpu(line3):
        cores = usable_cores()
        w3 = chr2l_windows()
        # a bounded sample: one 200 kb fly window costs the reference ~46 s on a free core
        sub = w3[: max(1, min(len(w3), cores // 2 if cores > 1 else 1))]
        v3, d3 = run_reference_sample(0, min(cores, len(sub)), seqs=sub, base_args=("--species=fly",), one_per_process=True)
        line3["cpu_baseline"] = {"value": v3, "unit": "Mbp/s", "cores": min(cores, len(sub)), "kind": "reference",
                                 "per_core_mbp_s": v3 / min(cores, len(sub)), "usable_cores": cores,
                                 "sample": "%d of the windows, one unmodified augustus --species=fly process per window on half of the usable cores (%.1f s wall; "
                                           "a lone process needs about 46 s per window)" % (len(sub), d3)}

    if args.config == 3:
        sampler = ClockSampler(local); sampler.start()
        l3 = config3()
        sampler.stop_flag = True; sampler.join(timeout=2)
        if rank == 0:
            if not args.no_cpu_baseline:
                config3_cpu(l3)
            line = {"metric": METRIC, "value": l3["value"], "unit": "Mbp/s", "n_gpus": world, "steps": 1, "warmup": 1, "ms_per_step": 1e3 * l3["seconds"],
                    "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int64 (Q23.40 fixed-point log scores) + f64 log-sum-exp",
                    "data": "examples/chr2L of the reference (real DNA)", "config": {"workload": l3["workload"], "windows": l3["windows"],
                    "l2": "31 Mbp of windows, 2.6 GB of workspace per GPU: larger than L2"},
                    "e2e": {"value": l3["value"], "unit": "Mbp/s", "h2d_bytes_per_step": int(31.4e6 / world), "d2h_bytes_per_step": int(12 * (l3["path_states"] + 40 * l3["sampled_paths"]) / world)},
                    "gpu_launches": 5 * world, "roofline": l3["roofline"], "clocks": sampler.summary(), "verified": l3["verified"],
                    "per_rank_kernel_ms": l3["per_rank_kernel_ms"]}
            if "cpu_baseline" in l3:
                line["cpu_baseline"] = l3["cpu_baseline"]
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------------------------------------------------------- config 2
    from augustus_b200 import shard
    M = args.windows
    digests = load_digests()
    my_idx = shard.shard_indices(world * M, rank, world)
    wins_b = [w.encode() for w in synth.windows_parallel_indices(my_idx, WINDOW_LEN)]
    # inputs of the config-4 side measurement (generated here, before CUDA work starts, by the same process pool)
    n4, l4 = 1000, 200000
    wins4_b = [w.encode() for w in synth.windows_parallel(n4, l4)] if (not args.no_secondary and rank == 0 and world == 1) else None
    dec = Decoder(util.blob_bytes(), local)
    stream = torch.cuda.ExternalStream(dec.stream, device=torch.device("cuda", local))

    # ---- a first pass with the block-cyclic deal measures every rank's sweep rate; the windows are then re-dealt in proportion, and once
    # more from the rates of the new deal (a partial last round of warps does not shrink in proportion to the window count) ----
    dec.stage(wins_b)
    have = dict(zip(my_idx, wins_b))
    deal = [list(range(r, world * M, world)) for r in range(world)]
    rate0 = None
    for it in range(1 if (args.no_balance or world == 1) else 2):
        dec.run_staged(); dec.run_staged()
        torch.cuda.synchronize()
        dec.fetch_staged()
        rates = per_rank(len(wins_b) / max(dec.last_sweep_ms, 1e-3))
        if rate0 is None:
            rate0 = rates
        new_deal = deal if args.no_balance else deal_windows(world, M, [float(x) for x in args.assume_rates.split(",")] if (args.assume_rates and it == 0) else rates)
        if new_deal == deal:
            break
        deal = new_deal
        if deal[rank] != my_idx:
            extra = [g for g in deal[rank] if g not in have]
            have.update(zip(extra, (w.encode() for w in synth.windows_parallel_indices(extra, WINDOW_LEN))))
            my_idx = deal[rank]
            wins_b = [have[g] for g in my_idx]
            dec.stage(wins_b)
    if rate0 is None:
        dec.run_staged(); torch.cuda.synchronize(); dec.fetch_staged()
        rate0 = per_rank(len(wins_b) / max(dec.last_sweep_ms, 1e-3))
    del have
    counts = [len(d) for d in deal]
    bases_mine = len(wins_b) * WINDOW_LEN
    bases_all = world * M * WINDOW_LEN

    # ---- device-resident throughput: inputs staged in HBM, K timed steps ----
    for _ in range(args.warmup):
        dec.run_staged()
    barrier()
    sampler = ClockSampler(local); sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 0
    e0.record(stream)
    for _ in range(args.steps):
        dec.run_staged()
        launches += dec.last_launch_count
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    paths = dec.fetch_staged()
    sweep_ms = dec.last_sweep_ms            # last run's sweep kernel, CUDA events around that launch
    assert all(p.status == 0 for p in paths)
    verified = verify_paths(lambda k: paths[k].as_tuples(), my_idx, digests)
    if args.dump_outputs:
        dump_paths(args.dump_outputs, my_idx, paths, DUMP_BYTES // world, "rank%d_" % rank if world > 1 else "")
    # ---- end-to-end through the public call, host buffers in, host paths out ----
    # untimed warm-up of the public call at full size (pinned + device buffers reach their final size; NCCL sets up its gather)
    raw = dec.decode_batch_raw(wins_b)
    if world > 1:
        shard.gather_to_rank0(shard.pack_paths(*raw), device="cuda")
    barrier()
    t0 = time.perf_counter()
    e2e_steps = args.steps
    d2h = 0
    for _ in range(e2e_steps):
        raw = dec.decode_batch_raw(wins_b)
        n_st, status, logp, offset, pb, pe, pt, ptr = raw
        assert not status.any()
        d2h = pb.nbytes + pe.nbytes + pt.nbytes + ptr.nbytes + 32 * len(n_st)
        if world > 1:   # the one gather of the final results (path arrays) over NCCL
            got = shard.gather_to_rank0(shard.pack_paths(*raw), device="cuda")
            if rank == 0:
                assert sum(int(v[0]) for v in got) == world * M
    barrier()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    sampler.stop_flag = True; sampler.join(timeout=2)
    verified_e2e = verify_paths(lambda k: raw_tuples(raw, k), my_idx, digests)

    ms, e2e_s = allmax([ms, e2e_s])
    sweep_all = per_rank(sweep_ms)
    ver_all = allsum([verified, verified_e2e])
    clk = sampler.summary()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    c = allmax([-(clk["sm_mhz"] or 0)] + [1.0 if n in clk["reasons"] else 0.0 for n in names])
    sms = per_rank(props.multi_processor_count)
    if world > 1:
        clk["sm_mhz"] = int(-c[0]); clk["reasons"] = [n for n, v in zip(names, c[1:]) if v > 0]
    clk["per_rank_sweep_ms"] = [round(x, 1) for x in sweep_all]
    sec3 = None
    if not args.no_secondary:
        dec.close()
        try:
            sec3 = config3()
        except Exception as ex:
            sec3 = {"error": repr(ex)}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    ms_per_step = ms / args.steps
    value = bases_all / 1e6 / (ms_per_step / 1e3)
    peak, how = peaks()
    achieved = ALG_BYTES["vit47"] * bases_mine / (sweep_ms / 1e3) / 1e9
    traffic = None
    try:   # DRAM bytes of the sweep kernel from the committed ncu --set full capture (per base, scaled to this launch)
        prof = json.load(open(os.path.join(ROOT, "profiles", "r2_sweep_592win.json")))
        traffic = prof["dram_bytes_per_base"] * bases_mine
    except Exception:
        try:
            prof = json.load(open(os.path.join(ROOT, "profiles", "r1_sweep_2368win_final.json")))
            traffic = prof["dram_bytes_per_base"] * bases_mine
        except Exception:
            pass
    line = {
        "metric": METRIC, "value": value, "unit": "Mbp/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int64 (Q23.40 fixed-point log scores)", "data": "synthetic",
        "config": {"workload": "%d synthetic 50 kb human-composition windows per GPU (%d in all), --species=human ab initio, 47 states (BASELINE.json configs[1])" % (M, world * M),
                   "window_len": WINDOW_LEN, "windows_per_gpu": counts,
                   "parallelism": "%d windows dealt to %d GPU(s) in proportion to each GPU's measured sweep rate, one warp per window" % (world * M, world),
                   "l2": "inputs per step (%.0f MB DNA + %.0f GB of per-window workspace written and read by the kernels) exceed the 126 MB L2" % (bases_mine / 1e6, bases_mine * 332 / 1e9)},
        "e2e": {"value": bases_all / 1e6 / e2e_s, "unit": "Mbp/s", "h2d_bytes_per_step": bases_mine, "d2h_bytes_per_step": int(d2h), "steps": e2e_steps},
        "gpu_launches": int(launches),
        "verified": int(ver_all[0]), "verified_e2e": int(ver_all[1]),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "kernel": "k_sweep", "peak_source": how,
                     "note": "achieved = 940 B/base (dense S=47 figure, SURVEY.md 8d) x rank 0's bases / its sweep-kernel time (CUDA events around the sweep launches of the last step); "
                             "traffic = ncu dram bytes/base of the committed capture x bases; the sweep stores only non-zero cells and is bound by instruction delivery "
                             "(GPC instruction cache at > 90 % of its request rate, profiles/), not by HBM"},
        "clocks": clk,
        "sweep_ms": sweep_ms,
        "devices": {"name": props.name, "sm_count_per_rank": [int(x) for x in sms], "first_pass_windows_per_ms_per_rank": [round(x, 1) for x in rate0]},
    }
    if not args.no_cpu_baseline:
        try:
            line["cpu_baseline"] = calibrated_reference()
        except Exception as ex:   # the reference binary did not travel: time the oracle port instead
            orc = util.Oracle(util.blob_bytes())
            t0 = time.perf_counter(); k = 8
            for i in range(k):
                orc.viterbi(wins_b[i].decode())
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": k * WINDOW_LEN / 1e6 / dt, "unit": "Mbp/s", "cores": 1, "kind": "port",
                                    "sample": "%d windows x 50 kb, oracle/ghmm_oracle.c, 1 thread (%s)" % (k, ex)}
    if not args.no_secondary:
        line["secondary"] = {}
        if sec3 is not None:
            if "error" not in sec3 and not args.no_cpu_baseline:
                try:
                    config3_cpu(sec3)
                except Exception as ex:
                    sec3["cpu_baseline"] = {"error": repr(ex)}
            line["secondary"]["config3_chr2L"] = sec3
    if not args.no_secondary and world == 1:
        # BASELINE.json configs[4]: --sample=100 --alternatives-from-sampling=true on 1000 x 50 kb windows (forward + sampling kernels)
        try:
            dec = Decoder(util.blob_bytes(), local)
            n5 = min(1000, len(wins_b))
            dec.decode_batch_sampling_raw(wins_b[:8], 100)
            torch.cuda.synchronize(); t0 = time.perf_counter()
            vit5, samp5 = dec.decode_batch_sampling_raw(wins_b[:n5], 100)
            torch.cuda.synchronize(); dt5 = time.perf_counter() - t0
            assert not samp5[1].any()
            sec = {"workload": "%d x 50 kb windows, --sample=100 --alternatives-from-sampling=true (Viterbi + forward + 99 sampled paths per window), 1 GPU, e2e from host buffers through augb200_decode_batch_sampling" % n5,
                   "value": n5 * WINDOW_LEN / 1e6 / dt5, "unit": "Mbp/s", "sampled_paths": int(len(samp5[0])), "kernel_ms": dec.last_sweep_ms}
            first5, total5 = dec.sample_first_occurrence(n5, 100)
            uniq5 = int((first5 == np.arange(99)[None, :]).sum())
            sec["dedup"] = {"unique_sampled_paths": uniq5, "path_states_all_samples": total5, "path_states_copied_to_host": int(len(samp5[4])),
                            "note": "k_pack_samples finds repeated state paths of a window on the device (SURVEY.md 8f next-1): only first occurrences cross PCIe"}
            if not args.no_cpu_baseline:
                try:
                    sec["cpu_baseline"] = calibrated_reference(n_per_proc=1, extra_args=("--sample=100", "--alternatives-from-sampling=true"))
                except RuntimeError as ex:          # no reference binary in this tree: the GPU measurement above still stands
                    sec["cpu_baseline"] = {"error": repr(ex)}
            line["secondary"]["config5_sampling"] = sec
            dec.close()
        except Exception as ex:
            line["secondary"]["config5_sampling"] = {"error": str(ex)}
        # BASELINE.json configs[3]: --species=human --UTR=on over 1000 x 200 kb windows (71 states: UtrModel next to the coding states)
        try:
            dec4 = Decoder(util.blob_bytes("human_utr"), local)
            dec4.decode_batch_raw(wins4_b[:16])
            torch.cuda.synchronize(); t0 = time.perf_counter()
            out4 = dec4.decode_batch_raw(wins4_b)
            torch.cuda.synchronize(); dt4 = time.perf_counter() - t0
            assert not out4[1].any()
            sec4 = {"workload": "%d x 200 kb synthetic windows, --species=human --UTR=on --softmasking=0 (71 states), 1 GPU, e2e from host buffers through augb200_decode_batch" % n4,
                    "value": n4 * l4 / 1e6 / dt4, "unit": "Mbp/s", "sweep_ms": dec4.last_sweep_ms, "path_states": int(out4[0].sum())}
            if not args.no_cpu_baseline:
                try:
                    sec4["cpu_baseline"] = calibrated_reference(n_per_proc=1, extra_args=("--UTR=on",), window_len=l4)
                except RuntimeError as ex:          # no reference binary in this tree: the GPU measurement above still stands
                    sec4["cpu_baseline"] = {"error": repr(ex)}
            line["secondary"]["config4_utr"] = sec4
            dec4.close()
        except Exception as ex:
            line["secondary"]["config4_utr"] = {"error": repr(ex)}
    if not args.no_secondary and world == 1 and args.dropin_windows >= 0:
        try:
            line["secondary"]["dropin_e2e"] = dropin_leg(args.dropin_windows)
        except Exception as ex:
            line["secondary"]["dropin_e2e"] = {"error": repr(ex)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
