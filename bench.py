#!/usr/bin/env python
"""Benchmark of the create_mega_reads hot path (BASELINE.json metric: PacBio bases aligned/s).

    python bench.py --gpus N --steps K --warmup W [--impl reference]

Workload (config.workload): BASELINE.json configs[1] -- synthetic yeast-size genome (12 Mbp),
super-reads k-unitig K=41, 50x simulated 10 kbp PacBio reads at 12 % error, production flags
(-m 15 --psa-min 13 --stretch-cap 10000 -B 17 -d 0.029 --max-count 5000, -u unitigs).  One step ==
one pass of the whole read set through the hot path, as a sequence of 64-Mbase batches.

  value : device-timed (CUDA events on the library's stream), read batches already resident in HBM,
          every kernel of mr_align_batch_device plus its result download
  e2e   : the same pass through the public host path (mr_align_batch from page-locked host memory:
          H2D + kernels + D2H, then mega-read tiling/printing on the host threads), wall clock
  N > 1 : one process per GPU (torchrun), index replicated, rank r aligns ITS OWN shard of the reads
          (shard r of an N x read set drawn from the same genome: disjoint reads, same size -- weak
          scaling), no collective on the data path; barrier + max over ranks.
  parity : before the line is printed, the records of the reads the CPU reference was run on are
          written by the GPU path and compared with the reference's file (per read, lines sorted;
          reads whose coords hold an exact (rs, re, ql) tie are the reference's own coin flip,
          SURVEY.md 0.7, and counted apart).  A difference on any other read makes the run fail.
  cli   : wall time of the drop-in binary itself (FASTA in -> record file out), next to e2e.
  roofline : seed_lookup_kernel (the largest kernel of the step).  Besides the contract's byte figures
          it carries `random_access`: lookups are random accesses into the index tables, and the ceiling for
          a table of the index's own size is measured in the same run (mr_selftest_random_gather).  With
          tables that fit the L2 the kernel is bound by instruction issue, with larger ones by the rate of
          random DRAM accesses (DESIGN.md section 4).
  --config human : the shape of BASELINE.json configs[3] on the GPUs given (3.1 Gbp genome with repeats,
          more than 2^32 super-read bases = an index of several parts, 15 kbp reads, k = 17); not the
          metric's configuration, reported in DESIGN.md.
  --workload lookup : configs[4], k-mer queries against a 1 Gbp suffix array.
  --dump-outputs DIR : after the timed steps, the coords rows the device-timed path returned in its last step, for a
          fixed, seeded sample of the reads, as DIR/<name>.npy (OutputDump); the inputs are the same from run to run,
          so two builds can be compared output for output.  Not offered for --workload lookup: that microbench
          times one kernel on random queries, and its results are checked against the oracle by the test suite.
"""
import argparse
import ctypes as C
import json
import os
import queue
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# the committed r01 ncu capture of seed_lookup_kernel describes the kernel as it was in round 1: it is no longer
# quoted (traffic, L2 hit rate come from profiles/r02_seed_lookup_summary.json, captured at the default batch size)
SEED_KERNEL_CHANGED = True

WORKLOAD = dict(genome=12_000_000, coverage=50.0, read_len=10000, error=0.12, sr_cov=3.0, repeat_frac=0.0,
                unitig_k=41, seed=43, mer=15, psa_min=13)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--genome", type=int, default=WORKLOAD["genome"])
    ap.add_argument("--coverage", type=float, default=WORKLOAD["coverage"])
    ap.add_argument("--config", default="yeast", choices=["yeast", "human"],
                    help="yeast: BASELINE.json configs[1] (the metric's configuration, default); human: the shape of configs[3] on "
                         "the GPUs given -- 3.1 Gbp genome with 20 %% repeats, > 2^32 super-read bases (an index of several parts), "
                         "15 kbp reads at 15 %% error, a 0.2x slice of reads per GPU unless --coverage is given")
    ap.add_argument("--host-threads", type=int, default=0)
    ap.add_argument("--batch-bases", type=int, default=64 << 20)
    ap.add_argument("--cpu-sample-reads", type=int, default=0, help="reads in the CPU baseline sample (0: auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="mega_reads", choices=["mega_reads", "lookup"],
                    help="lookup: BASELINE.json configs[4] microbench (k-mer queries against a random-text suffix array)")
    ap.add_argument("--fine-mer", type=int, default=0,
                    help="also run the -F fine pass with this mer (not part of the BASELINE metric: off by default)")
    ap.add_argument("--lookup-n", type=float, default=1e9)
    ap.add_argument("--lookup-queries", type=float, default=1e9)
    ap.add_argument("--lookup-k", type=int, default=17)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the rows the device-timed path returned in its last step (a seeded sample of the reads, at most "
                         "64 MB) as DIR/<name>.npy; rank 0's shard when --gpus > 1")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "mega_reads"):
        ap.error("--dump-outputs: only the GPU path of the mega_reads workload")
    return args


def data_files(args):
    """Rank 0 generates the synthetic inputs once; everybody else waits for the done marker."""
    w = dict(WORKLOAD, genome=args.genome, coverage=args.coverage)
    if getattr(args, "config", "yeast") == "human":
        w.update(genome=3_100_000_000 if args.genome == WORKLOAD["genome"] else args.genome,
                 coverage=0.2 if args.coverage == WORKLOAD["coverage"] else args.coverage,
                 read_len=15000, error=0.15, sr_cov=1.4, repeat_frac=0.2, seed=45,
                 mer=17)                       # mega_reads_assemble.sh:10 (MER=17): at 15 a random mer has ~8 chance matches in 8.7 G bases
    tag = "g%d_c%g_s%d_r%g_l%d" % (w["genome"], w["coverage"], w["seed"], w["repeat_frac"], w["read_len"])
    d = os.path.join(os.environ.get("MR_BENCH_DIR", os.path.join(tempfile.gettempdir(), "pacbio_b200_bench")), tag)
    prefix = os.path.join(d, "synth")
    done = prefix + ".done"
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1")) if getattr(args, "gpus", 1) > 1 else 1
    shards = world if getattr(args, "impl", "ours") == "ours" else 1   # rank r aligns shard r; the CPU arm runs on shard 0
    shard_done = lambda i: done if i == 0 else prefix + ".shard%d.done" % i

    def generate(first_shard, nshards):
        gen = os.path.join(ROOT, "pacbio_b200", "tools", "gen_synth")
        if not os.path.exists(gen):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", gen + ".cc", "-o", gen])
        out = subprocess.check_output([gen, "--genome", str(w["genome"]), "--coverage", str(w["coverage"]), "--read-len",
                                       str(w["read_len"]), "--error", str(w["error"]), "--seed", str(w["seed"]),
                                       "--sr-cov", str(w["sr_cov"]), "--repeat-frac", str(w["repeat_frac"]),
                                       "--unitig-k", str(w["unitig_k"]), "--threads", str(min(32, os.cpu_count() or 1)),
                                       "--shards", str(nshards), "--first-shard", str(first_shard), "--prefix", prefix])
        for i in range(first_shard, nshards):           # atomically: the other ranks poll for these files
            with open(shard_done(i) + ".tmp", "w") as f:
                f.write(out.decode())
            os.replace(shard_done(i) + ".tmp", shard_done(i))

    if rank == 0:
        os.makedirs(d, exist_ok=True)
        missing = [i for i in range(shards) if not os.path.exists(shard_done(i))]
        if missing:
            generate(min(missing), shards)
    mine = rank if shards > 1 else 0
    while not (os.path.exists(done) and os.path.exists(shard_done(mine))):
        time.sleep(0.5)
    info = json.loads(open(done).read())
    reads = prefix + ".reads.fa" if mine == 0 else prefix + ".reads.shard%d.fa" % mine
    return w, dict(sr=prefix + ".superreads.fa", reads=reads, reads0=prefix + ".reads.fa", unitigs=prefix + ".unitigs.fa",
                   unitigs_len=prefix + ".unitigs_len.txt", info=info, prefix=prefix, shard=mine)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe):
    ONE `nvidia-smi -lms 200` process per rank, started before the timed region and killed after it.
    (A new nvidia-smi per sample re-initialises NVML over every GPU of the box and forks a process
    that holds gigabytes of page-locked memory, five times a second per rank: at N > 1 that showed
    up as slower host-synchronising phases of the device-timed step.)"""

    def __init__(self, index):
        self.index, self.rows, self.proc, self.path = index, [], None, None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        if os.environ.get("MR_BENCH_NO_CLOCKS"):          # A/B switch: does the sampling itself cost anything?
            return
        try:
            import tempfile
            fd, self.path = tempfile.mkstemp(prefix="mr_clocks_", suffix=".csv")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=fd, stderr=subprocess.DEVNULL)
            os.close(fd)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is not None:
            try:
                self.proc.terminate()
                self.proc.wait(timeout=5)
            except Exception:
                try:
                    self.proc.kill()
                except Exception:
                    pass
            self.proc = None
        if self.path:
            try:
                for line in open(self.path):
                    r = [x.strip() for x in line.strip().split(",")]
                    if len(r) >= 6:
                        self.rows.append(r)
                os.remove(self.path)
            except Exception:
                pass
            self.path = None

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None, "reasons": reasons,
                "samples": len(self.rows)}


ALL_CPUS = sorted(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else []


PINNED = False


def unpin(cmd):
    """The subprocess arms (the reference binary, the drop-in binary) get every core of the box, whatever this rank is
    pinned to: the command is started through taskset.  (Not a preexec_fn: that makes Python fork() this process --
    CUDA context, NCCL threads and all -- and run Python code in the child before the exec.)"""
    if not (PINNED and ALL_CPUS):
        return cmd
    import shutil
    ts = shutil.which("taskset")
    return [ts, "-c", ",".join(map(str, ALL_CPUS))] + cmd if ts else cmd


def pin_rank(local_rank, nranks):
    """One process per GPU on one box: every rank keeps to its own share of the cores, on the NUMA node its GPU hangs
    off when the box says which (pinned host buffers are then allocated there too).  Without it the 8 ranks' threads
    migrate over all 32 cores and half of the host<->device traffic crosses the socket link.  MR_BENCH_PIN=0: off."""
    if nranks <= 1 or not ALL_CPUS or os.environ.get("MR_BENCH_PIN", "1") == "0":
        return None
    node_of = {}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,pci.bus_id", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout
        for line in out.splitlines():
            idx, bus = [x.strip() for x in line.split(",")]
            bus = bus.lower()
            if len(bus.split(":")[0]) == 8:
                bus = bus[4:]                                       # 00000000:1b:00.0 -> 0000:1b:00.0
            try:
                node_of[int(idx)] = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
            except (OSError, ValueError):
                pass
    except Exception:                                               # noqa: BLE001
        pass
    visible = os.environ.get("CUDA_VISIBLE_DEVICES")
    phys = [int(x) for x in visible.split(",")] if visible and all(x.strip().isdigit() for x in visible.split(",")) else list(range(nranks))
    nodes = [node_of.get(phys[r] if r < len(phys) else r, -1) for r in range(nranks)]
    mine = nodes[local_rank]
    cpus = list(ALL_CPUS)
    peers = list(range(nranks))
    if mine >= 0 and all(n >= 0 for n in nodes):
        try:
            node_cpus = []
            for part in open("/sys/devices/system/node/node%d/cpulist" % mine).read().strip().split(","):
                a, _, b = part.partition("-")
                node_cpus += list(range(int(a), int(b or a) + 1))
            node_cpus = [c for c in node_cpus if c in set(ALL_CPUS)]
            if node_cpus:
                cpus, peers = node_cpus, [r for r in range(nranks) if nodes[r] == mine]
        except (OSError, ValueError):
            pass
    k = peers.index(local_rank)
    share = cpus[len(cpus) * k // len(peers): len(cpus) * (k + 1) // len(peers)] or cpus
    os.sched_setaffinity(0, share)
    global PINNED
    PINNED = True
    return {"cpus": "%d-%d" % (share[0], share[-1]) if share == list(range(share[0], share[-1] + 1)) else ",".join(map(str, share)),
            "numa_node": mine}


def dist_setup(n):
    """One process per GPU under torchrun.  NCCL carries only the barrier and the max-over-ranks of
    the timing (MR_BENCH_BACKEND=gloo runs the same plumbing on CPU for the tests)."""
    if n <= 1 or int(os.environ.get("WORLD_SIZE", "1")) <= 1:
        return None
    import torch
    import torch.distributed as dist
    backend = os.environ.get("MR_BENCH_BACKEND", "nccl")
    if backend == "nccl":
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    # NCCL may print its version banner on stdout when the first communicator is created; stdout
    # must carry exactly one JSON line, so the banner is sent to stderr.
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        dist.init_process_group(backend)
        dist.barrier()
        if backend == "nccl":
            torch.cuda.synchronize()
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)
    return dist


def _reduce_device(dist):
    return "cuda" if dist.get_backend() == "nccl" else "cpu"


def barrier(dist):
    if dist is not None:
        dist.barrier()


def max_over_ranks(dist, x):
    if dist is None:
        return x
    import torch
    t = torch.tensor([x], dtype=torch.float64, device=_reduce_device(dist))
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(dist, x):
    if dist is None:
        return x
    import torch
    t = torch.tensor([x], dtype=torch.float64, device=_reduce_device(dist))
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


# --------------------------------------------------------------------------------------------------
# CPU arm: the reference's own create_mega_reads (oracle/_ref) or, if absent, the oracle port
# --------------------------------------------------------------------------------------------------
def write_sample(files, nreads_sample):
    """First nreads_sample records of shard 0 (any FASTA line layout) -> (path, bases, read names)."""
    sample = files["prefix"] + ".sample%d.fa" % nreads_sample
    nb, names = 0, []
    with open(files["reads0"]) as f, open(sample, "w") as g:
        for line in f:
            if line.startswith(">"):
                if len(names) >= nreads_sample:
                    break
                names.append(line[1:].split()[0] if line[1:].split() else "")
            else:
                nb += len(line.rstrip("\r\n"))
            g.write(line)
    return sample, nb, names


def production_flags(w, files, threads):
    """mega_reads_assemble.sh:175-177 with the defaults of mega_reads_assemble_cluster.sh:13-15"""
    return ["-s", "1M", "-m", str(w["mer"]), "--psa-min", str(w["psa_min"]), "--stretch-cap", "10000", "-k",
            str(w["unitig_k"]), "-u", files["unitigs"], "-t", str(threads), "-B", "17", "--max-count", "5000", "-d",
            "0.029", "-r", files["sr"]]


def cpu_run(w, files, nreads_sample, threads):
    """Aligns the first nreads_sample reads of shard 0 on the host cores; returns (bases/s of the
    alignment phase, meta).  The records stay in meta["out"] for the parity gate."""
    sample, nb, names = write_sample(files, nreads_sample)
    ref = os.path.join(ROOT, "oracle", "_ref", "create_mega_reads")
    out = files["prefix"] + ".cpu.out"
    if os.path.exists(ref):
        cmd = [ref] + production_flags(w, files, threads) + ["-p", sample, "-o", out]
        t0 = time.perf_counter()
        r = subprocess.run(unpin(cmd), stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        wall = time.perf_counter() - t0
        if r.returncode != 0:
            raise RuntimeError("reference run failed: " + r.stderr.decode()[-500:])
        align_s = None
        for line in r.stderr.decode().splitlines():        # -DSHOW_TIMING phase lines (global_timer.hpp:7-47)
            if line.startswith("Starting create mega reads ..."):
                align_s = float(line.split("...")[1])
        if align_s is None:
            align_s = wall
        kind = "reference"
    else:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from oracle_lib import Port
        nbp, ti, align_s = Port().run(0, files["sr"], sample, files["unitigs"], out, w["mer"], w["unitig_k"], threads=threads)
        kind = "port"
    return nb / align_s, dict(kind=kind, cores=threads, bases=nb, seconds=align_s, out=out, sample_path=sample, names=names,
                              sample="first %d reads (%d bases) of the workload, alignment phase only" % (len(names), nb))


def reference_arm(args, w, files):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    total_reads = int(files["info"]["reads"])
    v0, m0 = cpu_run(w, files, min(total_reads, 2000), threads)      # sizes the steps (and warms the page cache)
    # the whole read set when a step stays under a minute, else a bounded prefix (~30 s of alignment)
    nreads = args.cpu_sample_reads or (total_reads if files["info"]["read_bases"] / v0 <= 60.0
                                       else int(max(300, min(total_reads, 30.0 * v0 / w["read_len"]))))
    vals = []
    meta = None
    for _ in range(max(0, args.warmup - 1)):
        cpu_run(w, files, max(100, nreads // 10), threads)
    t_all = 0.0
    for _ in range(args.steps):
        v, meta = cpu_run(w, files, nreads, threads)
        vals.append(v)
        t_all += meta["seconds"]
    value = meta["bases"] * args.steps / t_all
    line = {"impl": "reference", "metric": "pacbio_bases_aligned_per_s", "value": value, "unit": "bases/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_all / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64+f64", "data": "synthetic",
            "config": config_dict(args, w), "cpu_baseline": {"value": value, "unit": "bases/s", "cores": meta["cores"],
                                                            "kind": meta["kind"], "sample": meta["sample"]},
            "e2e": {"value": value, "unit": "bases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def config_dict(args, w):
    name = "configs[1]: synthetic yeast-size genome" if getattr(args, "config", "yeast") == "yeast" else \
        "configs[3] shape: synthetic human-size genome (%g%% repeats, %gx super-reads)," % (100 * w["repeat_frac"], w["sr_cov"])
    return {"workload": "%s %d bp, %gx simulated %d bp PacBio reads at %g%% error, "
                        "k=%d, create_mega_reads production flags" % (name, w["genome"], w["coverage"], w["read_len"],
                                                                      100 * w["error"], w["mer"]),
            "genome_bp": w["genome"], "coverage": w["coverage"], "read_len": w["read_len"], "error": w["error"],
            "mer": w["mer"], "psa_min": w["psa_min"], "unitig_k": w["unitig_k"], "batch_bases": args.batch_bases,
            "l2": "inputs larger than L2: a step streams about %d MB of reads per GPU through batches of %d MB (L2: 126 MB)"
                  % (w["genome"] * w["coverage"] / 1e6, args.batch_bases >> 20),
            "parallelism": "reads sharded x%d (rank r aligns shard r of an %dx read set), index replicated" % (args.gpus, args.gpus)}


def parse_records(path):
    """create_mega_reads output -> {read name: sorted tuple of its lines} (record order is free, SURVEY.md 0.7)"""
    recs, cur = {}, None
    with open(path) as f:
        for line in f:
            line = line.rstrip("\n")
            if line.startswith(">"):
                cur = line[1:]
                recs[cur] = []
            elif cur is not None:
                recs[cur].append(line)
    return {k: tuple(sorted(v)) for k, v in recs.items()}


def reads_with_coords_ties(coords_path):
    """Reads whose coords hold an exact (rs, re, ql) tie: the reference orders those by unordered_map pointer
    hash + an unstable sort (create_mega_reads.cc:69-77), so its own record for such a read is a coin flip."""
    ties, cur, seen = set(), None, None
    with open(coords_path) as f:
        for line in f:
            if line.startswith(">"):
                cur, seen = line.split()[1], set()
            else:
                x = line.split()
                key = (x[0], x[1], x[10])
                if key in seen:
                    ties.add(cur)
                seen.add(key)
    return ties


def parity_gate(H, L, tool, host_threads, w, files, meta):
    """GPU records of the reads the CPU arm aligned vs the CPU arm's file (BASELINE.md 3.4)."""
    names = meta["names"]
    want = parse_records(meta["out"])
    # the batches that hold the first len(names) reads of shard 0 (rank 0 loaded shard 0)
    need, nb, have = len(names), int(H.mrh_tool_nbatches(tool)), 0
    import pacbio_b200.api as api
    count = 0
    while count < nb and have < need:
        nr = C.c_uint32()
        H.mrh_tool_batch_starts(tool, count, C.byref(nr))
        have += nr.value
        count += 1
    out = files["prefix"] + ".gpu.sample.out"
    if H.mrh_tool_run_range(tool, host_threads, out.encode(), 0, count) < 0:
        raise RuntimeError(H.mrh_tool_error(tool).decode())
    sample = set(names)
    got = {k: v for k, v in parse_records(out).items() if k in sample}
    diff = sorted(k for k in set(got) | set(want) if got.get(k) != want.get(k))
    ties = set()
    if diff:                                   # which of them are coords ties: our own jf_aligner on the same sample
        jfa = os.path.join(ROOT, "pacbio_b200", "bin", "jf_aligner")
        coords = files["prefix"] + ".gpu.sample.coords"
        cmd = [jfa, "-s", "1M", "-m", str(w["mer"]), "--psa-min", str(w["psa_min"]), "--stretch-cap", "10000", "-k", str(w["unitig_k"]),
               "-l", files["unitigs_len"], "-B", "17", "--max-count", "5000", "-H", "--coords", coords, "-r", files["sr"],
               "-p", meta["sample_path"]]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        if r.returncode == 0:
            ties = reads_with_coords_ties(coords)
    hard = [k for k in diff if k not in ties]
    return {"records": len(want), "records_gpu": len(got), "sample_reads": len(names), "differ": len(diff), "differ_non_tie": len(hard),
            "against": meta["kind"], "examples": hard[:3],
            "how": "records of the first %d reads of shard 0, GPU path (mr_align_batch + host tiling/printing, written to a file) vs "
                   "the CPU arm's file, per read with lines sorted; `differ` counts reads whose coords hold an exact (rs, re, ql) tie, "
                   "where the reference's own record depends on unordered_map order" % len(names)}


def file_sha256(path):
    import hashlib
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for chunk in iter(lambda: f.read(1 << 24), b""):
            h.update(chunk)
    return h.hexdigest()


def cli_run(w, files, total_bases, host_threads, gpus=1):
    """The drop-in binary itself: FASTA in -> record file out, whole process wall clock plus its own phase
    timers (the same stderr lines the reference prints with -DSHOW_TIMING)."""
    exe = os.path.join(ROOT, "pacbio_b200", "bin", "create_mega_reads")
    out = files["prefix"] + ".cli.out"
    cmd = [exe] + production_flags(w, files, host_threads) + ["-p", files["reads"], "-o", out]
    env = dict(os.environ, MR_SHOW_TIMING="1", MR_DEVICES=os.environ.get("LOCAL_RANK", "0"))
    best = None
    for _ in range(2):                           # second run: page cache warm, as for the reference arm
        t0 = time.perf_counter()
        r = subprocess.run(unpin(cmd), env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        wall = time.perf_counter() - t0
        if r.returncode != 0:
            raise RuntimeError("create_mega_reads failed: " + r.stderr.decode()[-300:])
        ph = {}
        for line in r.stderr.decode().splitlines():
            if line.startswith("stage busy seconds"):
                ph["stages"] = line.split(":", 1)[1].strip()
            if line.startswith("Starting ") and "..." in line:
                try:
                    ph[line[9:line.index("...")].strip()] = float(line.split("...")[1].split()[0])
                except ValueError:
                    pass
        cur = {"wall_s": wall, "phases_s": ph, "out_bytes": os.path.getsize(out)}
        if best is None or wall < best["wall_s"]:
            best = cur
    align_s = best["phases_s"].get("create mega reads")
    best["value"] = total_bases / align_s if align_s else None
    best["unit"] = "bases/s"
    best["what"] = ("bin/create_mega_reads <production flags> -p reads.fa -o out, best of 2 runs; value = read bases / its "
                    "'create mega reads' phase (read parsing + alignment + tiling + writing the record file), the phase "
                    "the reference arm times; wall_s is the whole process including super-read parsing and index build")
    if gpus > 1:
        # the product's own sharding (MR_GPUS: one context + index per device, batches dealt to whichever device is
        # free, ordered host gather) on the same file: the record file must not depend on the number of devices
        out_n = files["prefix"] + ".cli.n%d.out" % gpus
        cmd_n = [exe] + production_flags(w, files, os.cpu_count() or host_threads) + ["-p", files["reads"], "-o", out_n]
        env_n = {k: v for k, v in env.items() if k != "MR_DEVICES"}
        env_n["MR_GPUS"] = str(gpus)
        t0 = time.perf_counter()
        r = subprocess.run(unpin(cmd_n), env=env_n, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        wall = time.perf_counter() - t0
        if r.returncode != 0:
            best["multi_gpu"] = {"gpus": gpus, "error": r.stderr.decode()[-300:]}
        else:
            a_s = None
            for line in r.stderr.decode().splitlines():
                if line.startswith("Starting create mega reads ..."):
                    a_s = float(line.split("...")[1].split()[0])
            best["multi_gpu"] = {"gpus": gpus, "wall_s": wall, "value": total_bases / a_s if a_s else None,
                                 "records_equal_to_one_device": file_sha256(out) == file_sha256(out_n),
                                 "what": "MR_GPUS=%d bin/create_mega_reads on the same reads file (one process, reads dealt to "
                                         "the devices, ordered gather), record file compared byte for byte with the 1-device run" % gpus}
        try:
            os.remove(out_n)
        except OSError:
            pass
    try:
        os.remove(out)
    except OSError:
        pass
    return best


# --------------------------------------------------------------------------------------------------
# --dump-outputs
# --------------------------------------------------------------------------------------------------
DUMP_FIELDS = ("rs", "re", "qs", "qe", "nb_mers", "pb_cons", "sr_cons", "pb_cover", "sr_cover", "ql", "sr", "rn", "use_bwd",
               "stretch", "offset", "avg_err", "info_len", "start_node", "end_node", "lstart", "lprev", "lpath", "lunitigs",
               "component")
DUMP_BYTES = 63 << 20                   # array bytes; the .npy headers stay well inside the 64 MB the option promises


def _ranges(start, count):
    """start[i], start[i] + 1, ..., start[i] + count[i] - 1 for every i, one range after the other."""
    return np.repeat(start - (np.cumsum(count) - count), count) + np.arange(int(count.sum()))


class OutputDump:
    """The results of one step, for a fixed sample of the reads: an eighth of them drawn with a fixed seed, or fewer
    (those drawn first) when their rows would pass DUMP_BYTES.  write() leaves in DIR
      read_index.npy             the sampled reads, by position in the read file
      read_rows.npy              coords rows of each sampled read
      <field>.npy                every row field of mr_result_view (DUMP_FIELDS), rows of the sampled reads in read order;
                                 the overlap graph's fields only when the step ran the graph
      kmers_info.npy, bases_info.npy   the info lists of those rows one after the other, info_len entries each
    all float64, which holds every value of these int32 / uint32 / uint8 / double fields exactly.
    put() hands a result over; its rows are copied out on a thread of its own, so the next batch's kernels do not wait
    for the copy, and the result is freed there as soon as they are.  Freeing a result returns its page-locked slab to
    the context's pool; a copy takes about a millisecond of host time and a batch several milliseconds of GPU time, so
    the slab is normally back before the next batch asks for one and the step allocates no new page-locked memory."""

    def __init__(self, nreads, view, free, seed=0):
        self.view, self.free = view, free
        self.draw = np.random.default_rng(seed).permutation(nreads)          # read r is drawn draw[r]-th
        self.pick = np.flatnonzero(self.draw < max(1, nreads // 8))
        self.parts, self.errors = [], []
        self.queue = queue.Queue()
        self.thread = threading.Thread(target=self._drain, daemon=True)
        self.thread.start()

    def put(self, first_read, result):
        """result: what the batch whose first read is first_read returned."""
        self.queue.put((first_read, result))

    def _drain(self):
        while True:
            item = self.queue.get()
            if item is None:
                return
            try:
                if not self.errors:
                    self.parts.append((item[0], self._take(*item)))
            except Exception as e:                               # noqa: BLE001  (raised again by write())
                self.errors.append(e)
            finally:
                self.free(item[1])

    def _take(self, first, result):
        v = self.view(result)
        nr, n = int(v.nreads), int(v.ncoords)
        lo, hi = np.searchsorted(self.pick, [first, first + nr])
        reads = self.pick[lo:hi]
        rc = np.ctypeslib.as_array(v.read_coords, shape=(nr + 1,)).astype(np.int64)
        start, count = rc[reads - first], rc[reads - first + 1] - rc[reads - first]
        part = {"read_index": reads, "read_rows": count}
        if n == 0:
            return dict(part, **{f: np.zeros(0) for f in DUMP_FIELDS + ("kmers_info", "bases_info")})
        rows = _ranges(start, count)
        for f in DUMP_FIELDS:
            if getattr(v, f):
                part[f] = np.ctypeslib.as_array(getattr(v, f), shape=(n,))[rows]
        off = np.ctypeslib.as_array(v.info_off, shape=(n,))[rows].astype(np.int64)
        length = part["info_len"].astype(np.int64)
        at = _ranges(off, length)
        total = int((off + length).max()) if len(at) else 0
        for f in ("kmers_info", "bases_info"):
            part[f] = np.ctypeslib.as_array(getattr(v, f), shape=(total,))[at] if total else np.zeros(0)
        return part

    def write(self, path):
        self.queue.put(None)
        self.thread.join()
        if self.errors:
            raise self.errors[0]
        parts = [p for _, p in sorted(self.parts, key=lambda x: x[0])]
        out = {k: np.concatenate([p[k] for p in parts]).astype(np.float64) for k in parts[0] if all(k in p for p in parts)}
        rows, info = out["read_rows"].astype(np.int64), out["info_len"].astype(np.int64)
        row_fields = [k for k in out if k in DUMP_FIELDS]
        info_of_read = np.bincount(np.repeat(np.arange(len(rows)), rows), weights=info, minlength=len(rows))
        nbytes = 8 * (2 + len(row_fields) * rows + 2 * info_of_read)
        first = np.argsort(self.draw[out["read_index"].astype(np.int64)])
        keep = np.zeros(len(rows), bool)
        keep[first[np.cumsum(nbytes[first]) <= DUMP_BYTES]] = True
        keep_row = np.repeat(keep, rows)
        keep_info = np.repeat(keep_row, info)
        os.makedirs(path, exist_ok=True)
        for k, a in out.items():
            mask = keep if k in ("read_index", "read_rows") else keep_row if k in row_fields else keep_info
            np.save(os.path.join(path, k + ".npy"), a[mask])


# --------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------
def ours(args, w, files):
    import torch
    import pacbio_b200.api as api
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    pinned = pin_rank(local_rank, args.gpus if int(os.environ.get("WORLD_SIZE", "1")) > 1 else 1)
    dist = dist_setup(args.gpus)
    torch.cuda.set_device(local_rank)
    L = api.lib()                                   # raises if the CUDA library is missing
    H = C.CDLL(os.path.join(ROOT, "pacbio_b200", "libmegareads_host.so"))
    H.mrh_tool_create.restype = C.c_void_p
    H.mrh_tool_create.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_uint, C.c_uint, C.c_uint, C.c_int, C.c_char_p, C.c_size_t]
    H.mrh_tool_load_reads.restype = C.c_int64
    H.mrh_tool_load_reads.argtypes = [C.c_void_p, C.c_char_p, C.c_uint64, C.c_uint64]
    H.mrh_tool_run.restype = C.c_int64
    H.mrh_tool_run.argtypes = [C.c_void_p, C.c_uint, C.c_char_p]
    H.mrh_tool_run_range.restype = C.c_int64
    H.mrh_tool_run_range.argtypes = [C.c_void_p, C.c_uint, C.c_char_p, C.c_uint64, C.c_uint64]
    for f in ("mrh_tool_context", "mrh_tool_index", "mrh_tool_params"):
        getattr(H, f).restype = C.c_void_p
        getattr(H, f).argtypes = [C.c_void_p]
    for f in ("mrh_tool_nbatches", "mrh_tool_nreads", "mrh_tool_sr_bases", "mrh_tool_sr_count"):
        getattr(H, f).restype = C.c_uint64
        getattr(H, f).argtypes = [C.c_void_p]
    H.mrh_tool_batch_bases.restype = C.c_void_p
    H.mrh_tool_batch_bases.argtypes = [C.c_void_p, C.c_uint64, api.u64p]
    for f in ("mrh_tool_batch_codes", "mrh_tool_batch_nmask"):
        getattr(H, f).restype = api.u64p
        getattr(H, f).argtypes = [C.c_void_p, C.c_uint64, api.u64p]
    H.mrh_tool_batch_starts.restype = api.u64p
    H.mrh_tool_batch_starts.argtypes = [C.c_void_p, C.c_uint64, api.u32p]
    H.mrh_tool_last_stats.argtypes = [C.c_void_p, api.u64p]
    H.mrh_tool_stage_seconds.argtypes = [C.c_void_p, api.f64p, api.f64p]
    H.mrh_tool_error.restype = C.c_char_p
    H.mrh_tool_error.argtypes = [C.c_void_p]
    H.mrh_tool_destroy.argtypes = [C.c_void_p]

    err = C.create_string_buffer(512)
    t0 = time.perf_counter()
    psa_min = min(args.fine_mer, w["psa_min"]) if args.fine_mer else w["psa_min"]      # create_mega_reads.cc:131-132
    tool = H.mrh_tool_create(files["sr"].encode(), files["unitigs"].encode(), 1, w["mer"], psa_min, w["unitig_k"],
                             local_rank, err, 512)
    if not tool:
        raise RuntimeError("mrh_tool_create: " + err.value.decode())
    index_s = time.perf_counter() - t0
    ctx, idx, params = H.mrh_tool_context(tool), H.mrh_tool_index(tool), H.mrh_tool_params(tool)
    if args.fine_mer:
        C.cast(params, C.POINTER(api.Params)).contents.fine_mer = args.fine_mer
    H.mrh_tool_nstreams.restype = C.c_uint
    H.mrh_tool_nstreams.argtypes = [C.c_void_p]
    H.mrh_tool_stream_context.restype = C.c_void_p
    H.mrh_tool_stream_context.argtypes = [C.c_void_p, C.c_uint]
    nstreams = int(H.mrh_tool_nstreams(tool))      # batches in flight on this GPU (MR_STREAMS, default 1)
    ctxs = [H.mrh_tool_stream_context(tool, s_) for s_ in range(nstreams)]
    names = (C.c_char_p * 32)(); secs = (C.c_double * 32)()
    nt = L.mr_context_timers(ctx, names, secs, 32)
    index_timers = {names[i].decode(): secs[i] for i in range(nt)}
    # index file round trip (SURVEY 8f-3): what a second process pays instead of the build
    index_io = None
    try:
        if H.mrh_tool_sr_bases(tool) > 500_000_000:
            raise RuntimeError("skipped: index of more than 0.5 G super-read bases (tens of GB on disk)")
        path = os.path.join(os.path.dirname(files["sr"]), "index.rank%d.bin" % rank).encode()
        t1 = time.perf_counter()
        if L.mr_index_save(idx, path) != 0:
            raise RuntimeError(L.mr_last_error(ctx).decode())
        t2 = time.perf_counter()
        c2, i2 = C.c_void_p(), C.c_void_p()
        L.mr_context_create(local_rank, C.byref(c2))
        if L.mr_index_load(c2, path, C.byref(i2)) != 0:
            raise RuntimeError(L.mr_last_error(c2).decode())
        t3 = time.perf_counter()
        ok = L.mr_index_checksum(i2) == L.mr_index_checksum(idx)
        index_io = {"file_bytes": os.path.getsize(path), "save_s": t2 - t1, "load_s": t3 - t2, "checksum_matches": bool(ok)}
        L.mr_index_destroy(i2); L.mr_context_destroy(c2)
        os.remove(path)
    except Exception as e:                           # noqa: BLE001
        index_io = {"error": str(e)}
    total_bases = H.mrh_tool_load_reads(tool, files["reads"].encode(), args.batch_bases, 0)
    if total_bases < 0:
        raise RuntimeError(H.mrh_tool_error(tool).decode())
    nbatches = int(H.mrh_tool_nbatches(tool))
    host_threads = args.host_threads or max(1, (len(os.sched_getaffinity(0)) if pinned else (os.cpu_count() or 1) // max(1, args.gpus)))

    # ---- device-resident copies of every batch ------------------------------------------------------
    # (the form a batch travels and is aligned in: 2 bits per base + a non-ACGT mask, mr_pack_reads)
    dev = []
    for i in range(nbatches):
        nc, nm, nr = C.c_uint64(), C.c_uint64(), C.c_uint32()
        pc = H.mrh_tool_batch_codes(tool, i, C.byref(nc))
        pm = H.mrh_tool_batch_nmask(tool, i, C.byref(nm))
        ps = H.mrh_tool_batch_starts(tool, i, C.byref(nr))
        hc = np.ctypeslib.as_array(pc, shape=(nc.value,)).view(np.int64)
        hm = np.ctypeslib.as_array(pm, shape=(nm.value,)).view(np.int64)
        hs = np.ctypeslib.as_array(ps, shape=(nr.value + 1,))
        dev.append((torch.from_numpy(hc).cuda(), torch.from_numpy(hm).cuda(), torch.from_numpy(hs.astype(np.int64)).cuda(), hs.copy(), nr.value))
    stream = torch.cuda.ExternalStream(L.mr_context_stream(ctx))
    first_read = np.cumsum([0] + [d[4] for d in dev])

    phase = {}
    counters = dict(lookups=0, tails=0, hits=0, groups=0, coords=0, lists=0, buckets=0)

    import threading

    def device_lane(lane, collect, errors, dump):
        # one thread per context: batches lane, lane + nstreams, ... (the C call releases the GIL)
        c = ctxs[lane]
        lnames = (C.c_char_p * 32)(); lsecs = (C.c_double * 32)()
        ph, cn = {}, dict(lookups=0, tails=0, hits=0, groups=0, coords=0, lists=0, buckets=0)
        try:
            for b in range(lane, nbatches, nstreams):
                dc, dm, ds, hs, nr = dev[b]
                out = C.c_void_p()
                rc = L.mr_align_batch_device_packed(c, idx, C.cast(params, C.POINTER(api.Params)), C.c_void_p(dc.data_ptr()),
                                                    C.c_void_p(dm.data_ptr()), C.c_void_p(ds.data_ptr()),
                                                    hs.ctypes.data_as(api.u64p), nr, C.byref(out))
                if rc != 0:
                    raise RuntimeError(L.mr_last_error(c).decode())
                if collect:
                    n = L.mr_context_timers(c, lnames, lsecs, 32)
                    for i in range(n):
                        ph[lnames[i].decode()] = ph.get(lnames[i].decode(), 0.0) + lsecs[i]
                    v = api.ResultView()
                    L.mr_result_get(out, C.byref(v))
                    cn["lookups"] += v.n_kmers_looked_up; cn["tails"] += v.n_tail_entries; cn["hits"] += v.n_hits
                    cn["groups"] += v.n_groups; cn["coords"] += v.ncoords; cn["lists"] += v.n_lists; cn["buckets"] += v.n_buckets
                if dump is not None:
                    dump.put(int(first_read[b]), out)
                else:
                    L.mr_result_free(out)
        except Exception as e:                       # noqa: BLE001
            errors.append(e)
        return ph, cn

    def device_step(collect, dump=None):
        errors, results = [], [None] * nstreams
        def run(lane):
            results[lane] = device_lane(lane, collect, errors, dump)
        threads = [threading.Thread(target=run, args=(lane,)) for lane in range(1, nstreams)]
        for t in threads:
            t.start()
        run(0)
        for t in threads:
            t.join()
        if errors:
            raise errors[0]
        for ph, cn in results:
            for k_, v_ in ph.items():
                phase[k_] = phase.get(k_, 0.0) + v_
            for k_, v_ in cn.items():
                counters[k_] += v_

    for _ in range(args.warmup):
        device_step(False)
    torch.cuda.synchronize()
    barrier(dist)
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = sum(L.mr_context_launches(c_) for c_ in ctxs)
    dump = None
    if args.dump_outputs and rank == 0:
        def view(result):
            v = api.ResultView()
            if L.mr_result_get(result, C.byref(v)) != 0:
                raise RuntimeError("mr_result_get failed")
            return v
        dump = OutputDump(int(first_read[-1]), view, L.mr_result_free)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for step in range(args.steps):
        device_step(True, dump if step == args.steps - 1 else None)
    e1.record(stream)
    torch.cuda.synchronize()
    barrier(dist)
    dev_s = e0.elapsed_time(e1) * 1e-3
    launches = sum(L.mr_context_launches(c_) for c_ in ctxs) - launches0
    dev_s_max = max_over_ranks(dist, dev_s)
    job_bases = sum_over_ranks(dist, float(total_bases))        # every rank aligned its own shard
    value = job_bases * args.steps / dev_s_max

    # ---- end to end through the host path ----------------------------------------------------------------
    for _ in range(args.warmup):
        H.mrh_tool_run(tool, host_threads, None)
    torch.cuda.synchronize()
    barrier(dist)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        if H.mrh_tool_run(tool, host_threads, None) < 0:
            raise RuntimeError(H.mrh_tool_error(tool).decode())
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier(dist)
    sampler.stop()
    e2e_s_max = max_over_ranks(dist, e2e_s)
    stats = (C.c_uint64 * 8)()
    H.mrh_tool_last_stats(tool, stats)
    e2e_value = job_bases * args.steps / e2e_s_max
    st_align, st_format = C.c_double(), C.c_double()
    H.mrh_tool_stage_seconds(tool, C.byref(st_align), C.byref(st_format))
    if dump is not None:
        dump.write(args.dump_outputs)

    # ---- roofline of the dominant kernel ---------------------------------------------------------------
    # Phase timers are CUDA events recorded on the library's own stream around each phase; the
    # "seed lookup" phase is exactly one launch of seed_lookup_kernel per batch.  Algorithmic bytes
    # (DESIGN.md, kernel table): per read base 0.375 B read (2-bit code + mask bit) + 4 B written (list size);
    # per position that keeps a list 16 B written (lookup record); per looked-up k-mer 2 strands x 8 B (the
    # bucket's two bounds in the prefix table); 1 B per tail entry scanned in the tail array.
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    roof = None
    if phase:
        T = total_bases * args.steps
        kern = "seed lookup"
        nparts = int(L.mr_index_parts(idx))           # an index of several parts: every part is probed for every k-mer
        alg = T * 4.375 + counters["lists"] * 16 + counters["lookups"] * 16 * nparts + counters["tails"] * 1
        launches_k = nbatches * args.steps * nparts
        achieved = alg / phase[kern] / 1e9 if phase.get(kern, 0) > 0 else 0.0
        traffic, hit = None, None
        for name in ("r02_seed_lookup_summary.json", "r01_seed_lookup_summary.json"):
            try:                                 # per launch, from the committed ncu --set full capture of THIS configuration
                prof = json.load(open(os.path.join(ROOT, "profiles", name)))
                if prof.get("batch_bases") == args.batch_bases and prof.get("genome") == w["genome"] and \
                   prof.get("kernel", "seed_lookup_kernel") == "seed_lookup_kernel" and (name.startswith("r02") or not SEED_KERNEL_CHANGED):
                    traffic = prof["dram_bytes_per_launch"]
                    hit = prof["l2_sector_hit_rate_pct"] / 100.0
                    break
            except Exception:
                pass
        # The ceiling this kernel lives under (SURVEY.md 8d) is the rate of random DRAM accesses, not bytes:
        # mr_selftest_random_gather (pointer-chase-free 16-byte loads at random places of a 1 GiB table)
        # tops out at ~50 G loads/s on B200 whether a miss fetches 64 or 128 bytes (profiles/
        # r01_gather_probe.txt).  A lookup makes one random access per strand into the prefix table and one
        # more per non-empty bucket into the tail array.
        rnd = None
        try:
            g1, g2 = C.c_double(), C.c_double()
            tbl = int(L.mr_index_table_bytes(idx)) // max(1, nparts)       # prefix table + tails one launch reads at random
            if L.mr_selftest_random_gather(ctx, 1 << 30, 1 << 28, C.byref(g1)) == 0 and \
               L.mr_selftest_random_gather(ctx, tbl, 1 << 28, C.byref(g2)) == 0:
                acc = (2 * counters["lookups"] * nparts + counters["buckets"]) / phase[kern] / 1e9
                rnd = {"peak_G_accesses_per_s": g2.value / 32.0, "peak_table_bytes": tbl,
                       "peak_table": "a table of this index's own size (%d MB; the L2 holds 126 MB)" % (tbl >> 20),
                       "peak_G_accesses_per_s_1GiB_table": g1.value / 32.0,
                       "achieved_G_accesses_per_s": acc, "frac": acc / (g2.value / 32.0),
                       "l2_hit_rate_ncu": hit,
                       "how": "accesses = 2 x looked-up k-mers + non-empty buckets scanned (kernel counters) / CUDA-event time of the "
                              "launches; peak = 2^28 independent random 16-byte loads into a table as large as the index's lookup "
                              "tables, 8 in flight per thread, best of 3 launches, measured in this run; l2_hit_rate_ncu only "
                              "when profiles/ holds a capture of this very configuration"}
        except Exception:
            pass
        roof = {"kernel": "seed_lookup_kernel", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg / launches_k, "avg_launch_ms": 1e3 * phase[kern] / launches_k,
                "share_of_step": phase[kern] / sum(phase.values()),
                "random_access": rnd,
                "dram_gbs_from_traffic": (traffic / (phase[kern] / launches_k) / 1e9) if traffic else None,
                "lookup_table_bytes": int(L.mr_index_table_bytes(idx)), "index_parts": nparts,
                "note": "random gathers into the bucket-bound records and the tail array of the index (lookup_table_bytes over "
                        "index_parts parts).  When those tables fit the L2 (the yeast-size index: l2_hit_rate_ncu 0.88) the kernel "
                        "is bound by instruction issue (ncu: 70 % of the issue slots, 20 of 32 lanes active), so neither frac "
                        "(streaming bytes) nor random_access.frac (L2-resident random accesses) reaches 1; when they do not (the "
                        "human-size index) by the rate of random DRAM accesses (random_access, 1 GiB-table ceiling).  traffic is "
                        "below the algorithmic bytes because the table reads are L2 hits.  With streams_per_gpu > 1 the launch "
                        "runs next to the other stream's kernels, so avg_launch_ms is its duration while sharing the GPU; the "
                        "chaining kernels (phase 'chain coords') are bound by FP64 issue slots and shared-memory latency, see "
                        "DESIGN.md section 4 and profiles/",
                "phases_ms_per_step": {k: 1e3 * v / args.steps for k, v in phase.items()}}

    # ---- CPU baseline + parity gate (rank 0; every N) ----------------------------------------------------
    # The reference binary aligns a bounded prefix of shard 0 on the host cores; the GPU path then writes the
    # records of the very same reads (the batches that hold them) and the two files are compared per read.
    cpu, parity, cli = None, None, None
    if rank == 0 and not args.no_cpu_baseline:
        try:
            n1 = args.cpu_sample_reads or 300
            v1, m1 = cpu_run(w, files, n1, os.cpu_count() or 1)
            if not args.cpu_sample_reads:                       # scale the sample to ~15 s of CPU alignment work
                n2 = int(min(H.mrh_tool_nreads(tool), max(300, 15.0 * v1 / w["read_len"])))
                if n2 > 2 * n1:
                    v1, m1 = cpu_run(w, files, n2, os.cpu_count() or 1)
            cpu = {"value": v1, "unit": "bases/s", "cores": m1["cores"], "kind": m1["kind"], "sample": m1["sample"]}
            parity = parity_gate(H, L, tool, host_threads, w, files, m1)
        except Exception as e:                                  # the baseline is reported, never the measured path
            cpu = {"value": None, "unit": "bases/s", "cores": 0, "kind": "unavailable", "sample": str(e)[:200]}
    if rank == 0 and not os.environ.get("MR_BENCH_NO_CLI"):
        try:
            cli = cli_run(w, files, total_bases, host_threads, args.gpus)
        except Exception as e:                                  # noqa: BLE001
            cli = {"error": str(e)[:300]}

    if rank == 0:
        line = {"metric": "pacbio_bases_aligned_per_s", "value": value, "unit": "bases/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dev_s_max / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64+f64",
                "data": "synthetic", "config": config_dict(args, w),
                "run": {"streams_per_gpu": nstreams, "fine_mer": args.fine_mer, "shard_of_rank0": files["shard"], "rank0_pinned_to": pinned},
                "clocks": sampler.summary(),
                "e2e": {"value": e2e_value, "unit": "bases/s", "h2d_bytes_per_step": int(stats[1]),
                        "d2h_bytes_per_step": int(stats[2]), "ms_per_step": 1e3 * e2e_s_max / args.steps,
                        "host_threads": host_threads, "host_cores": os.cpu_count(), "text_bytes_per_step": int(stats[0]),
                        "stage_busy_ms_last_step": {"mr_align_batch": 1e3 * st_align.value, "host_format": 1e3 * st_format.value},
                        "timing": "wall clock (includes host tiling/printing), max over ranks", "cli": cli},
                "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cpu, "parity": parity,
                "index_build": {"file_round_trip": index_io, "seconds_total": index_s, "parts": int(L.mr_index_parts(idx)), "device_phases_s": index_timers,
                                "superread_bases": int(H.mrh_tool_sr_bases(tool)), "superreads": int(H.mrh_tool_sr_count(tool))},
                "work_per_step": {"read_bases": int(total_bases), "reads": int(H.mrh_tool_nreads(tool)), "batches": nbatches,
                                  "kmers_looked_up": counters["lookups"] // max(1, args.steps),
                                  "positions_with_list": counters["lists"] // max(1, args.steps),
                                  "tail_entries_scanned": counters["tails"] // max(1, args.steps),
                                  "buckets_scanned": counters["buckets"] // max(1, args.steps),
                                  "hits": counters["hits"] // max(1, args.steps), "groups": counters["groups"] // max(1, args.steps),
                                  "coords": counters["coords"] // max(1, args.steps)}}
        print(json.dumps(line))
        sys.stdout.flush()
    H.mrh_tool_destroy(tool)
    if dist is not None:
        dist.destroy_process_group()
    if rank == 0 and parity and parity.get("differ_non_tie", 0) > 0:
        sys.stderr.write("bench.py: PARITY FAILURE: %d records differ from the reference on reads without a coords tie\n"
                         % parity["differ_non_tie"])
        sys.exit(3)


def lookup_microbench(args):
    """configs[4]: queries/s of mr_lookup_batch_device (PSA::search replacement) on a random text of
    --lookup-n bases, half of the queries sampled from the text (both strands), half uniform random."""
    import torch
    import pacbio_b200.api as api
    n, q, k, m = int(args.lookup_n), int(args.lookup_queries), args.lookup_k, 13
    torch.cuda.set_device(0)
    L = api.lib()
    rng = np.random.default_rng(46)
    words = rng.integers(0, 2 ** 63, size=(n + 31) // 32 + 1, dtype=np.int64).astype(np.uint64) * np.uint64(2) + \
        rng.integers(0, 2, size=(n + 31) // 32 + 1, dtype=np.uint64)
    ctx = api.Context(0)

    class _SR:
        pass
    sr = _SR()
    sr.text2bit, sr.n, sr.starts, sr.names = words, n, np.array([0, n], dtype=np.uint64), ["random"]
    sr.unitig_ids, sr.unitig_off = np.zeros(1, np.uint32), np.zeros(2, np.uint64)
    t0 = time.perf_counter()
    idx = api.Index(ctx, sr, m, k)
    build_s = time.perf_counter() - t0
    dwords = torch.from_numpy(words.view(np.int64)).cuda()
    mers = torch.empty(q, dtype=torch.int64, device="cuda")
    chunk = 1 << 27
    g = torch.Generator(device="cuda")
    g.manual_seed(47)
    for lo in range(0, q, chunk):
        c = min(chunk, q - lo)
        half = c // 2
        pos = torch.randint(0, n - k, (half,), device="cuda", generator=g)
        fwd = torch.zeros(half, dtype=torch.int64, device="cuda")
        rc = torch.zeros(half, dtype=torch.int64, device="cuda")
        for j in range(k):
            b = pos + j
            code = (dwords[b >> 5] >> (2 * (b & 31))) & 3
            fwd = (fwd << 2) | code
            rc = rc | ((3 - code) << (2 * j))
        pick = torch.arange(half, device="cuda") & 1
        mers[lo:lo + half] = torch.where(pick == 1, rc, fwd)
        mers[lo + half:lo + c] = torch.randint(0, 4 ** k, (c - half,), device="cuda", generator=g)
        del pos, fwd, rc, pick
    out_i = torch.empty(q, dtype=torch.int64, device="cuda")
    out_n = torch.empty(q, dtype=torch.int64, device="cuda")
    stream = torch.cuda.ExternalStream(ctx.stream())

    def step():
        ctx.check(L.mr_lookup_batch_device(idx.h, C.c_void_p(mers.data_ptr()), q, C.c_void_p(out_i.data_ptr()),
                                           C.c_void_p(out_n.data_ptr())))
    torch.cuda.synchronize()
    for _ in range(args.warmup):
        step()
    ctx.sync()
    sampler = ClockSampler(0)
    sampler.start()
    l0 = ctx.launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    ctx.sync()
    torch.cuda.synchronize()
    sampler.stop()
    dt = e0.elapsed_time(e1) * 1e-3
    found = int((out_n > 0).sum().item())
    # end to end: host buffers in and out through mr_lookup_batch, on a bounded slice of the queries
    qe = min(q, 1 << 26)
    h_m = mers[:qe].cpu().numpy().view(np.uint64)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        idx.lookup(h_m)
    e2e_dt = time.perf_counter() - t0
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    alg = q * (8 + 16 + 8 + 4)          # query in, (index, nb) out, prefix pair, ~one tail
    line = {"metric": "kmer_lookups_per_s", "value": q * args.steps / dt, "unit": "queries/s", "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": "configs[4]: %g k-mer queries (half from the text, both strands; half random) against a "
                                   "%g bp random-text suffix array, k=%d, psa-min %d" % (q, n, k, m),
                       "l2": "index tables and query stream larger than L2"},
            "clocks": sampler.summary(),
            "e2e": {"value": qe * args.steps / e2e_dt, "unit": "queries/s", "h2d_bytes_per_step": qe * 8,
                    "d2h_bytes_per_step": qe * 16, "sample": "%d of the queries through mr_lookup_batch (host pointers)" % qe},
            "gpu_launches": int(ctx.launches() - l0),
            "roofline": {"kernel": "lookup_kernel", "bound": "hbm", "achieved": alg * args.steps / dt / 1e9, "peak": peak,
                         "unit": "GB/s", "frac": alg * args.steps / dt / 1e9 / peak, "traffic": None,
                         "note": "random-sector gathers; algorithmic bytes = 36 per query"},
            "cpu_baseline": None, "index_build_s": build_s, "queries_found": found}
    print(json.dumps(line))
    idx.close()
    ctx.close()


def main():
    # watchdog: a hung run dumps every thread's Python stack on stderr and exits instead of sitting on the GPU
    import faulthandler
    faulthandler.dump_traceback_later(int(os.environ.get("MR_BENCH_WATCHDOG", "900")), exit=True)
    args = parse_args()
    if args.workload == "lookup":
        if args.impl == "reference":
            print(json.dumps({"impl": "reference", "unavailable": "the lookup microbench has no reference arm here "
                              "(building the reference PSA for 1 Gbp takes minutes of CPU); see cpu_baseline of the default workload"}))
            return
        return lookup_microbench(args)
    if args.impl == "reference" and int(os.environ.get("RANK", "0")) != 0:
        return                                   # rank 0 alone runs the CPU arm
    w, files = data_files(args)
    if args.impl == "reference":
        reference_arm(args, w, files)
    else:
        ours(args, w, files)


if __name__ == "__main__":
    main()
