#!/usr/bin/env python
"""Benchmark of the per-read simulation hot path (BASELINE.json metric: simulated bases/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload config2] [--batch_reads B]
                    [--dump-outputs DIR]

Workloads = the BASELINE.json configs, built by the SURVEY.md 8(d) generators (tests/synth.py):

  config1  genome, 5 Mb synthetic E. coli-sized reference, guppy FAB49712 model, FASTA, 1000 reads per step
  config2  (default; the config the metric is quoted on) genome, guppy model + dorado_v3.2.1 quality table (the shipped
           guppy model has none, SURVEY.md 8d), FASTQ, 3.09 Gb synthetic reference (24 chromosomes with hg38 lengths)
  config3  transcriptome directRNA (dRNA_Bham1_guppy), 200k-transcript synthetic reference + expression profile, FASTA,
           --no_model_ir
  config4  metagenome, 50 species x 1-3 circular chromosomes of 2-6 Mb, Even abundance, ERR3152364_Even model, FASTQ,
           --chimeric
  config5  genome, dorado kit-v14 model, FASTQ -hp -k 6 --chimeric on the config-2 reference

ONE STEP is one batch of ``--batch_reads`` reads (aligned + unaligned in the model's ratio) = the unit the job is made
of, so bases/sec over K steps is the job's throughput.  Under torchrun every rank simulates its own batch per step (weak
scaling; read ids are disjoint shards) after ONE NCCL broadcast of the reference at init.

Printed JSON line: see the task contract.  ``value`` = bases / device time of the kernels (outputs stay in HBM);
``e2e`` = the same through ns_simulate + ns_fetch into pinned host buffers (D2H inside the timed region);
``roofline`` = emit kernel, 3 algorithmic bytes per base for FASTQ (1 reference byte read + 1 base + 1 quality written),
2 for FASTA; ``cpu_baseline`` / ``--impl reference`` = the oracle port (pure Python, like the reference) in a pool of
worker processes forked ONCE (one per host core, like ``simulator.py -t <cores>``), timed in steady state.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import synth  # noqa: E402  (tests/synth.py: the SURVEY 8d generators)

DATA = os.path.join(ROOT, "nanosim_b200", "data")

WORKLOADS = {
    "config1": dict(mode="genome", model="guppy_fab49712_plusq.npz", fastq=False, chimeric=False, kmer_bias=0, batch=1000,
                    text="genome FASTA, guppy FAB49712 model, 5 Mb synthetic reference (1 chr, i.i.d. ACGT, default_rng(0)), "
                         "1k-read job = one step"),
    "config2": dict(mode="genome", model="guppy_fab49712_plusq.npz", fastq=True, chimeric=False, kmer_bias=0, batch=262144,
                    text="genome FASTQ, guppy FAB49712 model + dorado_v3.2.1 quality table, 3.09 Gb synthetic hg38-sized reference "
                         "(24 chr, i.i.d. ACGT), 10M-read job"),
    "config3": dict(mode="transcriptome", model="drna_bham1_guppy_plusq.npz", fastq=False, chimeric=False, kmer_bias=0, batch=262144,
                    text="transcriptome directRNA FASTA (--no_model_ir), dRNA_Bham1_guppy model, 200k-transcript synthetic reference "
                         "(354 Mb, lengths clip(lognormal(7.3,0.6),300,20000)) + expression profile tpm~lognormal(2,1.5), 5M-read job"),
    "config4": dict(mode="metagenome", model="even_err3152364_v3.2.2.npz", fastq=True, chimeric=True, kmer_bias=0, batch=262144,
                    text="metagenome FASTQ --chimeric, ERR3152364_Even model, 50 species x 1-3 circular chromosomes of 2-6 Mb "
                         "(406 Mb, i.i.d. ACGT), Even abundance, 20M-read job"),
    "config5": dict(mode="genome", model="dorado_kitv14_v3.2.1.npz", fastq=True, chimeric=True, kmer_bias=6, batch=131072,
                    text="genome FASTQ -hp -k 6 --chimeric, dorado kit-v14 v3.2.1 model, 3.09 Gb synthetic hg38-sized reference, "
                         "240M-read job"),
}


def effective_cores():
    """CPUs this process can actually use: the affinity mask, capped by the cgroup CPU quota (cpu.max) of the container."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(round(int(quota) / int(period)))))
    except (OSError, ValueError):
        pass
    return n


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons, sampled every 50 ms from the warm-up on (nvidia-smi itself needs ~0.1 s to
    start, longer than a short timed region); samples are time-stamped and only the ones inside a timed region count."""

    def __init__(self, device):
        self.rows = []
        self.device = device
        self.proc = None
        self.windows = []

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def window(self, t0, t1, label):
        self.windows.append((t0, t1, label))

    def stop(self):
        if self.proc:
            self.proc.terminate()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        inside = [r for t, r in self.rows if any(a <= t <= b + 0.06 for a, b, _ in self.windows)]
        sm = [float(r[0]) for r in inside if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for _, r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = sorted({names[i] for r in inside if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm),
                "windows": "samples inside the timed regions: " + ", ".join("%s %.0f ms" % (lab, 1e3 * (b - a)) for a, b, lab in self.windows)}


# --------------------------------------------------------------------------------------------------------------------
# synthetic references (SURVEY 8d)
# --------------------------------------------------------------------------------------------------------------------
class SynthRef:
    """What a workload's reference looks like on the host side of the C ABI: base bytes (a CUDA tensor for the 3 Gb
    genome, numpy otherwise), chromosome offsets, and the mode's extras."""

    def __init__(self, bases, offsets, names, species=None, chrom_species=None, chrom_circular=None, tpm=None):
        self.bases, self.offsets, self.names = bases, np.ascontiguousarray(offsets, dtype=np.uint64), names
        self.species, self.chrom_species, self.chrom_circular, self.tpm = species, chrom_species, chrom_circular, tpm

    @property
    def max_chrom(self):
        return int(np.diff(self.offsets.astype(np.int64)).max())


def synth_genome_gpu(device, scale=1.0):
    """configs 2 and 5: 24 chromosomes with hg38 lengths, i.i.d. uniform ACGT, generated on the GPU (torch is plumbing)."""
    import torch

    lengths = [max(1000, int(x * scale)) for x in synth.HG38_LENGTHS]
    total = sum(lengths)
    dev = "cuda:%d" % device
    g = torch.Generator(device=dev)
    g.manual_seed(1)
    lut = torch.tensor([65, 67, 71, 84], dtype=torch.uint8, device=dev)
    out = torch.empty(total, dtype=torch.uint8, device=dev)
    step = 1 << 28
    for s in range(0, total, step):
        e = min(total, s + step)
        idx = torch.randint(0, 4, (e - s,), generator=g, device=dev, dtype=torch.uint8)
        out[s:e] = lut[idx.long()]
        del idx
    return SynthRef(out, np.concatenate([[0], np.cumsum(lengths)]), list(synth.HG38_NAMES))


def synth_genome_host(scale=1.0):
    rng = np.random.default_rng(1)
    lengths = [max(1000, int(x * scale)) for x in synth.HG38_LENGTHS]
    bases = np.concatenate([synth.synth_chrom(rng, n) for n in lengths])
    return SynthRef(bases, np.concatenate([[0], np.cumsum(lengths)]), list(synth.HG38_NAMES))


def build_reference(name, device, scale, on_gpu):
    mode = WORKLOADS[name]["mode"]
    if name == "config1":
        (nm, arr), = synth.ecoli5m()
        return SynthRef(arr, [0, len(arr)], [nm])
    if mode == "genome":
        return synth_genome_gpu(device, scale) if on_gpu else synth_genome_host(scale)
    if mode == "transcriptome":
        names, lengths, bases, tpm = synth.config3_transcriptome(max(100, int(200000 * scale)))
        return SynthRef(bases, np.concatenate([[0], np.cumsum(lengths)]), [n.split(".")[0] for n in names], tpm=tpm)
    genomes = synth.config4_metagenome(max(2, int(50 * scale)))
    from nanosim_b200.reference_fasta import MetaReference
    m = MetaReference.from_genomes(genomes)
    return SynthRef(m.bases, m.offsets, m.names, species=m.species, chrom_species=m.chrom_species, chrom_circular=m.chrom_circular)


# --------------------------------------------------------------------------------------------------------------------
# the reference's CPU implementation of the path == the oracle port, in a pool of workers forked once
# --------------------------------------------------------------------------------------------------------------------
class OraclePool:
    """``n_procs`` worker processes forked ONCE from a parent that already holds the reference (as Python strings, like the
    reference's seq_dict) and the parsed model -- the reference's ``-t n_procs`` fan-out (simulator.py:1590-1622) without
    paying the fork, the scipy import and the model parsing again at every step.  A step hands every worker its share of
    reads; the step's time is the wall clock until the last worker has answered."""

    def __init__(self, name, sref, n_procs):
        import multiprocessing as mp

        import scipy.stats  # noqa: F401  (imported before the fork: the oracle needs it for every quality draw)
        from conftest import oracle_model
        from nanosim_b200.model import CompiledModel
        import nanosim_oracle as no

        w = WORKLOADS[name]
        self.w, self.n = w, n_procs
        cm = CompiledModel.load(os.path.join(DATA, w["model"]))
        tmp = tempfile.mkdtemp(prefix="bench_oracle_")
        m = oracle_model(cm, tmp, fastq=w["fastq"], chimeric=w["chimeric"], homopolymer=bool(w["kmer_bias"]), mode=w["mode"])
        host = sref.bases if isinstance(sref.bases, np.ndarray) else sref.bases.cpu().numpy()
        offs = sref.offsets.astype(np.int64)
        seqs = [host[offs[i]:offs[i + 1]].tobytes().decode() for i in range(len(offs) - 1)]
        fastq, chim, kb = w["fastq"], w["chimeric"], (w["kmer_bias"] or None)
        if w["mode"] == "genome":
            oref = no.OracleReference(list(zip(sref.names, seqs)))

            def run(na, nu):
                s1, s2 = no.ReadSink(), no.ReadSink()
                no.simulation_aligned_genome(oref, m, s1, "linear", 50, oref.max_chrom, None, None, kb, fastq, na, False, chim)
                if nu:
                    no.simulation_unaligned(oref, m, s2, "linear", 50, oref.max_chrom, None, None, fastq, nu)
                return s1.records + s2.records
        elif w["mode"] == "transcriptome":
            oref = no.OracleTrxReference(list(zip(sref.names, seqs)), dict(zip(sref.names, sref.tpm.tolist())))

            def run(na, nu):
                s1, s2 = no.ReadSink(), no.ReadSink()
                no.simulation_aligned_transcriptome(oref, m, s1, None, "guppy", na, False, fastq, False, False, False)
                if nu:
                    no.simulation_unaligned_transcriptome(oref, m, s2, 50, oref.max_chrom, fastq, nu)
                return s1.records + s2.records
        else:
            genomes = {}
            for nm, sq, si in zip(sref.names, seqs, sref.chrom_species):
                sp = sref.species[int(si)]
                genomes.setdefault(sp, []).append((nm[len(sp) + 1:], sq))
            oref = no.OracleMetaReference(genomes)
            abun = {sp: 100.0 / len(sref.species) for sp in sref.species}
            infl = {sp: no.inflate_abun(abun, sp, m.abun_inflation) for sp in abun}
            mx = max(oref.max_chrom.values())

            def run(na, nu):
                s1, s2 = no.ReadSink(), no.ReadSink()
                no.simulation_aligned_metagenome(oref, m, s1, abun, infl, 50, mx, None, fastq, na, False, chim)
                if nu:
                    no.simulation_unaligned_meta(oref, m, s2, 50, mx, fastq, nu)
                return s1.records + s2.records
        self.split = m.split_counts
        ctx = mp.get_context("fork")
        self.res = ctx.Queue()
        self.cmd = [ctx.Queue() for _ in range(n_procs)]

        def loop(i):
            import random
            k = 0
            while True:
                job = self.cmd[i].get()
                if job is None:
                    return
                random.seed(1000003 * i + k)
                np.random.seed((1000003 * i + k) % (2 ** 31))
                k += 1
                t0 = time.perf_counter()
                recs = run(*job)
                txt = no.format_records(recs, fastq)        # the reference also formats (and writes) its records
                self.res.put((sum(len(r[1]) for r in recs), len(recs), time.perf_counter() - t0, len(txt)))

        self.procs = [ctx.Process(target=loop, args=(i,), daemon=True) for i in range(n_procs)]
        for p in self.procs:
            p.start()

    def step(self, reads_per_worker):
        na, nu = self.split(reads_per_worker)
        t0 = time.perf_counter()
        for q in self.cmd:
            q.put((na, nu))
        out = [self.res.get() for _ in self.procs]
        wall = time.perf_counter() - t0
        return sum(o[0] for o in out), sum(o[1] for o in out), wall, sum(o[2] for o in out)

    def close(self):
        for q in self.cmd:
            q.put(None)
        for p in self.procs:
            p.join(timeout=10)


# --------------------------------------------------------------------------------------------------------------------
# --dump-outputs: what the kernel-only arm left in a context's buffers after each batch of its last timed step
# --------------------------------------------------------------------------------------------------------------------
DUMP_READS = 1024       # reads sampled per batch (indices drawn with a fixed seed from the batch's read count)
DUMP_BASES = 2048       # bases (and qualities) kept per sampled read: one window at a seeded position inside the read
DUMP_LENGTHS = 1 << 20  # read lengths kept for the first DUMP_LENGTHS reads of a batch (all of them at the default sizes)
READ_COLS = ["seq_len", "head", "tail", "n_pieces", "reversed", "flags", "attempts"]
PIECE_COLS = ["read", "n_ops", "kind", "chrom", "pos", "ref_len", "out_len", "out_rel", "l_new", "ref_req", "ev_n_ops", "polya_len"]


def device_bytes(ptr, n, dev):
    """uint8 tensor over ``n`` bytes of device memory the library owns (no copy)."""
    import torch

    class View:
        __cuda_array_interface__ = {"shape": (int(n),), "typestr": "|u1", "data": (int(ptr), False), "version": 3, "stream": None}
    return torch.as_tensor(View(), device=dev)


def snapshot_batch(eng, info, fastq, dev):
    """Copies on the GPU, before the context runs its next batch, the batch's read and piece records and a window of
    DUMP_BASES bases (and qualities) of DUMP_READS reads picked with a fixed seed.  Bounded work: a few MB."""
    import torch
    from nanosim_b200 import _lib as L

    n, rb = int(info.n_reads), L.READ_DTYPE.itemsize
    buf = eng.device_buffers()
    reads = device_bytes(buf["reads"], n * rb, dev).clone()
    pieces = device_bytes(buf["pieces"], int(info.n_pieces) * L.PIECE_DTYPE.itemsize, dev).clone()
    rng = np.random.default_rng(0)
    idx = np.sort(rng.choice(n, size=min(n, DUMP_READS), replace=False))
    u = rng.random(len(idx))
    ii = torch.from_numpy(idx).to(dev)
    off = reads.view(torch.int64).view(n, rb // 8)[ii, 0]             # NsReadMeta: seq_off (u64), then seq_len (u32)
    ln = reads.view(torch.int32).view(n, rb // 4)[ii, 2].long()
    start = (torch.from_numpy(u).to(dev) * (ln - DUMP_BASES).clamp(min=0)).long()
    col = torch.arange(DUMP_BASES, device=dev)
    inside = col[None, :] < (ln - start)[:, None]
    pos = torch.where(inside, (off + start)[:, None] + col[None, :], 0)
    out = {"idx": idx, "start": start, "reads": reads, "pieces": pieces}
    for key in ("seq", "qual") if fastq else ("seq",):
        b = device_bytes(buf[key], int(info.seq_bytes), dev)
        out[key] = torch.where(inside, b[pos], 0)
    torch.cuda.current_stream(dev).synchronize()      # copies done before the context may overwrite its buffers
    return out


def write_dump(path, snaps, infos):
    """DIR/<kind>_<name>.npy for the aligned and the unaligned batch of the last timed step (float32 / float64):
    info (n_reads, n_pieces, total_bases, seq_bytes), read_len (the first DUMP_LENGTHS reads), sample (read indices),
    reads and pieces (the sampled reads' records without buffer offsets, columns READ_COLS / PIECE_COLS; pieces[:, 0] is
    the row of the read in `sample`), window_start, seq and qual (ASCII codes of each sampled read's window, 0 past the
    read's end).  The edit scripts (ops) are deliberately left out: the bases, qualities and records they produce are
    what a caller compares, and their layout may change between builds that emit the same reads."""
    from nanosim_b200 import _lib as L

    os.makedirs(path, exist_ok=True)
    arrays = {}
    for job, s in sorted(snaps.items()):
        kind = "aligned" if job[0] == L.NS_KIND_ALIGNED else "unaligned"
        info = infos[job]
        reads = s["reads"].cpu().numpy().view(L.READ_DTYPE)
        pieces = s["pieces"].cpu().numpy().view(L.PIECE_DTYPE)
        sel = reads[s["idx"]]
        rows = [(k, p) for k, r in enumerate(sel) for p in pieces[int(r["piece_first"]):int(r["piece_first"]) + int(r["n_pieces"])]]
        arrays[kind + "_info"] = np.array([info.n_reads, info.n_pieces, info.total_bases, info.seq_bytes], dtype=np.float64)
        arrays[kind + "_read_len"] = reads["seq_len"][:DUMP_LENGTHS].astype(np.float64)
        arrays[kind + "_sample"] = s["idx"].astype(np.float64)
        arrays[kind + "_reads"] = np.stack([sel[c].astype(np.float64) for c in READ_COLS], axis=1)
        arrays[kind + "_pieces"] = np.array([[k] + [float(p[c]) for c in PIECE_COLS[1:]] for k, p in rows], dtype=np.float64).reshape(-1, len(PIECE_COLS))
        arrays[kind + "_window_start"] = s["start"].cpu().numpy().astype(np.float64)
        for key in ("seq", "qual"):
            if key in s:
                arrays[kind + "_" + key] = s[key].cpu().numpy().astype(np.float32)
    total = sum(a.nbytes for a in arrays.values())
    assert total <= 64 << 20, "dump of %d bytes exceeds 64 MB" % total
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def cpu_sample_text(name, n_workers, per_worker, wall, worker_s, bases):
    extra = ""
    if WORKLOADS[name]["mode"] == "transcriptome":
        extra = "; the reference's select_nearest_kde2d is O(N) per read in the reads of a worker (N = %d here; at the job's " \
                "5M/%d reads per worker it is ~%dx slower per read)" % (per_worker, n_workers, max(1, 5000000 // n_workers // max(per_worker, 1)))
    return ("pure-Python oracle port of simulator.py (same algorithm as the reference, record formatting included, no file I/O), "
            "%d worker processes forked once, %d reads per worker in steady state, %.1f s wall; per core %.3g bases/s%s"
            % (n_workers, per_worker, wall, bases / max(worker_s, 1e-9), extra))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="config2", choices=sorted(WORKLOADS))
    ap.add_argument("--batch_reads", type=int, default=0, help="reads per step per GPU (0 = the workload's default)")
    ap.add_argument("--ref_scale", type=float, default=1.0, help="scale the synthetic reference (tests only)")
    ap.add_argument("--depth", type=int, default=4, help="overlapped contexts per GPU")
    ap.add_argument("--timeline", default=None, help="write the per-batch phase intervals of the timed steps to this file")
    ap.add_argument("--max_len", type=int, default=0, help="experiments only: cap the read length (-max); 0 = the reference's default")
    ap.add_argument("--cpu_reads", type=int, default=0, help="reads PER WORKER in a CPU-baseline step (0 = auto)")
    ap.add_argument("--cpu_procs", type=int, default=0, help="CPU-baseline worker processes (0 = all host cores)")
    ap.add_argument("--no_cpu_baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a seeded sample of what the kernel-only arm computed in its last step "
                         "(rank 0) to DIR/<name>.npy, for comparing two builds output for output.  The sample is copied "
                         "on the GPU inside the timed region, so the timing of a dump run is not one to compare")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    cores = effective_cores()
    n_procs = args.cpu_procs or cores
    W = WORKLOADS[args.workload]
    batch_reads = args.batch_reads or W["batch"]
    workload = "%s: %s, %d reads per step" % (args.workload, W["text"], batch_reads)
    algo_bytes = 3.0 if W["fastq"] else 2.0

    import torch

    if args.impl == "reference":
        # the reference's CPU implementation of the path == the oracle port (Python, one process per host core)
        if rank != 0:
            return
        sref = build_reference(args.workload, local, args.ref_scale, torch.cuda.is_available())
        pool = OraclePool(args.workload, sref, n_procs)
        del sref
        # a step = a bounded sample: sized from the first (untimed) step so that a timed step takes about 6 s of wall clock
        probe = 16 if W["mode"] != "transcriptome" else 64
        pool.step(probe)
        _, pr_reads, pr_wall, _ = pool.step(probe)
        per_worker = args.cpu_reads or int(min(4000, max(1000, 6.0 * probe / max(pr_wall, 1e-3))))
        vals = []
        for s in range(args.warmup + args.steps):
            bases, nreads, wall, wsum = pool.step(per_worker if s >= args.warmup else max(8, per_worker // 8))
            if s >= args.warmup:
                vals.append((bases, nreads, wall, wsum))
        pool.close()
        tb, tt, tw = sum(v[0] for v in vals), sum(v[2] for v in vals), sum(v[3] for v in vals)
        v = tb / tt
        print(json.dumps({"impl": "reference", "metric": "simulated_bases_per_sec", "value": v, "unit": "bases/s",
                          "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": 1e3 * tt / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                          "config": {"workload": workload},
                          "reads_per_sec": sum(v[1] for v in vals) / tt,
                          "cpu_baseline": {"value": v, "unit": "bases/s", "cores": n_procs, "kind": "port",
                                           "per_core": tb / max(tw, 1e-9), "reads_per_step": per_worker * n_procs,
                                           "sample": cpu_sample_text(args.workload, n_procs, per_worker, tt / max(args.steps, 1), tw, tb) + " per step"},
                          "e2e": {"value": v, "unit": "bases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    from nanosim_b200 import _lib as L
    from nanosim_b200.engine import Engine
    from nanosim_b200.model import CompiledModel, DeviceTables, build_alias

    from nanosim_b200 import hostbind
    all_cpus = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    binding = hostbind.bind_to_gpu_node(local)       # this rank's threads and pinned buffers next to its GPU
    torch.cuda.set_device(local)
    dev = "cuda:%d" % local
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device(dev))

    # ---- init (not timed): reference generated on rank 0, ONE broadcast over NCCL, model tables to HBM
    if rank == 0:
        sref = build_reference(args.workload, local, args.ref_scale, True)
        meta = [sref.offsets, sref.names, sref.species, sref.chrom_species, sref.chrom_circular, sref.tpm]
    else:
        sref, meta = None, [None] * 6
    if world > 1:
        dist.broadcast_object_list(meta, src=0)
    n_bases = int(meta[0][-1])
    if rank == 0:
        ref_t = sref.bases if not isinstance(sref.bases, np.ndarray) else torch.from_numpy(sref.bases).to(dev)
    else:
        ref_t = torch.empty(n_bases, dtype=torch.uint8, device=dev)
        sref = SynthRef(None, *meta)
    if world > 1:
        dist.broadcast(ref_t, src=0)
    torch.cuda.synchronize()
    cm = CompiledModel.load(os.path.join(DATA, W["model"]))
    tables = DeviceTables(cm, fastq=W["fastq"], chimeric=W["chimeric"], homopolymer=bool(W["kmer_bias"]), mode=W["mode"])
    eng = Engine(device=local, seed=20260924)
    eng.set_reference_ptr(ref_t.data_ptr(), n_bases, sref.offsets, chrom_species=sref.chrom_species,
                          chrom_circular=sref.chrom_circular, n_species=len(sref.species) if sref.species else 0)
    keep_host = rank == 0 and world == 1 and not args.no_cpu_baseline          # CPU baseline: N=1 only
    if keep_host and not isinstance(sref.bases, np.ndarray):
        sref.bases = ref_t.cpu().numpy()
    del ref_t
    torch.cuda.empty_cache()
    eng.set_model(tables)
    n_al, n_un = tables.split_counts(batch_reads)
    if W["mode"] == "transcriptome":
        pr, al = build_alias(sref.tpm)
        eng.set_expression(pr, al, np.arange(len(sref.tpm), dtype=np.uint32), None)
    if W["mode"] == "metagenome":
        abun = [100.0 / len(sref.species)] * len(sref.species)
        eng.set_abundance(abun, [1 - (1 - a) * tables.abun_inflation for a in abun] if W["chimeric"] else None)
    eng.configure(fastq=W["fastq"], chimeric=W["chimeric"], kmer_bias=W["kmer_bias"], min_len=50, max_len=min(sref.max_chrom, args.max_len) if args.max_len else sref.max_chrom,
                  metagenome=W["mode"] == "metagenome", transcriptome=W["mode"] == "transcriptome",
                  # the reference's 2-D KDE sample has one row per aligned read of a worker (simulator.py:1072): 5M-read job / cores
                  kde2d_sample=max(1, int(5000000 * n_al / max(batch_reads, 1)) // cores) if W["mode"] == "transcriptome" else 0)
    static = W["mode"] == "metagenome"           # species quotas live in a context: job j -> context j % depth

    total_steps = args.warmup + args.steps
    from nanosim_b200.pipeline import BatchPipeline

    def jobs_for(steps):
        """One step = one batch of the job on this rank: its aligned reads, then its unaligned reads."""
        out = []
        for step in steps:
            if n_al:
                out.append((L.NS_KIND_ALIGNED, (step * world + rank) * n_al, n_al))
            if n_un:
                out.append((L.NS_KIND_UNALIGNED, (step * world + rank) * n_un, n_un))
        return out

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def row(info):
        return (info.total_bases, info.seq_bytes, info.n_reads, info.n_pieces, info.n_launches, info.ms_total,
                info.ms_plan, info.ms_scan, info.ms_script, info.ms_emit, info.ms_setup, info.t_begin_ms, info.t_end_ms)

    # ---- kernel-only arm: outputs stay in HBM.  `depth` contexts (ns_clone) share the reference; the latency-bound tails
    #      of one batch's plan / unaligned kernels overlap the emit kernel of another.  Every step simulates new read ids;
    #      a batch's working set (GBs written + a reference sampled at random) is far larger than the 126 MB L2 (config 1,
    #      a 5 Mb reference and 9 MB of output per step, is the exception: the reference's own tiny case).
    pipe = BatchPipeline(eng, depth=args.depth, fetch=False)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    pipe.warm(jobs_for(range(1)))                   # every context sizes its buffers once (untimed)
    dump = bool(args.dump_outputs) and rank == 0
    dump_jobs = set(jobs_for([args.warmup - 1])) if dump and args.warmup else set()
    snaps, snap_infos = {}, {}

    def keep_snapshot(e, info, job):
        # a context's buffers are overwritten by its next batch: copy what the dump needs before the context moves on
        if job in dump_jobs:
            snaps[job], snap_infos[job] = snapshot_batch(e, info, W["fastq"], dev), info
    # the last warm-up step is snapshotted too (and dropped), so that the copies' device memory is allocated before t0
    pipe.run(jobs_for(range(args.warmup)), static_assign=static, after_simulate=keep_snapshot if dump else None)
    if dump:
        dump_jobs = set(jobs_for([total_steps - 1]))
        snaps.clear()
        snap_infos.clear()
    barrier()
    t0 = time.perf_counter()
    rows = [row(i) for i in pipe.run(jobs_for(range(args.warmup, total_steps)), static_assign=static,
                                     after_simulate=keep_snapshot if dump else None)]
    barrier()
    wall = time.perf_counter() - t0
    clocks.window(t0, t0 + wall, "kernel-only arm")
    pipe.close()
    if dump:
        write_dump(args.dump_outputs, snaps, snap_infos)
    if args.timeline and rank == 0:
        with open(args.timeline, "w") as f:       # phases are back to back on a context's stream: begin + cumulative durations
            f.write("reads\tbegin\tsetup_end\tplan_end\tscan_end\tscript_end\temit_end\n")
            t00 = min(r[11] for r in rows)
            for r in sorted(rows, key=lambda r: r[11]):
                t = r[11] - t00
                cells = [t, t + r[10], t + r[10] + r[6], t + r[10] + r[6] + r[7], t + r[10] + r[6] + r[7] + r[8], r[12] - t00]
                f.write("%d\t%s\n" % (r[2], "\t".join("%.2f" % c for c in cells)))
    bases = sum(r[0] for r in rows)
    dev_ms = max(r[12] for r in rows) - min(r[11] for r in rows)     # device timeline: first batch start -> last batch end
    emit_ms = sum(r[9] for r in rows)
    launches = sum(r[4] for r in rows)
    n_reads_done = sum(r[2] for r in rows)
    stat = torch.tensor([bases, dev_ms, wall * 1e3, n_reads_done], dtype=torch.float64, device=dev)
    if world > 1:
        mx = stat.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = stat.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        total_bases, t_ms, total_reads = float(sm[0]), float(mx[1]), float(sm[3])
    else:
        total_bases, t_ms, total_reads = bases, dev_ms, n_reads_done
    value = total_bases / (t_ms * 1e-3)

    # ---- roofline leg: the dominant kernel timed ALONE.  With several overlapped contexts the CUDA events around a
    #      launch also span the other contexts' kernels sharing the SMs, so the per-kernel durations of the arm above
    #      over-state every kernel; here the same batches run through one context (fresh read ids, same sizes).
    n_roof = max(1, min(args.steps, 3))
    pipe1 = BatchPipeline(eng, depth=1, fetch=False)
    pipe1.run(jobs_for(range(total_steps, total_steps + 1)))
    barrier()
    rows1 = [row(i) for i in pipe1.run(jobs_for(range(total_steps + 1, total_steps + 1 + n_roof)))]
    barrier()
    pipe1.close()
    al1 = [r for r in rows1 if r[2] == n_al]                         # aligned batches -> the emit kernel's big launches
    emit_alone_ms = sum(r[9] for r in al1) / max(len(al1), 1)
    emit_alone_bases = sum(r[0] for r in al1) / max(len(al1), 1)
    plan_alone_ms = sum(r[6] for r in al1) / max(len(al1), 1)
    un1 = [r for r in rows1 if r[2] != n_al]
    total_steps += 1 + n_roof

    # ---- end-to-end arm: the public API (BatchPipeline): ns_simulate + ns_fetch into pinned host buffers every batch
    pipe_e = BatchPipeline(eng, depth=args.depth, fetch=True)
    base_step = total_steps                          # fresh read ids
    e_warm = max(3, args.depth + 1)                  # every context's pinned buffers must have seen an aligned batch
    pipe_e.warm(jobs_for(range(base_step, base_step + 1)))
    pipe_e.run(jobs_for(range(base_step, base_step + e_warm)), static_assign=static)
    barrier()
    t0 = time.perf_counter()
    rows_e = [row(i) for i in pipe_e.run(jobs_for(range(base_step + e_warm, base_step + e_warm + args.steps)), static_assign=static)]
    barrier()
    wall_e = time.perf_counter() - t0
    clocks.window(t0, t0 + wall_e, "end-to-end arm")
    clk = clocks.stop() if rank == 0 else None
    pipe_e.close()
    bases_e = sum(r[0] for r in rows_e)
    # bytes that cross PCIe: qualities as ASCII, bases as 2 bits when the library packs them (ns_fetch) + read / piece metadata
    packed = bool(eng.fetch_packs_bases())
    per_base = (1.25 if packed else 2.0) if W["fastq"] else (0.25 if packed else 1.0)
    d2h = sum((per_base if r[1] >= (1 << 20) else (2.0 if W["fastq"] else 1.0)) * r[1] + 32 * r[2] + 64 * r[3] for r in rows_e) / max(args.steps, 1)
    stat = torch.tensor([bases_e, wall_e], dtype=torch.float64, device=dev)
    if world > 1:
        mx = stat.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = stat.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        e2e_value = float(sm[0]) / float(mx[1])
    else:
        e2e_value = bases_e / wall_e

    if rank != 0:
        return
    peak, peak_src = measured_peak()
    achieved = algo_bytes * emit_alone_bases / (emit_alone_ms * 1e-3) / 1e9
    kernel = "emit_kernel<%s>" % ("FASTQ" if W["fastq"] else "FASTA")
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic_%s.json" % args.workload)   # written by tools/ncu_traffic.py from an ncu --set full capture
    if os.path.exists(tp):
        with open(tp) as f:
            traffic = json.load(f)
    line = {
        "metric": "simulated_bases_per_sec", "value": value, "unit": "bases/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": t_ms / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": workload, "reads_per_step_per_gpu": batch_reads, "aligned_per_step": n_al,
                   "unaligned_per_step": n_un, "l2": "inputs larger than L2 (reference sampled at random, GBs written per step)"
                   if args.workload != "config1" else "config 1 is the reference's tiny case: 5 Mb reference, 9 MB written per step (fits L2)",
                   "contexts_per_gpu": args.depth,
                   "timing": "device timeline (CUDA events vs a common base event): first batch start to last batch end of the K "
                             "timed steps, %d overlapped contexts per GPU, max over ranks" % args.depth},
        "reads_per_sec": total_reads / (t_ms * 1e-3),
        "clocks": clk,
        "e2e": {"value": e2e_value, "unit": "bases/s", "h2d_bytes_per_step": 48, "d2h_bytes_per_step": int(d2h),
                "d2h_gb_per_s_per_gpu": d2h * args.steps / wall_e / 1e9,
                "note": "reference + model are resident in HBM (uploaded once at init); per-step input is the read-id range; the "
                        "timed region ends with ASCII bases + qualities + metadata in pinned host buffers" +
                        (" (bases cross PCIe as 2 bits and are expanded by host threads inside ns_fetch)" if packed else "")},
        "gpu_launches": int(launches),
        "phase_ms_per_step": {"plan": sum(r[6] for r in rows) / args.steps, "scan": sum(r[7] for r in rows) / args.steps,
                              "script": sum(r[8] for r in rows) / args.steps, "emit": emit_ms / args.steps,
                              "setup": sum(r[10] for r in rows) / args.steps,
                              "note": "sums of per-batch CUDA-event durations; batches of the overlapped contexts share the GPU, so these add up to more than ms_per_step"},
        "wall_ms_per_step": 1e3 * wall / max(args.steps, 1),
        "roofline": {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak,
                     "traffic": traffic["dram_bytes_per_launch"] if traffic else None,
                     "traffic_source": traffic["source"] if traffic else "no ncu --set full capture of this workload committed",
                     "peak_source": peak_src,
                     "algorithmic_bytes_per_base": algo_bytes,
                     "bases_per_launch": emit_alone_bases, "ms_per_launch": emit_alone_ms,
                     "plan_kernel_ms_per_launch": plan_alone_ms,
                     "alone_ms": {"aligned_batch_total": sum(r[5] for r in al1) / max(len(al1), 1),
                                  "unaligned_batch_total": sum(r[5] for r in un1) / max(len(un1), 1),
                                  "unaligned_plan": sum(r[6] for r in un1) / max(len(un1), 1),
                                  "unaligned_emit": sum(r[9] for r in un1) / max(len(un1), 1)},
                     "measured": "CUDA events on the launching stream around %s, %d aligned batches of %d reads run "
                                 "through ONE context after the timed region (kernels of overlapped contexts share SMs, which "
                                 "stretches every per-launch duration)" % (kernel, len(al1), n_al),
                     "whole_path_frac": algo_bytes * total_bases / (t_ms * 1e-3) / 1e9 / peak / max(world, 1)},
    }
    if keep_host:
        # ---- to-file arm: the drop-in driver's simulation() (nanosim_b200/simulator.py: names, FASTA/FASTQ records and the
        #      error profile formatted and pwrite()n by library threads) into RAM-backed files, on a bounded number of reads
        import shutil
        from types import SimpleNamespace
        from nanosim_b200 import simulator
        out_dir = tempfile.mkdtemp(prefix="bench_to_file_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
        host_ref = SimpleNamespace(names=list(sref.names), bases=sref.bases, offsets=sref.offsets)
        nthr = max(1, min(32, cores))
        tf = {}
        import contextlib
        try:
            for label, errp, nsteps in (("with_error_profile", True, 2), ("reads_only", False, 4)):
                prof = SimpleNamespace(ref=host_ref, tables=tables, engine=eng, number_aligned=n_al * nsteps, number_unaligned=n_un * nsteps,
                                       seed=20260924, ir=None, n_trx=0)
                t0 = time.perf_counter()
                with contextlib.redirect_stdout(sys.stderr):           # the driver's progress lines are not part of the JSON line
                    tot = simulator.simulation(prof, W["mode"], os.path.join(out_dir, label), "linear", False, W["kmer_bias"] or None, "guppy",
                                               sref.max_chrom, 50, nthr, W["fastq"], chimeric=W["chimeric"], batch_reads=batch_reads,
                                               error_profile=errp)
                dt = time.perf_counter() - t0
                tf[label] = {"value": tot["bases"] / dt, "unit": "bases/s", "reads": tot["reads"], "file_gb": tot["bytes"] / 1e9,
                             "gb_per_s": tot["bytes"] / dt / 1e9, "seconds": dt}
                for fn in os.listdir(out_dir):
                    os.remove(os.path.join(out_dir, fn))
        finally:
            shutil.rmtree(out_dir, ignore_errors=True)
        tf["note"] = "simulator.simulation() of the drop-in CLI writing into %s, %d formatter / writer threads (-t), pipeline depth 2, " \
                     "first batch included" % (os.path.dirname(out_dir), nthr)
        line["to_file"] = tf
    line["host"] = {"cpus": os.cpu_count(), "cpus_allowed": len(all_cpus) if all_cpus else None, "cpus_effective": cores,
                    "note": "cpus_effective = affinity mask capped by the container's cgroup CPU quota (cpu.max)", "numa_binding": binding}
    if keep_host:
        hostbind.unbind(all_cpus)                                # the CPU baseline may use every core of the box
        pool = OraclePool(args.workload, sref, n_procs)
        probe = 16 if W["mode"] != "transcriptome" else 64
        pool.step(probe)                                         # the workers' first call (lazy imports, page faults)
        _, _, pr_wall, _ = pool.step(probe)
        per_worker = args.cpu_reads or int(min(8000, max(1000, 15.0 * probe / max(pr_wall, 1e-3))))      # >= 1000 reads per worker, ~15 s of wall clock
        cb, cr, ct, cw = pool.step(per_worker)
        pool.close()
        line["cpu_baseline"] = {"value": cb / ct, "unit": "bases/s", "cores": n_procs, "kind": "port", "per_core": cb / max(cw, 1e-9),
                                "reads_per_sec": cr / ct,
                                "sample": cpu_sample_text(args.workload, n_procs, per_worker, ct, cw, cb)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
