#!/usr/bin/env python
"""bench.py -- SV signatures clustered per second (BASELINE.json metric) on N B200s.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the oracle port on all host cores

A "step" = one pass of the hot path (density filter -> sort -> chain-linkage clustering -> consensus -> genotype)
over one batch of synthetic signature arrays.  N = 1: BASELINE.json configs[1] "synthetic 30x ONT whole-genome
signature arrays, resolution_INS + resolution_DEL on 1xB200" (16 777 216 signatures, 7.75 M reads-table rows,
--genotype).  N > 1: BASELINE.json configs[3]: the SAME genome contig-sharded (LPT) over the N GPUs -- one process
per GPU, csv_set_shard, no data-path collective -- and the step ENDS with csv_allgather (ONE gather of the final
records -- stores into the peers' mail boxes over NVLink, or ONE ncclAllGather with CUTESV_B200_GATHER=nccl -- + the
device merge into the single-GPU order), inside the timed region ("scaling": "strong").
--weak keeps one genome-equivalent per GPU instead.

  value  device-resident throughput (inputs already in HBM), CUDA events on the launching stream, max over ranks
  e2e    the reference-facing call: pinned HOST columns in, host records out (H2D + kernels [+ all-gather] + D2H
         inside the timed region)
--config 5 adds the extraction leg (csv_extract over an ONT ultra-long shaped CIGAR packet) as `e2e_extract`.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from cutesv_b200 import _abi, synth  # noqa: E402

METRIC = "sv_signatures_clustered_per_sec"
UNIT = "signatures/s"
WORKLOADS = {
    2: "config2: synthetic 30x ONT WGS signature arrays, resolution_INS + resolution_DEL, --genotype",
    3: "config3: synthetic 50x PacBio HiFi, all five SV types (INS/DEL/INV/DUP/TRA) + cal_GL genotyping (TRA from the all-alignments table)",
    4: "config2: synthetic 30x ONT WGS signature arrays, resolution_INS + resolution_DEL, --genotype",
    5: "config5: synthetic 100x ONT ultra-long (deep pile-ups), all five SV types + genotyping",
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scale", type=float, default=1.0, help="workload scale (1.0 = BASELINE config)")
    ap.add_argument("--config", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--weak", action="store_true", help="N > 1: one genome-equivalent of contigs per GPU instead of ONE genome sharded over the GPUs")
    ap.add_argument("--strong", action="store_true", help="(default for N > 1, kept for compatibility)")
    ap.add_argument("--extract-reads", type=int, default=0, help="config 5 extraction leg: alignment records in the CIGAR packet (0 = default)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="--impl b200: write the records of the last timed step to DIR/<name>.npy (see dump_outputs)")
    return ap.parse_args()


def workload(config_id, scale, rank):
    return synth.make_config(config_id, scale, seed=synth.SEED0 + config_id + 1000 * rank)


def algorithmic_bytes(cfg, n_cand):
    """SURVEY.md 8(d): 3 x record per signature (48 B DEL-like, 60 B INS/TRA), 16 B per reads row, 64 B per candidate."""
    per = {"DEL": 48, "DUP": 48, "INV": 48, "INS": 60, "TRA": 60}
    b = sum(per[k] * len(v["chrom"]) for k, v in cfg["sigs"].items())
    return b + 16 * len(cfg["reads"]["chrom"]) + 64 * n_cand


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        threading.Thread.__init__(self, daemon=True)
        self.index = index
        self.rows = []
        self.stop_flag = False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows for i in range(4) if len(r) > 2 + i and r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def cpu_baseline(cfg, params, threads, repeats=1):
    """The oracle port (oracle/cutesv_oracle.c) on the host cores: sort + cluster + genotype."""
    from oracle import oracle_lib
    oracle_lib.lib()
    best = None
    nc = 0
    for _ in range(repeats):
        t0 = time.perf_counter()
        c, g, n = oracle_lib.cluster(params, cfg["lens"], cfg["sigs"], cfg["reads"], n_threads=threads)
        dt = time.perf_counter() - t0
        nc = len(c)
        best = dt if best is None else min(best, dt)
    return cfg["n_sigs"] / best, best, nc


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path = the oracle port (the Python reference cannot
    travel to the GPU box; its tuple/pickle path is ~2 orders of magnitude slower, see BASELINE.md section 3)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = workload(args.config, args.scale, 0)
    params = _abi.default_params(**cfg["params"])
    threads = os.cpu_count() or 1
    budget_s = float(os.environ.get("CUTESV_B200_REF_BUDGET_S", "180"))
    # one full-workload pass doubles as warm-up and as the probe that sizes the per-step sample: the whole run
    # (steps x sample) is kept within ~budget_s seconds by shrinking the sample (same generator, smaller scale)
    _, dt0, _ = cpu_baseline(cfg, params, threads)
    sample_scale = args.scale
    sample = "full workload per step"
    if dt0 * args.steps > budget_s:
        frac = max(budget_s / (dt0 * args.steps), 0.01)
        sample_scale = args.scale * frac
        cfg = workload(args.config, sample_scale, 0)
        params = _abi.default_params(**cfg["params"])
        sample = "%.3f of the workload per step (same generator at scale %.4f; the full pass took %.2f s)" % (frac, sample_scale, dt0)
    times = []
    for _ in range(args.steps):
        _, dt, nc = cpu_baseline(cfg, params, threads)
        times.append(dt)
    total = sum(times)
    value = cfg["n_sigs"] * args.steps / total
    world = max(args.gpus, 1)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * total / args.steps, "higher_is_better": True,
        "scaling": "weak" if (args.weak or world == 1) else "strong",
        "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": WORKLOADS[args.config],
                   "scale": args.scale, "sample_scale": sample_scale, "n_signatures": cfg["n_sigs"],
                   "n_reads": int(len(cfg["reads"]["chrom"])),
                   "note": "CPU arm: rank 0 only, all host cores; per-step sample sized so that the run ends within minutes"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": sample + " (oracle/cutesv_oracle.c, OpenMP over (type, contig))"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


DUMP_BUDGET_BYTES = 64 << 20


def dump_outputs(out_dir, cands, genos, names):
    """What a caller of the timed path receives (csv_fetch, or csv_fetch_gathered for N > 1) as float64 tables, one column
    per record field in dtype order (int32 fields and the float64 QUAL convert exactly): cands.npy (_abi.CAND_DTYPE),
    genos.npy (_abi.GENO_DTYPE), names.npy (supporting read ids) and counts.npy = [candidates, read ids].  The device
    places each candidate's read-id slice wherever an atomic lands it, so the slices are written in candidate order and
    names_off is rewritten to match.  Tables that together exceed 64 MB keep the same fraction of their rows, chosen by
    a fixed seed, in order, so that two builds computing the same records write the same files."""
    os.makedirs(out_dir, exist_ok=True)
    off = cands["names_off"].astype(np.int64)
    cnt = cands["names_cnt"].astype(np.int64)
    new_off = np.cumsum(cnt) - cnt
    names = names[np.repeat(off - new_off, cnt) + np.arange(int(cnt.sum()))]
    cands = cands.copy()
    cands["names_off"] = new_off

    def table(a):
        if a.dtype.names is None:
            return a.astype(np.float64)
        return np.concatenate([a[f].reshape(len(a), *(a.dtype[f].shape or (1,))) for f in a.dtype.names], axis=1).astype(np.float64)
    tables = {"cands": table(cands), "genos": table(genos), "names": table(names)}
    total = sum(t.nbytes for t in tables.values())
    frac = min(1.0, (DUMP_BUDGET_BYTES - 4096) / max(total, 1))   # 4 KB for the .npy headers and counts.npy
    for k, t in tables.items():
        if frac < 1.0:
            keep = int(len(t) * frac)
            t = t[np.sort(np.random.default_rng(0).choice(len(t), keep, replace=False))]
        np.save(os.path.join(out_dir, k + ".npy"), t)
    np.save(os.path.join(out_dir, "counts.npy"), np.array([len(cands), len(names)], dtype=np.float64))


def pinned_copy(torch, cols):
    out = {}
    for k, v in cols.items():
        if v is None:
            out[k] = None
            continue
        t = torch.empty(v.shape, dtype=torch.from_numpy(v[:1].copy()).dtype, pin_memory=True)
        a = t.numpy()
        a[...] = v
        out[k] = a
        out["_t_" + k] = t  # keep the pinned tensor alive
    return out


def strip(d):
    return {k: v for k, v in d.items() if not k.startswith("_t_")}


# ---- per-kernel algorithmic bytes of one step (DESIGN.md section 3): n signatures of the type, S survivors of the density
# filter, M members of kept chain clusters, R reads rows, C candidates, P (read, window) pairs, B histogram buckets ----
def kernel_bytes(name, q):
    n, S, M, R, C, P, B = q["n"], q["S"], q["M"], q["R"], q["C"], q["P"], q["B"]
    rec = 22.0 * M + 64.0 * C + 4.0 * M     # 16 B record (+ 4 B c of INS) per member read, 64 B row + read ids written
    table = {
        "k_indel_hist": 8.0 * n,
        "k_bucket_prefix<1>": 8.0 * B, "k_bucket_prefix<2>": 8.0 * B, "k_bucket_prefix<3>": 8.0 * B, "k_bucket_prefix<4>": 8.0 * B,
        "k_bucket_prefix<5>": 8.0 * B, "k_bucket_prefix<6>": 8.0 * B, "k_bucket_prefix<7>": 8.0 * B, "k_bucket_prefix<8>": 8.0 * B,
        "k_bucket_prefix<0>": 8.0 * B,
        "k_indel_scatter": 8.0 * n + 8.0 * S,
        "k_bucket_fixup": 16.0 * S + 4.0 * B,
        "k_select_heads": 4.0 * S + 36.0 * M,
        # the register kernel takes the clusters of <= 32 members (~85 % of the members), the general kernel the rest
        "k_cluster_small<DEL>": 0.85 * rec, "k_cluster_small<INS>": 0.85 * rec,
        "k_cluster_warp<DEL,keep-all>": 0.15 * rec, "k_cluster_warp<INS,keep-all>": 0.15 * rec,
        "k_cluster_warp<DEL>": rec, "k_cluster_warp<INS>": rec, "k_cluster_warp<INDEL>": rec,
        "k_reads_pass<true>": 17.0 * R, "k_reads_pass<false>": 17.0 * R,
        "k_pairs_test<true>": 48.0 * P, "k_pairs_test<false>": 16.0 * P,
        "k_indel_keys<uint32_t, true>": 20.0 * n,
        "k_indel_keys<uint32_t, false>": 20.0 * n,
        "k_prefilter": 4.0 * n + 8.0 * S,
        "k_rs_onesweep<K, false>": 16.0 * S,
        "k_rs_onesweep<K, true>": 12.0 * S,
    }
    return table.get(name)


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    import torch
    import torch.distributed as dist
    from cutesv_b200 import shard
    from cutesv_b200.engine import Engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    stream = torch.cuda.Stream(device=dev)  # a real (non-default) stream shared by torch events and the library
    torch.cuda.set_stream(stream)

    strong = world > 1 and not args.weak
    cfg = workload(args.config, args.scale, 0 if strong else rank)
    n_contigs = len(cfg["lens"])
    total_genome_sigs = cfg["n_sigs"]
    owned = None
    if strong:  # every rank builds the same seeded genome and keeps its LPT share of the contigs
        owner = shard.lpt_assign(shard.contig_weights(cfg["sigs"], n_contigs), world)
        my_sigs, my_reads, my_index = shard.shard_inputs(cfg["sigs"], cfg["reads"], owner, rank)
        full_reads = cfg["reads"]
        cfg = dict(cfg, sigs=my_sigs, reads=my_reads, n_sigs=int(sum(len(v["chrom"]) for v in my_sigs.values())))
        owned = shard.owned_mask(owner, rank)
    else:
        full_reads = cfg["reads"]
    params = _abi.default_params(**cfg["params"])
    eng = Engine(local, stream=stream.cuda_stream, params=params, contig_lens=cfg["lens"])
    if owned is not None:
        eng.set_shard(owned)
    if world > 1:  # the library's own communicator (csv_comm_init); torch.distributed only ships the id and the timings
        uid = [eng.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        eng.comm_init(uid[0], rank, world)
    sigs_p = {k: pinned_copy(torch, v) for k, v in cfg["sigs"].items()}
    reads_p = pinned_copy(torch, cfg["reads"])
    sigs_h = {k: strip(v) for k, v in sigs_p.items()}
    reads_h = strip(reads_p)
    dev_in = sum(v.nbytes for s in sigs_h.values() for v in s.values() if v is not None) + sum(v.nbytes for v in reads_h.values())
    # e2e inputs: the same rows grouped by contig (as the reference holds them: one list per chromosome, cuteSV:817-857)
    # with row offsets instead of the 4-byte contig column (csv_cluster_host_grouped), in pinned host memory
    sigs_gp = {k: pinned_copy(torch, _abi.group_by_contig(v, n_contigs)) for k, v in cfg["sigs"].items()}
    reads_gp = pinned_copy(torch, _abi.group_by_contig(cfg["reads"], n_contigs))
    sigs_g = {k: strip(v) for k, v in sigs_gp.items()}
    reads_g = strip(reads_gp)
    h2d = sum(v.nbytes for s in sigs_g.values() for v in s.values() if v is not None) + sum(v.nbytes for v in reads_g.values())
    type_mask = sum(1 << _abi.TYPE_IDS[k] for k in cfg["sigs"])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if "TRA" in cfg["sigs"] and cfg["params"].get("genotype"):  # TRA genotyper input: every alignment record in BAM order
        order = np.lexsort((np.arange(len(full_reads["chrom"])), full_reads["start"], full_reads["chrom"]))
        eng.upload_alignments({k: v[order] for k, v in full_reads.items()})

    def step_device():
        eng.cluster_device(type_mask)
        if world > 1:
            eng.allgather()   # pack + ONE ncclAllGather + device merge, asynchronous on the same stream

    # ---------------- device-resident: value ----------------
    eng.upload(sigs_h, reads_h)
    warm = max(args.warmup, 3)
    eng.cluster_device(type_mask)
    n_cand, n_names = eng.counts()      # also validates the inputs / sizes the n**0.5 table before the first gather
    for _ in range(warm):
        step_device()
    gathered = eng.gathered_counts() if world > 1 else (n_cand, n_names)
    sampler = ClockSampler(local)
    sampler.start()
    l0, g0 = eng.launch_count(), eng.graph_replays()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step_device()
    e1.record(stream)
    barrier()
    dev_ms = e0.elapsed_time(e1)
    launches = eng.launch_count() - l0
    replays = eng.graph_replays() - g0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *(eng.fetch_gathered() if world > 1 else eng.fetch()))
    if world > 1:
        gathered = eng.gathered_counts()
    # noise bar: the same K steps timed once more, every step between its own events
    per_step = []
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    evs[0].record(stream)
    for k in range(args.steps):
        step_device()
        evs[k + 1].record(stream)
    barrier()
    per_step = [evs[k].elapsed_time(evs[k + 1]) for k in range(args.steps)]
    # ---------------- per-kernel durations: K steps with the SV-type lanes serialised, every launch between its own events ----
    eng.set_lanes(False)
    eng.set_profiling(True)
    eng.cluster_device(type_mask)
    eng.fetch()
    barrier()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record(stream)
    for _ in range(args.steps):
        eng.cluster_device(type_mask)
    s1.record(stream)
    barrier()
    serial_ms = s0.elapsed_time(s1) / args.steps
    cands, genos, names = eng.fetch()  # also collects the per-stage / per-kernel events
    stages = {k: v / args.steps for k, v in eng.stage_ms().items()}  # events accumulate over the K steps
    ktimes = eng.kernel_times()
    ctrs = eng.counters()
    eng.set_profiling(False)
    eng.set_lanes(True)
    # all-gather alone (N > 1): warmed, between its own events, after a barrier
    allgather_ms, allgather_other_ms, gather_mode, other_mode = 0.0, 0.0, None, None
    if world > 1:
        for _ in range(3):
            eng.allgather()
        barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record(stream)
        for _ in range(10):
            eng.allgather()
        a1.record(stream)
        barrier()
        allgather_ms = a0.elapsed_time(a1) / 10.0
        eng.gathered_counts()
        gather_mode = eng.gather_mode()
        # A/B: the other gather (ncclAllGather <-> peer-to-peer stores), same protocol
        eng.set_gather(gather_mode == "nccl")
        for _ in range(3):
            eng.allgather()
        barrier()
        a0.record(stream)
        for _ in range(10):
            eng.allgather()
        a1.record(stream)
        barrier()
        allgather_other_ms = a0.elapsed_time(a1) / 10.0
        other_mode = eng.gather_mode()
        eng.gathered_counts()
        eng.set_gather(gather_mode != "nccl")

    # ---------------- end to end through the public call: e2e ----------------
    cap_c = max(2 * max(n_cand, gathered[0]) + 1024, 1024)
    cap_n = 2 * max(n_names, gathered[1]) + 1024
    pin = [torch.empty(cap_c * 64, dtype=torch.uint8, pin_memory=True), torch.empty(cap_c * 40, dtype=torch.uint8, pin_memory=True),
           torch.empty(cap_n * 4, dtype=torch.uint8, pin_memory=True)]
    out = (pin[0].numpy().view(_abi.CAND_DTYPE), pin[1].numpy().view(_abi.GENO_DTYPE), pin[2].numpy().view(np.int32))

    def step_e2e():
        if world == 1:
            return eng.cluster(sigs_g, reads_g, type_mask, out=out, grouped=True)   # H2D + kernels + D2H
        eng.upload(sigs_g, reads_g, grouped=True)                                  # H2D (pinned, grouped by contig)
        eng.cluster_device(type_mask)
        eng.allgather()
        return eng.fetch_gathered(out=out)                                         # D2H of the merged records

    for _ in range(warm):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        c2, g2, n2 = step_e2e()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    sampler.stop_flag = True
    sampler.join(timeout=2)
    d2h = c2.nbytes + g2.nbytes + n2.nbytes

    # ---------------- config 5: extraction leg (csv_extract over an ONT ultra-long shaped CIGAR packet) ----------------
    extract = None
    if args.config == 5 and rank == 0:
        extract = extract_leg(torch, eng, args, stream)

    # ---------------- max over ranks ----------------
    t = torch.tensor([dev_ms, e2e_s * 1000.0], device=dev, dtype=torch.float64)
    n_sig_total = torch.tensor([float(cfg["n_sigs"])], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(n_sig_total, op=dist.ReduceOp.SUM)
    dev_ms_max, e2e_ms_max = float(t[0].item()), float(t[1].item())
    total_sigs = float(n_sig_total.item())

    if rank == 0:
        value = total_sigs * args.steps / (dev_ms_max / 1000.0)
        e2e_value = total_sigs * args.steps / (e2e_ms_max / 1000.0)
        peak, peak_src = measured_peak()
        # per-kernel rooflines from THIS run's own events (lanes serialised pass)
        n_sig = cfg["n_sigs"]
        n_types = max(len(cfg["sigs"]), 1)
        lin_total = float(np.sum(np.asarray(cfg["lens"], dtype=np.float64)[owned.astype(bool)] if owned is not None else cfg["lens"]))
        kernels = {}
        for nm, (n_l, ms) in ktimes.items():
            per_launch = n_l / float(args.steps)
            # per-launch quantities: INS/DEL kernels run once per type
            indel = [k for k in ("DEL", "INS") if k in cfg["sigs"]]
            q = dict(n=np.mean([len(cfg["sigs"][k]["chrom"]) for k in indel]) if indel else 0.0,
                     S=np.mean([(ctrs["domain"][k] or len(cfg["sigs"][k]["chrom"])) for k in indel]) if indel else 0.0,   # no density filter: every signature is sorted
                     M=np.mean([ctrs["members"][k] for k in indel]) if indel else 0.0,
                     R=float(len(cfg["reads"]["chrom"])), C=float(n_cand) / n_types, P=float(ctrs["pairs"]), B=lin_total / 256.0)
            nbytes = kernel_bytes(nm, q)
            if nm.startswith("k_rs_") and len(cfg["sigs"]) > len(indel):
                nbytes = None   # launches of very different sizes under one name (INS/DEL passes + the small types' passes): no per-launch figure
            avg_ms = ms / n_l
            kernels[nm] = {"launches_per_step": per_launch, "avg_us": 1e3 * avg_ms, "ms_per_step": ms / args.steps,
                           "algorithmic_bytes_per_launch": nbytes,
                           "achieved": (nbytes / 1e9 / (avg_ms / 1e3)) if nbytes else None,
                           "frac": (nbytes / 1e9 / (avg_ms / 1e3) / peak) if nbytes else None}
        ksum = sum(v["ms_per_step"] for v in kernels.values())
        dom = max(kernels, key=lambda k: kernels[k]["ms_per_step"])
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "r02_traffic.json")
        if os.path.exists(tp):
            try:
                tj = json.load(open(tp))
                if dom in tj.get("kernels", {}) and args.config == tj.get("config") and world == 1 and args.scale == 1.0:
                    traffic, traffic_src = tj["kernels"][dom], tj.get("source")
            except Exception:
                pass
        alg = algorithmic_bytes(cfg, n_cand)
        ps = np.asarray(per_step, dtype=np.float64)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "int32", "data": "synthetic",
            "config": {"workload": WORKLOADS[args.config],
                       "scale": args.scale, "n_signatures": int(total_sigs), "n_signatures_rank0": cfg["n_sigs"],
                       "n_reads_rank0": int(len(cfg["reads"]["chrom"])),
                       "n_candidates_rank0": int(n_cand), "n_candidates_gathered": int(gathered[0]),
                       "parallelism": ("contig-shard x%d: ONE genome, contigs LPT-packed over the GPUs (csv_set_shard), step = pipeline + csv_allgather"
                                       if strong else "contig-shard x%d: one genome-equivalent of contigs per GPU, step = pipeline + csv_allgather"
                                       if world > 1 else "single GPU x%d") % world,
                       "l2": "inputs (%.0f MB/step on rank 0) larger than the 126 MB L2, no explicit flush" % (dev_in / 1e6),
                       "e2e_inputs": "host columns grouped by contig + row offsets (csv_upload_*_grouped), pinned",
                       "allgather_ms_alone": allgather_ms, "allgather_in_step": world > 1, "allgather_mode": gather_mode,
                       "allgather_ms_alone_other_mode": {other_mode: allgather_other_ms} if other_mode else None,
                       "density_filter_survivors": ctrs["domain"], "kept_clusters": ctrs["kept"],
                       "graph_replays_in_timed_region": int(replays)},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": e2e_ms_max / args.steps},
            "gpu_launches": int(launches),
            "clocks": sampler.summary(),
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["achieved"], "peak": peak,
                         "unit": "GB/s", "frac": kernels[dom]["frac"], "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": kernels[dom]["algorithmic_bytes_per_launch"],
                         "avg_us_per_launch": kernels[dom]["avg_us"],
                         "share_of_step": kernels[dom]["ms_per_step"] / max(ksum, 1e-9),
                         "timing": "CUDA events around every launch on its launching stream, K steps with the SV-type lanes serialised "
                                   "(%.4f ms/step; the timed region overlaps the lanes and replays a CUDA graph: %.4f ms/step)" % (serial_ms, dev_ms_max / args.steps),
                         "dominant_by": "largest per-kernel total of this run's own events",
                         "note": "bound by the rate of uncoalesced 4-8 B accesses / instruction issue, not by DRAM bytes (profiles/); roofline_kernels lists every kernel"},
            "roofline_kernels": kernels,
            "roofline_pipeline": {"algorithmic_bytes_per_step": alg, "achieved": alg / 1e9 / (dev_ms_max / args.steps / 1e3), "unit": "GB/s",
                                  "frac": alg / 1e9 / (dev_ms_max / args.steps / 1e3) / peak},
            "stages_ms_per_step": stages,
            "ms_per_step_lanes_serialised": serial_ms,
            "ms_per_step_noise": {"median": float(np.median(ps)), "p10": float(np.percentile(ps, 10)), "p90": float(np.percentile(ps, 90)),
                                  "note": "rank 0, the K steps timed once more, each between its own events"},
        }
        if extract is not None:
            line["e2e_extract"] = extract
        if not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            full = workload(args.config, args.scale, 0) if strong else cfg
            v, dt, nc = cpu_baseline(full, params, threads)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": "full workload (%d signatures), 1 run of oracle/cutesv_oracle.c (%.2f s)" % (full["n_sigs"], dt)}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        eng.close()
        dist.destroy_process_group()


def extract_leg(torch, eng, args, stream):
    """Kernel (a): csv_extract over a vectorised ONT ultra-long shaped packet (1 CIGAR op / 7 bp, 20 % of the reads with
    SA segments).  device = CUDA events around k_extract; e2e = the public call (H2D of the packet + kernel + counters)."""
    n_reads = args.extract_reads or max(int(60000 * args.scale), 2000)
    pk, names, lens = synth.synth_cigar_packet(n_reads, mean_indels=7000, seed=11, sa_frac=0.2)
    from cutesv_b200.engine import Engine
    e2 = Engine(eng.device, params=_abi.default_params(), contig_lens=lens)
    pkp = e2.pin_packet(pk)
    e2.set_profiling(True)
    for _ in range(3):
        r = e2.extract(pkp)
    ms, wall = [], []
    for _ in range(10):
        t0 = time.perf_counter()
        r = e2.extract(pkp)
        wall.append(time.perf_counter() - t0)
        ms.append(e2.stage_ms()["extract"])
    e2.set_profiling(False)
    n_ops = int(len(pk["cigar"]))
    n_sa = int(len(pk["sa"]["chrom"]))
    alg = 4.0 * n_ops + 44.0 * n_reads + 28.0 * n_sa
    peak, _ = measured_peak()
    dev = float(np.median(ms))
    wl = float(np.median(wall))
    h2d = int(pk["cigar"].nbytes + sum(pk[k].nbytes for k in ("chrom", "ref_start", "ref_end", "flag", "mapq", "query_len", "read_id", "cigar_off", "sa_off"))
              + sum(v.nbytes for v in pk["sa"].values()))
    e2.close()
    return {"workload": "ONT ultra-long shaped alignment packet: %d records, %d CIGAR ops, %d SA segments" % (n_reads, n_ops, n_sa),
            "signatures": r["counts"], "device_ms": dev, "cigar_ops_per_s": n_ops / (dev / 1e3),
            "roofline": {"bound": "hbm", "kernel": "k_extract", "achieved": alg / 1e9 / (dev / 1e3), "peak": peak, "unit": "GB/s",
                         "frac": alg / 1e9 / (dev / 1e3) / peak, "algorithmic_bytes_per_launch": alg},
            "e2e_ms": wl * 1e3, "e2e_cigar_ops_per_s": n_ops / wl, "h2d_bytes_per_step": h2d, "h2d_GBs": h2d / 1e9 / wl}


if __name__ == "__main__":
    main()
