#!/usr/bin/env python3
"""bench.py — 802.11a 54 Mbps RX PHY throughput (IQ in, bits out) on B200, BASELINE.json's metric.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--frames F] [--impl reference]

A "step" = one pass of the whole RX hot path (carrier sense -> LTS -> OFDM demod -> soft demap -> Viterbi -> descramble
-> CRC) over one batch of F synthetic capture slots (BASELINE config #2: 54 Mbps, PSDU 1500 B, 9824 samples per slot at
40 Msps, AWGN 30 dB).
  value        Msamples/s with the IQ already resident in HBM (device-timed, CUDA events, max over ranks);
  e2e          the same through the C ABI with pinned HOST buffers: H2D of the IQ and D2H of bytes + verdicts inside the timed region.  Three
               documented ways to call it are timed — the whole 40 Msps capture copied as it is; option "host_decimate" (host threads
               gather the even samples TDownSample2 keeps, half the bytes cross PCIe); and the same with "host_decimate_mix" = 1, where the
               library decides per chunk between the two so that link and host cores are both busy — the best is reported (`e2e.mode`);
  mgpu         (N > 1) the partitioning BASELINE.json's north_star names: all N*F slots enter on rank 0's GPU, NCCL scatters the IQ slabs to
               the ranks over NVLink, every rank decodes its slab, NCCL gathers bytes + verdicts back to rank 0; all inside the timed region;
  roofline     dominant kernel (the Viterbi) against the HBM roofline; cpu_baseline: the SSE CPU oracle on the box's host cores in the three
               topologies of SURVEY.md §8(d): one thread, the reference's two-thread pipeline, all cores.
`--impl reference` times that CPU implementation alone.  Before any timing the result of every unique slot is compared field by field
(status, rate, length, FCS, symbol count, detect index, CFO estimate, bytes) with the CPU oracle on the same IQ.
`--dump-outputs DIR` writes what the last timed step computed (rank 0's verdicts and PSDU bytes of a fixed, seeded sample of slots) to
DIR/<name>.npy; the input is seeded, so two builds run with the same arguments can be compared output for output.
Multi-GPU (torchrun): slots are independent, so every rank decodes its own F slots (weak scaling, no data-path collective in `value` / `e2e`).
"""
import argparse, json, os, re, subprocess, sys, time, threading
import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the tree as it found it (it may be read-only)

SLOT = 9824            # 9760 samples of PPDU + 64 zero samples of gap (32 before, 32 after)
PSDU = 1500
RATE = 54000
ALG_BYTES_PER_SAMPLE = 4.0 + (PSDU + 16) / SLOT      # SURVEY.md §8(d): 4 B in per sample + (PSDU + 16 B status) out per slot
METRIC = "802.11a RX PHY Msamples/s (IQ in, bits out)"
WORKLOAD = "802.11a 54 Mbps RX chain, synthetic 20 MHz IQ @40 Msps, PSDU 1500 B, AWGN 30 dB, one frame per 9824-sample slot (BASELINE config #2)"

def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"

# ---- host description: what this process may really use ------------------------------------------------------------------------------------
def effective_cpus():
    """CPUs this process can use: scheduler affinity capped by the cgroup CPU quota (os.cpu_count() ignores both)."""
    try: aff = len(os.sched_getaffinity(0))
    except Exception: aff = os.cpu_count() or 1
    quota = None
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]                    # cgroup v2
        if q != "max": quota = float(q) / float(p)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())   # cgroup v1
            if q > 0: quota = q / p
        except Exception: pass
    n = aff if quota is None else max(1, min(aff, int(quota)))
    return n, {"os_cpu_count": os.cpu_count(), "affinity": aff, "cgroup_quota_cpus": quota}

def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"): return line.split(":", 1)[1].strip()
    except Exception: pass
    return "unknown"

def numa_bind(local):
    """Pin this rank to the CPUs of its GPU's NUMA node (pinned staging memory is then allocated there as well).  Returns a description."""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=pci.bus_id", "--format=csv,noheader"], capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if bus.startswith("00000000:"): bus = bus[4:]
        p = f"/sys/bus/pci/devices/{bus}/local_cpulist"
        cpus = set()
        for part in open(p).read().strip().split(","):
            a, _, b = part.partition("-"); cpus.update(range(int(a), int(b or a) + 1))
        cur = os.sched_getaffinity(0); new = cur & cpus
        if new and new != cur:
            os.sched_setaffinity(0, new)
            node = open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip()
            return f"gpu {local} ({bus}) -> numa node {node}, {len(new)} cpus"
        return f"gpu {local} ({bus}): affinity left as is ({len(cur)} cpus)"
    except Exception as e:
        return f"not bound ({type(e).__name__})"

class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms (B200_PROFILING.md recipe).  The process is started before the warm-up
    (nvidia-smi needs up to a second before its first line) and every line is stamped on arrival; stop() keeps the lines that arrived
    between mark() and stop(), i.e. under the load of the timed steps."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    def __init__(self, index):
        self.rows = []; self.p = None; self.index = index; self.t0 = None
    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.p = None
    def _read(self):
        for line in self.p.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))
    def mark(self):
        self.t0 = time.perf_counter()
    def seen(self):
        return sum(1 for t, _ in self.rows if self.t0 is not None and t >= self.t0)
    def stop(self):
        if self.p:
            self.p.terminate()
            try: self.p.wait(timeout=2)
            except Exception: pass
        rows = [r for t, r in self.rows if self.t0 is None or t >= self.t0]
        sm = [float(r[0]) for r in rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            if len(r) >= 7:
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"): reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}

def make_input(nframes, unique):
    from sora_b200 import synth
    unique = min(unique, nframes)
    iq, ps = synth.make_frames(unique, psdu_len=PSDU, rate_kbps=RATE, snr_db=30.0, lead=32, trail=32)
    assert iq.shape[1] == SLOT, iq.shape
    return iq, ps, unique

# ---- CPU arm: the SSE oracle (oracle/, kind "port": the MSVC-only reference cannot be compiled here) ------------------------------------------
def cpu_run(iq_unique, nframes, nthreads, topology="independent"):
    """`nframes` slots of the workload on the host: `independent` = nthreads threads over independent slots (each thread runs the whole
    chain), `two_thread` = nthreads // 2 pipelines of the reference's front-end thread | Viterbi thread pair.  Returns (seconds, FRAME_OK count)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_py
    U = iq_unique.shape[0]
    flat = iq_unique.reshape(-1, 2)
    off = (np.arange(nframes, dtype=np.uint64) % U) * SLOT
    ln = np.full(nframes, SLOT, np.uint32)
    t = time.perf_counter()
    if topology == "two_thread": res, _ = oracle_py.rx11a_batch_2t(flat, off, ln, out_stride=PSDU, npipes=max(1, nthreads // 2))
    else: res, _ = oracle_py.rx11a_batch(flat, off, ln, out_stride=PSDU, nthreads=nthreads)
    dt = time.perf_counter() - t
    return dt, int((res["status"] == 1).sum())

def cpu_baseline(iq_u, ncores, budget_s=18.0):
    """SURVEY.md §8(d): (i) one thread, (ii) the reference topology (front end | Viterbi on two threads), (iii) all cores; each on a bounded
    sample sized from a calibration run so that the whole baseline stays within `budget_s` seconds of CPU wall time."""
    cpu_run(iq_u, 16, 1)                                                        # warm the tables
    dt1, _ = cpu_run(iq_u, 32, 1); per1 = dt1 / 32
    share = budget_s / 4.0
    out = {}
    n = int(max(16, min(4096, share / per1)))
    dt, ok = cpu_run(iq_u, n, 1)
    out["one_thread"] = {"value": n * SLOT / dt / 1e6, "threads": 1, "slots": n, "seconds": round(dt, 2)}
    n = int(max(16, min(8192, 1.6 * share / per1)))
    dt, ok = cpu_run(iq_u, n, 2, "two_thread")
    out["reference_two_thread"] = {"value": n * SLOT / dt / 1e6, "threads": 2, "slots": n, "seconds": round(dt, 2)}
    n = int(max(64, min(65536, 0.7 * ncores * share / per1)))
    dt, ok = cpu_run(iq_u, n, ncores)
    out["all_cores_independent"] = {"value": n * SLOT / dt / 1e6, "threads": ncores, "slots": n, "seconds": round(dt, 2)}
    if ncores >= 2:
        dt2, _ = cpu_run(iq_u, n, ncores, "two_thread")
        out["all_cores_two_thread_pipelines"] = {"value": n * SLOT / dt2 / 1e6, "threads": ncores // 2 * 2, "slots": n, "seconds": round(dt2, 2)}
    best = max(("all_cores_independent", "all_cores_two_thread_pipelines"), key=lambda k: out.get(k, {"value": 0})["value"])
    return out, best

def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ncores, how = effective_cpus()
    iq, _, U = make_input(256, 256)
    cpu_run(iq, 64, ncores)                               # warm the tables / threads
    # size the per-step sample so the whole run stays within minutes: calibrate on 256 slots
    dt, _ = cpu_run(iq, 256, ncores)
    per_step = int(max(256, min(16384, 256 * (8.0 / max(dt, 1e-3)) / max(1, args.steps))))
    for _ in range(args.warmup): cpu_run(iq, min(per_step, 512), ncores)
    t_tot = 0.0; okc = 0
    for _ in range(args.steps):
        dt, ok = cpu_run(iq, per_step, ncores); t_tot += dt; okc += ok
    val = per_step * args.steps * SLOT / t_tot / 1e6
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "Msamples/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int16 (fixed point)", "data": "synthetic",
            "config": {"workload": WORKLOAD, "slots_per_step": per_step, "psdu_bytes": PSDU, "samples_per_slot": SLOT},
            "cpu_baseline": {"value": val, "unit": "Msamples/s", "cores": ncores, "kind": "port", "cpu_model": cpu_model(), "cores_how": how,
                             "sample": f"{per_step} slots/step x {args.steps} steps, {ncores} host threads over independent slots (oracle/ SSE restatement; MSVC-only reference is unbuildable here)"},
            "e2e": {"value": val, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "frames_ok_fraction": okc / float(per_step * args.steps)}
    print(json.dumps(line))

def brick_leg(iq_u, nframes=256, instances=16):
    """The BRICK path end to end: sora_b200/brick/demo_graph (TMemSamples -> TB200Dot11aRx -> sink, driven like RxThread) over a dump file of
    `nframes` frames, `instances` graph instances in as many threads (K radios); host samples in, events out, engine shared, windows batched."""
    import tempfile
    from sora_b200.dumpfile import write_dump
    exe = os.path.join(ROOT, "sora_b200", "brick", "demo_graph")
    if not os.path.exists(exe): subprocess.check_call(["make", "-C", os.path.dirname(exe)], stdout=subprocess.DEVNULL)
    cap = iq_u[:nframes].reshape(-1, 2); cap = cap[: len(cap) // 28 * 28]
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "bench.dmp"); write_dump(p, cap)
        out = subprocess.run([exe, p, "--threads", str(instances), "--repeat", "2"], capture_output=True, text=True, timeout=600).stdout
    s = json.loads([l for l in out.splitlines() if l.startswith("{")][-1])
    assert s["frames_ok"] == 2 * instances * nframes, s
    return {"value": s["msamples_per_s"], "unit": "Msamples/s", "frames_per_s": s["frames_per_s"], "graph_instances": instances, "frames_per_capture": nframes,
            "note": "brick graphs driven like RxThread (fb11a_demod.cpp:29-81); continuous-capture semantics (every frame search starts where the previous event ended): a header-only scout pass per event, then all frames of all graphs in one batch"}

def oracle_gate(eng, torch, iq_u, ps_u, U, res_dev, out_dev, ncores, rank):
    """Every result field and every byte of the U unique slots against the CPU oracle on the same IQ (the remaining slots are copies of these)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_py
    from sora_b200 import api
    off = np.arange(U, dtype=np.uint64) * SLOT; ln = np.full(U, SLOT, np.uint32)
    ores, oout = oracle_py.rx11a_batch(iq_u.reshape(-1, 2), off, ln, out_stride=PSDU, nthreads=max(1, ncores))
    got = res_dev[:U].cpu().numpy().view(api.RESULT_DTYPE).reshape(-1)
    gb = out_dev[:U].cpu().numpy()
    fields = ("status", "rate_kbps", "length", "crc32", "nsym", "detect_index", "cfo_est", "peak_index")
    bad = np.zeros(U, bool)
    for k in fields: bad |= got[k] != ores[k]
    bad |= (gb != oout[:, :PSDU]).any(axis=1)
    idx = np.nonzero(bad)[0]
    if len(idx):    # a second opinion before blaming the device: the same slots once more, one oracle thread, nothing else running in this process
        print(f"[bench] rank {rank}: {len(idx)} of {U} slots differ from the threaded oracle run, slots {idx[:8].tolist()}: "
              f"device status {got['status'][idx[:8]].tolist()} oracle status {ores['status'][idx[:8]].tolist()}; re-running them single-threaded", file=sys.stderr)
        r2, o2 = oracle_py.rx11a_batch(iq_u.reshape(-1, 2), off[idx], ln[idx], out_stride=PSDU, nthreads=1)
        for k in fields:
            assert (got[k][idx] == r2[k]).all(), f"rank {rank}: field {k} differs from the oracle on {(got[k][idx] != r2[k]).sum()} of {U} slots (threaded and single-threaded oracle runs)"
        assert (gb[idx] == o2[:, :PSDU]).all(), "decoded bytes differ from the oracle's"
    assert (got["status"] == 1).all() and (got["length"] == PSDU).all()
    assert (gb == ps_u).all(), "decoded bytes differ from the transmitted PSDUs"
    oracle_gate.rerun = int(len(idx))
    return U

DUMP_SLOTS = 4096      # 4096 x (1500 float32 bytes + 9 float64 fields) = 25 MB

def sample_outputs(torch, res_dev, out_dev):
    """What a caller of the timed path receives — the verdict fields and the PSDU bytes of every slot — for a fixed, seeded sample of
    DUMP_SLOTS slots (all of them when there are fewer), as float64 / float32 arrays by name."""
    from sora_b200 import api
    F = res_dev.shape[0]
    idx = np.arange(F) if F <= DUMP_SLOTS else np.sort(np.random.default_rng(0xD0).choice(F, DUMP_SLOTS, replace=False))
    it = torch.from_numpy(idx).to(res_dev.device)
    res = res_dev.index_select(0, it).cpu().numpy().view(api.RESULT_DTYPE).reshape(-1)
    arrays = {"slot_index": idx.astype(np.float64), "psdu": out_dev.index_select(0, it).cpu().numpy().astype(np.float32)}
    for k in api.RESULT_DTYPE.names:
        arrays["result_" + k] = res[k].astype(np.float64)
    return arrays

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--frames", type=int, default=65536, help="capture slots per step per GPU (BASELINE config #2: 65536)")
    ap.add_argument("--unique", type=int, default=2048, help="distinct synthetic frames generated on the host, tiled to --frames in HBM")
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--chunk", type=int, default=4096, help="slots per pipeline chunk inside the library (0 = no chunking)")
    ap.add_argument("--chunk-device", type=int, default=0, help="slots per pipeline chunk for device-resident IQ (0 = one pass; >0 overlaps the front end of chunk k+1 with the Viterbi of chunk k)")
    ap.add_argument("--host-threads", type=int, default=-1, help="host threads of the decimating e2e path (option host_decimate); -1 = from the CPUs this rank may use")
    ap.add_argument("--front-stage", type=int, default=-1, help="experiment: sample staging of the OFDM front end (0 direct, 1 register double buffer, 2 bulk async copy); -1 = library default")
    ap.add_argument("--vq-pad-smem", type=int, default=0, help="experiment: extra dynamic shared memory per Viterbi CTA (occupancy sweep)")
    ap.add_argument("--e2e-sweep", action="store_true", help="experiment: host thread counts x chunk sizes of the e2e modes, printed to stderr")
    ap.add_argument("--e2e-wc", action="store_true", help="experiment: also time the decimating modes with write-combined staging buffers (option host_stage_wc)")
    ap.add_argument("--vl-pad-smem", type=int, default=0, help="experiment: extra dynamic shared memory per lane-kernel CTA (occupancy sweep)")
    ap.add_argument("--vl-defer", type=int, default=-1, help="experiment: 1 = the lane kernel's traceback spread over the step loop (one look-up per chunk), 0 = at the trigger; -1 = library default")
    ap.add_argument("--vl-hist-block", type=int, default=0, help="experiment: columns per history block of the lane kernel (6 | 8); 0 = library default")
    ap.add_argument("--vl-l2-hints", type=int, default=-1, help="experiment: L2 eviction hints of the lane kernel (bit 0 ring evict_last, bit 1 soft values evict_first); -1 = library default")
    ap.add_argument("--lane-min", type=int, default=-1, help="experiment: option viterbi_lane_min (smallest launch, in code blocks, the one-lane-per-code-block Viterbi takes); -1 = library default")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-mgpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy (rank 0, a seeded sample of at most %d slots)" % DUMP_SLOTS)
    args = ap.parse_args()
    if args.steps < 1: ap.error("--steps must be at least 1")
    if args.warmup < 3: args.warmup = 3
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    from sora_b200 import api
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the product path)")
    torch.cuda.set_device(local)
    aff0 = os.sched_getaffinity(0)                       # the CPU baseline gets the whole box back; the GPU arm runs next to its GPU's NUMA node
    numa = numa_bind(local)
    ncores, cores_how = effective_cpus()
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    # CPUs this rank may count on: after the NUMA binding the affinity is its GPU's node, shared with the other ranks whose GPUs sit there
    ranks_sharing = max(1, (local_world + 1) // 2) if "numa node" in numa else max(1, local_world)
    cores_rank = max(1, ncores // ranks_sharing)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    F = args.frames
    iq_u, ps_u, U = make_input(F, args.unique)
    eng = api.Engine(local)
    eng.set_option("chunk_frames", args.chunk)
    eng.set_option("chunk_frames_device", args.chunk_device)
    eng.set_option("slot_table_immutable", 1)             # the slot tables below are written once and never touched again
    if args.vq_pad_smem: eng.set_option("vq_pad_smem", args.vq_pad_smem)
    if args.front_stage >= 0: eng.set_option("front_stage", args.front_stage)
    if args.lane_min >= 0: eng.set_option("viterbi_lane_min", args.lane_min)
    if args.vl_pad_smem: eng.set_option("vl_pad_smem", args.vl_pad_smem)
    if args.vl_hist_block: eng.set_option("vl_hist_block", args.vl_hist_block)
    if args.vl_defer >= 0: eng.set_option("vl_defer_walk", args.vl_defer)
    if args.vl_l2_hints >= 0: eng.set_option("vl_l2_hints", args.vl_l2_hints)
    stream = torch.cuda.current_stream()
    # ---- HBM-resident input: U unique slots tiled to F (distinct addresses: 2.6 GB at F=65536 >> 126 MB L2) ----
    iq_unique_dev = torch.from_numpy(iq_u.reshape(U, -1)).to(dev)
    reps = (F + U - 1) // U
    iq_dev = iq_unique_dev.repeat(reps, 1)[:F].contiguous()
    off_dev = (torch.arange(F, dtype=torch.int64, device=dev) * SLOT)
    len_dev = torch.full((F,), SLOT, dtype=torch.int32, device=dev)
    out_dev = torch.zeros((F, PSDU), dtype=torch.uint8, device=dev)
    res_dev = torch.zeros((F, 7), dtype=torch.int32, device=dev)
    def step_dev():
        eng.rx11a_raw(iq_dev.data_ptr(), F * SLOT, off_dev.data_ptr(), len_dev.data_ptr(), F, out_dev.data_ptr(), PSDU, res_dev.data_ptr(), stream.cuda_stream)
    # correctness gate before timing: every slot FRAME_OK, and every field + byte of the unique slots equal to the CPU oracle's
    step_dev(); torch.cuda.synchronize()
    st = res_dev[:, 0].cpu().numpy().astype(np.uint32)
    assert (st == 1).all(), f"rank {rank}: {(st != 1).sum()} slots not FRAME_OK"
    gated = oracle_gate(eng, torch, iq_u, ps_u, U, res_dev, out_dev, cores_rank, rank)
    clocks = ClockSampler(local); clocks.start()
    for _ in range(args.warmup): step_dev()
    torch.cuda.synchronize()
    if dist: dist.barrier()
    clocks.mark()
    l0 = eng.launches
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    ktimes = np.zeros(4)
    torch.cuda.synchronize(); e0.record(stream)
    for _ in range(args.steps):
        step_dev()
    e1.record(stream); torch.cuda.synchronize()
    ms_total = e0.elapsed_time(e1)
    launches = eng.launches - l0
    if args.dump_outputs and rank == 0:                    # before the passes below write the output buffers again
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in sample_outputs(torch, res_dev, out_dev).items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    if dist: dist.barrier()
    # per-kernel times of the dominant kernel, measured live with CUDA events on the launch stream (extra pass, same inputs)
    nk = max(3, min(args.steps, 5))
    eng.set_option("chunk_frames", 0); eng.set_option("chunk_frames_device", 0)   # un-pipelined pass: kernels back to back on one stream
    step_dev()
    for _ in range(nk):
        step_dev(); ktimes += np.array(eng.last_kernel_times())
    ktimes /= nk
    vit_kernel = eng.last_viterbi_kernel()                 # which Viterbi kernel the library chose for a launch of F code blocks
    eng.set_option("chunk_frames", args.chunk); eng.set_option("chunk_frames_device", args.chunk_device)
    t_wait = time.perf_counter()                           # a short run can end between two nvidia-smi lines: keep the same load on, untimed, until two have landed
    while clocks.p and clocks.seen() < 2 and time.perf_counter() - t_wait < 2.0:
        step_dev(); torch.cuda.synchronize()
    clk = clocks.stop()
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if dist: dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_step = ms_total / args.steps
    value = world * F * SLOT / (ms_step * 1e-3) / 1e6

    def timed_max(fn, n, warm=3):
        """n calls of fn between CUDA events on `stream`, barrier + synchronize on both sides, max over ranks; ms per call."""
        for _ in range(warm): fn()
        torch.cuda.synchronize()
        if dist: dist.barrier()
        e0.record(stream)
        for _ in range(n): fn()
        e1.record(stream); torch.cuda.synchronize()
        if dist: dist.barrier()
        tt = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if dist: dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item()) / n

    # ---- e2e: pinned host IQ -> C ABI -> pinned host bytes + verdicts, copies inside the timed region ----
    e2e = None
    if not args.no_e2e:
        iq_host = torch.empty((F, SLOT * 2), dtype=torch.int16).pin_memory()
        src_u = torch.from_numpy(iq_u.reshape(U, -1))
        for r in range(reps):
            n = min(U, F - r * U)
            iq_host[r * U: r * U + n].copy_(src_u[:n])
        off_h = (np.arange(F, dtype=np.uint64) * SLOT); len_h = np.full(F, SLOT, np.uint32)
        out_host = torch.empty((F, PSDU), dtype=torch.uint8).pin_memory()
        res_host = torch.empty((F, 7), dtype=torch.int32).pin_memory()
        def step_e2e():
            eng.rx11a_raw(iq_host.data_ptr(), F * SLOT, off_h.ctypes.data, len_h.ctypes.data, F, out_host.data_ptr(), PSDU, res_host.data_ptr(), stream.cuda_stream)
        ne = max(3, min(args.steps, 5))
        nth = args.host_threads if args.host_threads >= 0 else int(max(1, min(16, cores_rank - 2)))
        modes = {}
        d2h = int(F * PSDU + F * 28)
        def run_mode(name, threads, mix, note=None):
            res_host.zero_(); out_host[:U].zero_()
            eng.set_option("host_decimate", threads); eng.set_option("host_decimate_mix", mix)
            ms = timed_max(step_e2e, ne)
            nbytes, chunks, gathered = eng.last_transfer()     # what the last call really sent (the adaptive mode decides per chunk)
            eng.set_option("host_decimate", 0); eng.set_option("host_decimate_mix", 1)
            assert (res_host[:, 0].numpy().astype(np.uint32) == 1).all() and (out_host[:U].numpy() == ps_u).all(), f"e2e {name}: results differ"
            modes[name] = {"value": world * F * SLOT / (ms * 1e-3) / 1e6, "ms_per_step": ms, "h2d_bytes_per_step": int(nbytes + F * (20 if threads else 12)),
                           "d2h_bytes_per_step": d2h, "chunks": chunks, "chunks_gathered_on_host": gathered}
            if threads: modes[name]["host_threads_per_rank"] = threads
        run_mode("full_rate_copy", 0, 1)
        if nth > 0:
            run_mode("host_decimate", nth, 0)
            run_mode("host_decimate_adaptive", nth, 1)
        if nth > 0 and args.e2e_wc:                           # experiment: write-combined staging buffers
            eng.set_option("host_stage_wc", 1)
            run_mode("host_decimate_wc", nth, 0); run_mode("host_decimate_adaptive_wc", nth, 1)
            eng.set_option("host_stage_wc", 0)
        if args.e2e_sweep:                                   # experiment: thread counts and chunk sizes of the adaptive mode, to stderr
            for ch in (2048, 4096):
                eng.set_option("chunk_frames", ch)
                for th in sorted({4, 8, 12, nth, 16, 24, 32}):
                    for mix in (0, 1):
                        run_mode(f"sweep_chunk{ch}_t{th}_mix{mix}", th, mix)
                        m = modes.pop(f"sweep_chunk{ch}_t{th}_mix{mix}")
                        print(f"[e2e sweep] chunk {ch} threads {th} mix {mix}: {m['ms_per_step']:.2f} ms/step, {m['value'] / 1e3:.2f} G samples/s, gathered {m['chunks_gathered_on_host']}/{m['chunks']}, h2d {m['h2d_bytes_per_step'] / 1e9:.3f} GB", file=sys.stderr, flush=True)
            eng.set_option("chunk_frames", args.chunk)
        best = max(modes, key=lambda k: modes[k]["value"])
        e2e = {"value": modes[best]["value"], "unit": "Msamples/s", "ms_per_step": modes[best]["ms_per_step"], "mode": best,
               "h2d_bytes_per_step": modes[best]["h2d_bytes_per_step"], "d2h_bytes_per_step": modes[best]["d2h_bytes_per_step"], "modes": modes,
               "note": "full_rate_copy: the 40 Msps capture crosses PCIe as it is.  host_decimate: T host threads per rank gather the even samples of every chunk (TDownSample2, samples.hpp:27-49: "
                       "the chain never reads the odd ones) into pinned staging inside the timed region, half the bytes cross.  host_decimate_adaptive: per chunk the library gathers, or sends the chunk as it is "
                       "when the queued copies would run out before a gather could finish, so the link and the host cores are both kept busy; h2d_bytes_per_step is what the library reports it copied (sb200_last_transfer)"}
        del iq_host, out_host, res_host

    # ---- mgpu: rank 0 owns all N*F slots; NCCL scatter of IQ slabs, decode, NCCL gather of bytes + verdicts (north_star's partitioning) ----
    mgpu = None
    if dist and not args.no_mgpu:
        P = 4                                              # pieces per slab: the scatter of piece p+1 overlaps the decode of piece p
        Fp = F // P; assert Fp * P == F
        slab = torch.empty((F, SLOT * 2), dtype=torch.int16, device=dev); slab32 = slab.view(torch.int32)   # NCCL has no 16-bit integer type: one COMPLEX16 = one int32
        root = iq_unique_dev.repeat((world * F + U - 1) // U, 1)[: world * F].contiguous().view(torch.int32).view(world, P, Fp, SLOT) if rank == 0 else None
        out_all = torch.empty((world, F, PSDU), dtype=torch.uint8, device=dev) if rank == 0 else None
        res_all = torch.empty((world, F, 7), dtype=torch.int32, device=dev) if rank == 0 else None
        offp = (torch.arange(Fp, dtype=torch.int64, device=dev) * SLOT); lenp = torch.full((Fp,), SLOT, dtype=torch.int32, device=dev)
        def step_mgpu():
            works = []
            for p in range(P):
                lst = [root[r, p] for r in range(world)] if rank == 0 else None
                works.append(dist.scatter(slab32[p * Fp:(p + 1) * Fp], lst, src=0, async_op=True))
            for p in range(P):
                works[p].wait()
                eng.rx11a_raw(slab[p * Fp:(p + 1) * Fp].data_ptr(), Fp * SLOT, offp.data_ptr(), lenp.data_ptr(), Fp,
                              out_dev[p * Fp:(p + 1) * Fp].data_ptr(), PSDU, res_dev[p * Fp:(p + 1) * Fp].data_ptr(), stream.cuda_stream)
            dist.gather(out_dev, [out_all[r] for r in range(world)] if rank == 0 else None, dst=0)
            dist.gather(res_dev, [res_all[r] for r in range(world)] if rank == 0 else None, dst=0)
        nm = max(3, min(args.steps, 5))
        ms_m = timed_max(step_mgpu, nm, warm=2)
        if rank == 0:
            assert (res_all[:, :, 0].cpu().numpy().astype(np.uint32) == 1).all(), "mgpu: a gathered slot is not FRAME_OK"
            assert (out_all[world - 1, :U].cpu().numpy() == ps_u).all(), "mgpu: gathered bytes differ"
            mgpu = {"value": world * F * SLOT / (ms_m * 1e-3) / 1e6, "unit": "Msamples/s", "ms_per_step": ms_m, "collective": "NCCL scatter (IQ slabs, root -> ranks) + gather (bytes, verdicts -> root)",
                    "nccl_ranks": world, "scatter_bytes_per_step": int((world - 1) * F * SLOT * 4), "gather_bytes_per_step": int((world - 1) * F * (PSDU + 28)),
                    "pieces_per_slab": P, "note": "all N*F slots resident on rank 0's GPU at the start of the step; bound by rank 0's NVLink egress"}
        del slab, slab32, root, out_all, res_all
        # the host-side sharding helper the CPU (gloo) tests cover, on the GPUs: the U unique slots split into contiguous blocks per rank
        # (sora_b200/shard.py), every rank decodes its block from host IQ, verdicts and bytes gathered on rank 0 over NCCL and compared whole
        from sora_b200 import shard
        offu = np.arange(U, dtype=np.uint64) * SLOT; lnu = np.full(U, SLOT, np.uint32)
        def decode_block(iq, off, ln):
            r_, o_ = eng.rx11a_batch(iq, off, ln, out_stride=PSDU)
            return r_, o_
        res_s, out_s = shard.decode_sharded(decode_block, iq_u.reshape(-1, 2), offu, lnu, dist=dist, device=dev)
        if rank == 0:
            assert (res_s["status"] == 1).all() and (res_s["length"] == PSDU).all() and (out_s[:, :PSDU] == ps_u).all(), "sharded decode: gathered results differ"
            mgpu["sharded_check"] = f"{U} slots decoded in {world} contiguous blocks (shard.decode_sharded), gathered over NCCL, all FRAME_OK with the transmitted bytes"
    del iq_unique_dev
    if rank != 0:
        if dist: dist.destroy_process_group()
        return
    peak, how = load_peaks()
    vit_ms = float(ktimes[2])
    alg_bytes = ALG_BYTES_PER_SAMPLE * F * SLOT           # whole-chain algorithmic bytes attributed to the dominant kernel's launch
    achieved = alg_bytes / (vit_ms * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try: tj = json.load(open(tp)); traffic = tj.get(vit_kernel + "_dram_bytes_per_frame", 0) * F or None
        except Exception: traffic = None
    line = {"metric": METRIC, "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int16 (fixed point; uint8 path metrics)", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "slots_per_step_per_gpu": F, "unique_slots": U, "samples_per_slot": SLOT, "psdu_bytes": PSDU,
                       "parallelism": f"independent slots, {world} GPU(s), no data-path collective",
                       "l2_policy": "input 2.6 GB per step >> 126 MB L2 (no flush needed)" if F * SLOT * 4 > 4e8 else "input smaller than L2: increase --frames",
                       "oracle_gate": f"{gated} unique slots compared field by field and byte by byte with the CPU oracle before timing"
                                      + (f" ({oracle_gate.rerun} slots where the threaded oracle run disagreed were settled by a single-threaded oracle run)" if getattr(oracle_gate, "rerun", 0) else ""),
                       "numa": numa},
            "kernel_ms": {"carrier_sense": float(ktimes[0]), "ofdm_front_end": float(ktimes[1]), "viterbi_descramble_crc": vit_ms, "pack": float(ktimes[3])},
            "roofline": {"bound": "hbm", "kernel": f"{vit_kernel}<CR_34> (+ work lists, frame sink)", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": how,
                         "note": "achieved = 4.154 B/sample x samples per launch / Viterbi kernel time; the chain is integer-ALU/issue bound, not HBM bound (DESIGN.md)"},
            "clocks": clk, "gpu_launches": int(launches), "e2e": e2e}
    if mgpu: line["mgpu"] = mgpu
    if world == 1 and not args.no_e2e:
        try: line["e2e_brick"] = brick_leg(iq_u)
        except Exception as e: line["e2e_brick"] = {"unavailable": f"{type(e).__name__}: {e}"}
    if not args.no_cpu and world == 1:
        os.sched_setaffinity(0, aff0); ncores, cores_how = effective_cpus()
        variants, best = cpu_baseline(iq_u, ncores)
        line["cpu_baseline"] = {"value": variants[best]["value"], "unit": "Msamples/s", "cores": ncores, "kind": "port", "cpu_model": cpu_model(), "cores_how": cores_how,
                                "sample": f"{variants[best]['slots']} slots of the same workload, {variants[best]['threads']} host threads ({best}), {variants[best]['seconds']} s (oracle/ SSE restatement)",
                                "variants": variants}
    print(json.dumps(line))
    if dist: dist.destroy_process_group()

if __name__ == "__main__":
    main()
