#!/usr/bin/env python
"""bench.py -- headline benchmark: ciphertext-ops/s of the Sobel program
(examples/image_processing.py:39-63, compiled by the reference compiler:
N=16384, 5x60-bit primes, 61 ciphertext ops) on N B200s, plus the NTT HBM GB/s
roofline line.  See the driver contract in the task description.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

* our arm: the product path only (eva_b200 -> C-ABI -> CUDA); inputs/keys are
  synthetic uniform residues (every kernel is data-independent integer work).
* --impl reference: the reference's SEAL path cannot be built here (no SEAL);
  the CPU arm is the oracle port of that path (oracle/, kind "port") run with
  all host threads on the same workload.
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
WORKLOAD = "sobel"          # workloads/sobel.json: the reference compiler's output for examples/image_processing.py
METRIC = "ciphertext-ops/sec"
DUMP_BYTES = 60 * 10 ** 6   # --dump-outputs: all files together (npy headers aside) stay below 64 MB


def load_workload(name):
    """a reference-compiled program dump by name (workloads/, then the test fixtures) or by path -- plain json/gzip,
    so that the CPU reference arm never imports the product package"""
    import gzip
    cands = [name] if (os.path.sep in name or name.endswith((".json", ".gz"))) else \
        [os.path.join(ROOT, dd, name + ext) for dd in ("workloads", os.path.join("tests", "golden", "programs")) for ext in (".json", ".json.gz")]
    path = next((c for c in cands if os.path.exists(c)), cands[0])
    with (gzip.open(path, "rt") if path.endswith(".gz") else open(path)) as f:
        return json.load(f)


def bench_config(name, d, nops, B):
    """identical in both arms (the driver compares them)"""
    return {"workload": workload_desc(name, d, nops) + "; one step = batch of %d independent program instances (images) per GPU" % B,
            "instances_per_step": B, "l2": "GPU arm: flushed between timed steps (256 MiB memset, untimed)"}


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region"""

    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.stop_flag = gpu, [], False
        self.proc = None

    def run(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
                if self.stop_flag:
                    break
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        sm, smax, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); smax = max(smax, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax or None, "reasons": sorted(reasons), "samples": len(sm)}


def synthetic_inputs(d, primes, seed):
    """uniform residues in [0, q_i) as ciphertexts / keys (valid evaluator inputs)"""
    rng = np.random.default_rng(seed)
    N, k = d["poly_modulus_degree"], len(primes)

    def uni(shape_prefix, prime_idx):
        a = np.empty(tuple(shape_prefix) + (len(prime_idx), N), dtype=np.uint64)
        for j, pi in enumerate(prime_idx):
            a[..., j, :] = rng.integers(0, primes[pi], size=tuple(shape_prefix) + (N,), dtype=np.uint64)
        return a
    relin = uni((k - 1, 2), list(range(k)))
    galois = {}
    for t in d["terms"]:
        if t["op"] in ("RotateLeftConst", "RotateRightConst") and t["rotation"] != 0:
            steps = t["rotation"] if t["op"] == "RotateLeftConst" else -t["rotation"]
            s = steps if steps > 0 else N // 2 + steps
            elt = pow(3, s, 2 * N)
            if elt not in galois:
                galois[elt] = uni((k - 1, 2), list(range(k)))
    cts = {}
    for name, info in d["signature"].items():
        ell = k - 1 - info["level"]
        cts[name] = (uni((2,), list(range(ell))), 2.0 ** info["scale"])
    return relin, galois, cts


def workload_desc(name, d, nops):
    head = "sobel_64x64 (examples/image_processing.py)" if name == "sobel" else name
    return "%s compiled by the reference compiler: N=%d, prime_bits=%s, %d ciphertext ops per instance" % (
        head, d["poly_modulus_degree"], "[60]*5" if d["prime_bits"] == [60] * 5 else str(d["prime_bits"]), nops)


def multi_seed(rank, index):
    from eva_b200 import multi
    return multi.instance_seed(rank, index)


def dump_outputs(outdir, wl, d, outs, budget):
    """The output ciphertexts that the last timed step handed to the caller (execute_batch_result: one valuation per
    instance), as DIR/<workload>_<output>.npy, float64 [instances][polys][ell][coefficients][2]: every residue (< 2^60)
    split exactly into its high and low 30 bits.  Above `budget` bytes per workload, a fixed seeded choice of
    coefficient indices (the same in every run) is kept."""
    os.makedirs(outdir, exist_ok=True)
    names = sorted(d["outputs"])
    for name in names:
        arr = np.stack([np.asarray(o.get(name)[1]) for o in outs]).astype(np.uint64)
        per_coeff = arr.size // arr.shape[-1] * 16
        keep = max(1, min(arr.shape[-1], budget // len(names) // per_coeff))
        if keep < arr.shape[-1]:
            arr = arr[..., np.sort(np.random.default_rng(0).choice(arr.shape[-1], keep, replace=False))]
        split = np.stack([arr >> np.uint64(30), arr & np.uint64((1 << 30) - 1)], axis=-1).astype(np.float64)
        np.save(os.path.join(outdir, "%s_%s.npy" % (wl, name)), split)


def measure_workload(args, wl, steps, rank, world, local, dump_budget=0):
    """device-resident value, e2e through execute_batch and single-instance latency of one workload"""
    import torch
    import torch.distributed as dist
    from eva_b200 import b200, program_io
    d = load_workload(wl)
    B = args.instances
    N = d["poly_modulus_degree"]
    primes = b200.create_coeff_modulus(N, d["prime_bits"])
    relin, galois, cts = synthetic_inputs(d, primes, seed=1234 + rank)
    pub = b200.context_from_raw_keys(N, primes, relin, galois, local)
    pub.set_options(num_streams=args.streams, use_graph=not args.no_graph, cache_constants=not args.no_const_cache, dedup_constants=not args.no_dedup)
    # B independent program instances (different input ciphertexts, same keys), organised as
    # G concurrent plan replays (one CUDA graph each, on its own stream) x F instances fused
    # into every kernel launch of a plan (execute_batch / evab_set_batch):  B = G * F
    F = max(1, min(args.fuse, B))
    G = B // F
    assert G * F == B, "--instances must be a multiple of --fuse"
    prog, params, sig, terms = program_io.build_program(d)
    all_vals = []
    for i in range(B):
        _, _, cts_i = synthetic_inputs({**d, "terms": []}, primes, seed=multi_seed(rank, i))
        val = b200.B200Valuation()
        for name, (ct, scale) in cts_i.items():
            val.set_cipher(name, ct, scale)   # host image in page-locked memory
        all_vals.append(val)
    groups = [all_vals[g * F:(g + 1) * F] for g in range(G)]   # plan replica g executes instances gF .. gF+F-1
    nops = pub.cipher_op_count(prog)
    main = torch.cuda.current_stream()
    streams = [torch.cuda.Stream() for _ in range(G)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident():
        fork = torch.cuda.Event()
        fork.record(main)
        for g in range(G):
            streams[g].wait_event(fork)
            pub.run_resident(prog, streams[g].cuda_stream, F, g)
            ev_ = torch.cuda.Event()
            ev_.record(streams[g])
            main.wait_event(ev_)

    # ---- launches per step: one un-graphed replay of one group's plan, times G
    opts = dict(num_streams=args.streams, cache_constants=not args.no_const_cache, dedup_constants=not args.no_dedup, fuse=F,
                approx_hoist=args.approx_hoist, rotation_chunk=args.rotation_chunk)
    pub.set_options(use_graph=False, **opts)
    pub.drop_plan(prog, 1)   # (cipher_op_count above built a batch-1 plan)
    pub.drop_plan(prog, F)
    pub.stage_inputs(prog, groups[0], main.cuda_stream)
    pub.run_resident(prog, main.cuda_stream, F)
    torch.cuda.synchronize()
    l0 = pub.launch_count()
    pub.run_resident(prog, main.cuda_stream, F)
    torch.cuda.synchronize()
    launches_per_step = (pub.launch_count() - l0) * G
    pub.set_options(use_graph=not args.no_graph, **opts)
    pub.drop_plan(prog, F)
    for g in range(G):
        pub.stage_inputs(prog, groups[g], main.cuda_stream, g)
    torch.cuda.synchronize()
    for _ in range(max(3, args.warmup)):
        step_resident()
    torch.cuda.synchronize()
    for _ in range(max(3, args.warmup)):       # warm the e2e path (same plan replicas; fills the pinned-buffer pool)
        outs = pub.execute_batch(prog, all_vals)
    def pipelined(n):
        """n steps with two calls in flight: step i+1 is submitted before step i is collected"""
        pending, outs = None, None
        for i in range(n):
            nxt = pub.execute_batch_async(prog, all_vals, i & 1)
            if pending is not None:
                outs = pub.execute_batch_result(pending)
            pending = nxt
        return pub.execute_batch_result(pending)
    pipelined(2 * max(3, args.warmup))          # ... and the pipelined form: both slots, and the page-locked pool at its steady size (three result sets alive)

    sampler = ClockSampler(local)
    sampler.start()
    # ---- device-resident value: K steps, each bracketed by events, L2 flushed between steps (untimed)
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for i in range(steps):
        flush.zero_()
        ev[i][0].record(main)
        step_resident()
        ev[i][1].record(main)
    barrier()
    step_ms = sorted(a.elapsed_time(b) for a, b in ev)
    t_res = sum(step_ms) * 1e-3
    # ---- single-instance latency (batch-1 plan, one graph launch, nothing else on the GPU)
    prog0 = prog
    pub.stage_inputs(prog0, all_vals[:1], main.cuda_stream)
    for _ in range(3):
        pub.run_resident(prog0, main.cuda_stream, 1)
    torch.cuda.synchronize()
    lat = []
    for i in range(10):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(main); pub.run_resident(prog0, main.cuda_stream, 1); b.record(main)
        torch.cuda.synchronize()
        lat.append(a.elapsed_time(b))
    lat.sort()
    # ---- e2e through the public API: host buffers in/out (H2D + D2H inside the timed region);
    #      G concurrent execute_batch() calls of F valuations each per step
    barrier()
    t0 = time.perf_counter()
    for i in range(steps):
        outs = pub.execute_batch(prog, all_vals)
    torch.cuda.synchronize()
    t_e2e_sync = time.perf_counter() - t0
    # the same K steps with two calls in flight (execute_batch_async / execute_batch_result, slots 0 and 1): step i+1 is submitted
    # before step i is collected, so the ramp-up of one batch overlaps the drain of the other.  Every step still copies its own
    # inputs host -> device and its own outputs device -> host inside the timed region.
    barrier()
    t0 = time.perf_counter()
    outs = pipelined(steps)
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    barrier()
    clocks = sampler.finish()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, wl, d, outs, dump_budget)
    h2d = sum(ct.nbytes for ct, _ in cts.values()) * B
    okind, oarr, _ = outs[0].get(list(d["outputs"].keys())[0])
    d2h = int(oarr.nbytes) * B
    # ---- final gather of the outputs on rank 0 (north_star: NCCL only for the final gather)
    from eva_b200 import multi
    if world > 1:
        gathered = multi.gather_outputs(oarr, rank, world, device="cuda")
        assert rank != 0 or len(gathered) == world
        t_res, t_e2e, t_e2e_sync = multi.max_over_ranks([t_res, t_e2e, t_e2e_sync], world, device="cuda")
    total_ops = multi.aggregate_ops(nops, B, steps, world)
    result = {
        "metric": METRIC, "value": total_ops / t_res, "unit": "ops/s", "n_gpus": world, "steps": steps, "warmup": args.warmup,
        "ms_per_step": t_res / steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic",
        "config": bench_config(wl, d, nops, B),
        "step_ms": {"median": step_ms[len(step_ms) // 2], "p95": step_ms[min(len(step_ms) - 1, int(0.95 * len(step_ms)))], "min": step_ms[0], "max": step_ms[-1],
                    "note": "per-step CUDA-event durations on this rank (the headline uses their sum, max over ranks)"},
        "details": {"instances_per_gpu": B, **({"approx_hoist": "ON: results are NOT bit-identical to the reference (one mod-down per weighted rotation sum)"} if args.approx_hoist else {}),
                   "parallelism": "replicas x%d GPUs (independent program instances, no data-path collective; NCCL gather of outputs)" % world,
                   "l2": "flushed between timed steps (256 MiB memset, untimed)", "scheduler": ("%d concurrent cuda-graphs" % G if not args.no_graph else "streams") + " x %d instances fused per kernel launch, %d streams inside a plan" % (F, args.streams),
                   "const_encode": "cached per plan" if not args.no_const_cache else ("every Encode term is evaluated on the GPU inside every execute, as in the reference"
                                    + ("; identical constants share one plaintext and replicated scalars use the one-pass encoder (bit-identical to the FP64 FFT + NTT path)" if not args.no_dedup else ""))},
        "e2e": {"value": total_ops / t_e2e, "unit": "ops/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": t_e2e / steps * 1e3,
                "blocking": {"value": total_ops / t_e2e_sync, "ms_per_step": t_e2e_sync / steps * 1e3,
                             "note": "the same with one blocking B200Public.execute_batch call per step (no overlap between steps)"},
                "note": "one B200Public.execute_batch_async(program, %d host-resident valuations) per step, collected with execute_batch_result after the next step has been submitted (two steps in flight, disjoint plan replicas): %d concurrent plan replicas x %d fused instances, page-locked host buffers, H2D + graph + D2H per replica stream (host wall clock)" % (B, G, F)},
        "single_instance": {"latency_ms": lat[len(lat) // 2], "ops_per_s": nops / (lat[len(lat) // 2] * 1e-3)},
        "gpu_launches": int(launches_per_step * steps),
        "clocks": clocks,
    }
    for g in range(G):
        pub.drop_plan(prog, F, g)       # release the replicas' arenas before the next workload
    pub.drop_plan(prog, 1)
    return result, pub, main


def run_ours(args):
    if args.ntt_cluster is not None:
        from eva_b200 import cabi
        assert cabi.load().evab_set_ntt_cluster(args.ntt_cluster) == 0
    import torch
    import torch.distributed as dist
    from eva_b200 import b200
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1)); local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    extra_workloads = [] if (world > 1 or args.no_extras) else [n for n in ("harris", "polynomial") if n != args.workload]
    dump_budget = DUMP_BYTES // (1 + len(extra_workloads))
    result, pub, main = measure_workload(args, args.workload, args.steps, rank, world, local, dump_budget)
    if extra_workloads:
        # BASELINE configs 1 and 4 next to the headline (config 3): the same measurement
        extras = {}
        for name in extra_workloads:
            r, _, _ = measure_workload(args, name, args.steps, rank, world, local, dump_budget)
            extras[name] = {"workload": r["config"]["workload"], "value": r["value"], "unit": "ops/s", "ms_per_step": r["ms_per_step"],
                            "e2e_value": r["e2e"]["value"], "single_instance": r["single_instance"]}
        result["other_workloads"] = extras
    if world > 1 and not args.no_dag_sharded:
        # north_star's other multi-GPU mode: ONE compiled program sharded over the GPUs (BASELINE configs 4 and 5)
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import dagshard_bench
        shard_res = []
        for wl in ("wide4096", "harris"):
            shard_res.append(dagshard_bench.measure(wl, rank, world, local, steps=args.steps, warmup=3, quiet=True))
        result["dag_sharded"] = [{k: r.get(k) for k in ("workload", "cipher_ops", "ms_single_gpu", "ms_sharded", "speedup", "bit_identical", "auto_choice", "stages", "note") if k in r} for r in shard_res]
    if rank == 0:
        result["roofline"] = ntt_roofline(pub, b200.create_coeff_modulus(16384, [60] * 4), 16384, main.cuda_stream)   # always the BASELINE shape
        if world == 1 and not args.no_cpu:
            result["cpu_baseline"] = cpu_baseline(load_workload(args.workload), args.instances, sample_steps=1, single_thread=True)
        print(json.dumps(result))
    if world > 1:
        dist.destroy_process_group()


def ntt_roofline(pub, primes, N, stream):
    """dominant kernel: the register-resident NTT.  Timed live with CUDA events on the
    launching stream, batch footprint 1 GiB (>> L2); algorithmic bytes = 2*8*N per residue."""
    import ctypes as C
    import torch
    from eva_b200 import cabi
    lib = cabi.load()
    peaks, which = load_peaks()
    L = 4
    pa = np.array(primes[:L], dtype=np.uint64)
    h = C.c_void_p()
    assert lib.evab_ctx_create(N, pa.ctypes.data_as(cabi.u64p), L, torch.cuda.current_device(), C.byref(h)) == 0
    cnt = (1 << 30) // (N * 8)
    data = torch.randint(0, 1 << 59, (cnt, N), dtype=torch.int64, device="cuda")
    pidx = (C.c_int * L)(*range(L))
    st = C.c_void_p(stream)
    for _ in range(3):
        lib.evab_ntt_fwd(h, C.c_void_p(data.data_ptr()), cnt, pidx, L, st)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    iters = 10
    e0.record()
    for _ in range(iters):
        lib.evab_ntt_fwd(h, C.c_void_p(data.data_ptr()), cnt, pidx, L, st)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    algo = 2.0 * cnt * N * 8
    ach = algo / (ms * 1e-3) / 1e9
    del data
    lib.evab_ctx_destroy(h)
    # DRAM traffic of the same launch from the committed ncu --set full capture (profiles/)
    traffic, traffic_src = None, None
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_ntt_fwd.json")))
        if prof.get("residues_per_launch") == cnt:
            traffic, traffic_src = prof["traffic_bytes_per_launch"], prof["source"]
    except Exception:
        pass
    return {"bound": "hbm", "kernel": "k_ntt_fwd<14> (batched, %d residues/launch)" % cnt, "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "frac": ach / peaks["hbm_gbs"], "traffic": traffic, "traffic_source": traffic_src, "peak_source": which + " (MEASURED_PEAKS.json hbm_gbs)" if which == "measured" else "fallback 6650",
            "algorithmic_bytes_per_launch": algo, "launch_ms": ms}


def cpu_baseline(d, B, sample_steps=1, threads=None, single_thread=False):
    """the oracle port of the reference's CPU path on the host cores: the same step
    (a batch of B Sobel instances) scheduled on one dependency-counting thread pool"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle import oracle as o
    from oracle_exec import OracleProgram, run_many
    threads = threads or len(os.sched_getaffinity(0))
    N = d["poly_modulus_degree"]
    orc = o.Oracle(N, d["prime_bits"]).keygen(1)
    op = OracleProgram(d, orc)
    op.prepare_keys()
    rng = np.random.default_rng(0)
    batch = []
    for i in range(B):
        inputs = {}
        for name, info in d["signature"].items():
            ell = orc.k - 1 - info["level"]
            inputs[name] = ("cipher", orc.encrypt(orc.encode(rng.uniform(0, 0.2, d["vec_size"]), 2.0 ** info["scale"], ell), seed=i), 2.0 ** info["scale"])
        batch.append(inputs)
    nops = op.cipher_op_count()
    run_many(op, batch[:max(1, min(B, threads // 8))], threads)  # warm-up
    t0 = time.perf_counter()
    for _ in range(sample_steps):
        run_many(op, batch, threads)
    dt = time.perf_counter() - t0
    res = {"value": nops * B * sample_steps / dt, "unit": "ops/s", "cores": threads, "kind": "port", "ops_per_instance": nops,
           "sample": "%d step(s) of %d program instances (%d ops each) on the oracle port (not SEAL), one dependency-counting thread pool over %d threads" % (sample_steps, B, nops, threads),
           "ms_per_step": dt / sample_steps * 1e3}
    if single_thread:      # BASELINE.md: the 1-thread figure next to the all-core one (one program instance, sequential)
        t0 = time.perf_counter()
        op.run(batch[0], threads=1, keep=set())
        dt1 = time.perf_counter() - t0
        res["single_thread"] = {"value": nops / dt1, "unit": "ops/s", "cores": 1, "sample": "1 program instance (%d ops), sequential" % nops}
    return res


def run_reference(args):
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1))
    if rank != 0:
        return
    d = load_workload(args.workload)     # plain json: this arm never imports the product package or its libraries
    cb = None
    t0 = time.perf_counter()
    # each step is a bounded sample of the workload: as many program instances of the batch as the host
    # cores can run concurrently (4 threads each), so K steps end within a few minutes on any host
    threads = len(os.sched_getaffinity(0))
    Bs = max(1, min(args.instances, threads // 4))
    cb = cpu_baseline(d, Bs, sample_steps=max(1, args.steps))
    nops = cb["ops_per_instance"]
    dt = time.perf_counter() - t0
    res = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "ops/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
           "config": bench_config(args.workload, d, nops, args.instances),
           "details": {"cpu_sample_instances_per_step": Bs,
                       "note": "reference SEAL+Galois path cannot be built (SEAL absent); CPU oracle port of the same path, all host threads; each step is a bounded sample of the batch"},
           "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": "ops/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "wall_s": dt}
    print(json.dumps(res))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--streams", type=int, default=8)
    ap.add_argument("--instances", type=int, default=32, help="independent Sobel program instances per GPU per step")
    ap.add_argument("--fuse", type=int, default=1, help="instances fused into each kernel launch (instances/fuse concurrent graphs)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--const-cache", dest="no_const_cache", action="store_false",
                    help="encode constant plaintexts once per plan instead of inside every execute (default: every execute, like the reference)")
    ap.set_defaults(no_const_cache=True)
    ap.add_argument("--no-dedup", action="store_true", help="encode every Encode term separately even when constants repeat")
    ap.add_argument("--approx-hoist", action="store_true",
                    help="NOT bit-exact with the reference: one mod-down per weighted sum of rotations (SURVEY 8f-4); off in every reported line")
    ap.add_argument("--rotation-chunk", type=int, default=16, help="rotations of one ciphertext per evab_rotate_modup_many call (1: one call each)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the Harris / polynomial lines (other_workloads)")
    ap.add_argument("--no-dag-sharded", action="store_true", help="N > 1: skip the DAG-sharded wide4096 / Harris measurement (dag_sharded)")
    ap.add_argument("--workload", default=WORKLOAD, help="program under workloads/ (default: the BASELINE workload, sobel); e.g. harris")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last e2e step of every workload as DIR/<workload>_<output>.npy "
                         "(rank 0, replica workloads; not the N > 1 dag_sharded runs; nothing with --impl reference, whose CPU arm "
                         "runs other inputs)")
    ap.add_argument("--ntt-cluster", type=int, default=None, help="CTAs per residue transform (1, 2, 4); default: library default")
    args = ap.parse_args()
    if args.impl == "reference":
        if args.dump_outputs:
            print("bench.py: --dump-outputs writes nothing with --impl reference", file=sys.stderr)
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
