#!/usr/bin/env python
"""bench.py — headline metric of BASELINE.json: ciphertext multiply+relinearize per second at n=8192,
218-bit BFVDefault chain (k=4 data residues + special prime), batch = 1024 ciphertext pairs per GPU.

  python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path (one rank per GPU under torchrun)
  python bench.py --impl reference --steps K --warmup W  # the reference's own CPU implementation (oracle/_ref)

One "step" = one pass of the hot path (Evaluator::multiply then ::relinearize) over the whole batch.
`value` = device-resident throughput (inputs already in HBM).
`e2e`   = the same metric through the reference-facing PLUGIN calls (the SEAL-named C ABI, include/b200_sealc.h) with HOST
          buffers: pinned host words -> B200_Ciphertext_SetWordsBatch -> B200_Evaluator_MultiplyRelinBatch ->
          B200_Ciphertext_GetWordsBatch -> pinned host words, copies inside the timed region, a few worker threads each
          driving chunks of the batch (the call pattern of sunscreen_runtime's rayon workers, run.rs:237-282,415-469).
`e2e_host_slab`     = the layer-1 host-buffer entry point b200_multiply_relin_host (last round's `e2e`).
`plugin_per_handle` = Evaluator_Multiply + Evaluator_Relinearize per ciphertext handle from 8 threads (what unmodified
          sunscreen_runtime issues today), handles device-resident.
`roofline` is measured live on the dominant kernel (the batched NTT, BASELINE config 2: 4096 polynomials x 4 residues) with
CUDA events on the launching stream, `roofline_keyswitch` on the batched relinearisation (key-switch inner product);
`cpu_baseline` times the unmodified reference on this box's host cores on a bounded sample of the same workload and says how
many cores the box actually grants.  Under torchrun (N > 1) a `sharded` leg runs the north-star split: rank 0 holds the batch,
NCCL scatter -> every rank computes -> NCCL gather, checked against the 1-GPU words.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

N_POLY = 8192
MODULI = [0x7fffffd8001, 0x7fffffc8001, 0xfffffffc001, 0xffffff6c001, 0xfffffebc001]
PLAIN = 1032193
BATCH = 1024
NTT_POLYS = 4096  # BASELINE config 2
DUMP_ITEMS = 64  # ciphertexts of the last timed step written by --dump-outputs: 64 x 2 x 4 x 8192 float64 = 32 MiB


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def cpu_quota():
    """What the box really grants: CPUs in the affinity mask and the cgroup CPU bandwidth limit (cores' worth), if any."""
    info = {"logical_cpus": os.cpu_count(), "affinity_cpus": None, "cgroup_quota_cores": None}
    try:
        info["affinity_cpus"] = len(os.sched_getaffinity(0))
    except Exception:
        pass
    try:
        txt = open("/sys/fs/cgroup/cpu.max").read().split()
        if txt and txt[0] != "max":
            info["cgroup_quota_cores"] = float(txt[0]) / float(txt[1])
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                info["cgroup_quota_cores"] = q / per
        except Exception:
            pass
    eff = [v for v in (info["affinity_cpus"], info["cgroup_quota_cores"], info["logical_cpus"]) if v]
    info["effective_cores"] = min(eff) if eff else None
    return info


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, index=0):
        self.samples = []
        self.mark = 0
        self.proc = None
        self.index = index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "25",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], 0, set()
        for s in self.samples[max(self.mark - 1, 0):]:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def bind_to_gpu_numa(index):
    """Pin this process to the CPUs of the NUMA node the GPU hangs off, so pinned host buffers are node-local."""
    try:
        bdf = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(index)],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if bdf.startswith("00000000:"):
            bdf = "0000:" + bdf[9:]
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def cpu_reference_rate(threads, iters, warmup=2):
    """Unmodified reference (oracle/_ref/libsealc_ref.so): threads x iters multiply+relinearize_inplace, own pool per thread."""
    import numpy as np
    import refseal
    R = refseal.RefContext(N_POLY, MODULI, PLAIN)
    rng = np.random.default_rng(0)
    k = 4

    def rand_ct():
        w = np.empty((2, k, N_POLY), dtype=np.uint64)
        for i in range(k):
            w[:, i, :] = rng.integers(0, MODULI[i], size=(2, N_POLY), dtype=np.uint64)
        return R.new_ct(w)

    key = np.empty((k, 2, 5, N_POLY), dtype=np.uint64)
    for i in range(5):
        key[:, :, i, :] = rng.integers(0, MODULI[i], size=(k, 2, N_POLY), dtype=np.uint64)
    a, b, rlk = rand_ct(), rand_ct(), R.new_ksk({0: key})
    secs = R.time_mul_relin(a, b, rlk, threads, iters, warmup)
    return threads * iters / secs, secs


def run_reference(args):
    """The reference's own CPU implementation (oracle/_ref) on all host cores; one step = a bounded sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np
    import refseal
    cores = os.cpu_count() or 1
    iters = 16  # per thread per step: cores*16 multiply+relinearize per step
    R = refseal.RefContext(N_POLY, MODULI, PLAIN)
    rng = np.random.default_rng(0)
    k = 4
    w = np.empty((2, 2, k, N_POLY), dtype=np.uint64)
    key = np.empty((k, 2, 5, N_POLY), dtype=np.uint64)
    for i in range(k):
        w[:, :, i, :] = rng.integers(0, MODULI[i], size=(2, 2, N_POLY), dtype=np.uint64)
    for i in range(5):
        key[:, :, i, :] = rng.integers(0, MODULI[i], size=(k, 2, N_POLY), dtype=np.uint64)
    a, b, rlk = R.new_ct(w[0]), R.new_ct(w[1]), R.new_ksk({0: key})
    for _ in range(max(args.warmup, 1)):
        R.time_mul_relin(a, b, rlk, cores, 4, 1)
    secs = 0.0
    for _ in range(args.steps):
        secs += R.time_mul_relin(a, b, rlk, cores, iters, 0)
    rate = args.steps * cores * iters / secs
    line = {
        "metric": "ciphertext mul+relin/sec", "value": rate, "unit": "ops/s", "impl": "reference", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": 1000.0 * secs / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": "Evaluator::multiply + relinearize, n=8192, BFVDefault 218-bit chain (k=4 + special), "
                               f"bounded sample of {cores * iters} ct pairs per step", "batch_per_step": cores * iters,
                   "parallelism": f"{cores} host threads, one memory pool each (oracle/_ref = unmodified reference)"},
        "cpu_baseline": {"value": rate, "unit": "ops/s", "cores": cores, "kind": "reference",
                         "sample": f"{args.steps} steps x {cores} threads x {iters} multiply+relinearize_inplace, "
                                   "uniform-random ciphertext words",
                         # threads used vs what the lease really grants (a CPU-quota'd 1-GPU lease gives ~16 cores' worth)
                         "box": cpu_quota(),
                         "build": "unmodified reference sources, -O3, Intel HEXL off (not buildable offline)"},
        "e2e": {"value": rate, "unit": "ops/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


class PluginLegs:
    """The reference-facing plugin calls of OUR library (include/b200_sealc.h), driven the way seal_fhe's wrappers do:
    opaque handles, one Evaluator, relinearization keys as a KSwitchKeys handle."""

    def __init__(self, ctx, device, k, n, rlk_dev):
        import ctypes as C
        import numpy as np
        from sealc_driver import Sealc
        from sunscreen_b200.lib import B200Lib
        self.C, self.np = C, np
        self.vp, self.u64 = C.c_void_p, C.c_uint64
        self.S = Sealc(B200Lib.default().lib)
        self.O = self.S.context(N_POLY, MODULI, PLAIN)
        self.k, self.n = k, n
        key = rlk_dev.cpu().numpy().view(np.uint64)  # (k, 2, K, n) key-level NTT-form words
        self.rlk = self.O.new_ksk({0: key})
        # worker threads spin while their call completes: with many ranks on one host keep their total below the cores the lease
        # grants (8 ranks x 8 spinning threads on a 96-core quota was seen to get the whole job throttled)
        world = int(os.environ.get("WORLD_SIZE", "1"))
        self.threads = int(os.environ.get("B200_BENCH_E2E_THREADS", "8" if world <= 4 else "4"))
        self.chunk = int(os.environ.get("B200_BENCH_E2E_CHUNK", "64" if world <= 4 else "128"))
        self.pool = {}

    def _handles(self, tag, count):
        hs = self.pool.get(tag)
        if hs is None or len(hs) < count:
            hs = [self.O._dst() for _ in range(count)]
            self.pool[tag] = hs
        return hs[:count]

    def _arr(self, hs):
        return (self.vp * len(hs))(*hs)

    def _ptr(self, t):
        return self.C.cast(t.data_ptr(), self.C.POINTER(self.u64))

    def batch_step(self, abh, oh, B):
        """host words -> handles -> MultiplyRelinBatch -> host words, chunks of the batch driven by worker threads.
        abh: pinned (chunks, 2, chunk, 2, k, n) — per chunk the first operands, then the second operands, so that ONE
        B200_Ciphertext_SetWordsBatch call (one transfer) loads both operand sets of a chunk."""
        S, O, u64, C = self.S, self.O, self.u64, self.C
        chunks = [(lo, min(lo + self.chunk, B)) for lo in range(0, B, self.chunk)]
        errs = []

        def work(tid):
            try:
                for ci in range(tid, len(chunks), self.threads):
                    lo, hi = chunks[ci]
                    cnt = hi - lo
                    ha, hb = self._handles(("a", ci), cnt), self._handles(("b", ci), cnt)
                    D = self._arr(self._handles(("d", ci), cnt))
                    S.call("B200_Ciphertext_SetWordsBatch", O.ctx, u64(2 * cnt), self._arr(ha + hb), O.first_id, u64(2), C.c_bool(False),
                           self._ptr(abh[ci]))
                    S.call("B200_Evaluator_MultiplyRelinBatch", O.ev, u64(cnt), self._arr(ha), self._arr(hb), self.rlk, D)
                    S.call("B200_Ciphertext_GetWordsBatch", O.ctx, u64(cnt), D, self._ptr(oh[lo]), u64(cnt * 2 * self.k * self.n))
            except Exception as ex:  # surfaced by the caller
                errs.append(ex)

        ts = [threading.Thread(target=work, args=(t,)) for t in range(self.threads)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        if errs:
            raise errs[0]

    def per_handle_prepare(self, ah, bh, pairs):
        S, O, u64, C = self.S, self.O, self.u64, self.C
        self.pa, self.pb = self._handles("pa", pairs), self._handles("pb", pairs)
        self.pm, self.pr = self._handles("pm", pairs), self._handles("pr", pairs)
        S.call("B200_Ciphertext_SetWordsBatch", O.ctx, u64(pairs), self._arr(self.pa), O.first_id, u64(2), C.c_bool(False), self._ptr(ah))
        S.call("B200_Ciphertext_SetWordsBatch", O.ctx, u64(pairs), self._arr(self.pb), O.first_id, u64(2), C.c_bool(False), self._ptr(bh))

    def _native_probe(self):
        """tools/libplugin_probe.so: the per-handle calls from NATIVE threads (no interpreter lock between the calls)"""
        if hasattr(self, "_probe"):
            return self._probe
        self._probe = None
        so = os.path.join(ROOT, "tools", "libplugin_probe.so")
        src = os.path.join(ROOT, "tools", "plugin_probe.cpp")
        try:
            if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
                # the tree may be read-only: a missing or stale harness is compiled into a temporary directory
                import tempfile
                so = os.path.join(tempfile.mkdtemp(prefix="b200_bench_"), "libplugin_probe.so")
                subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-pthread", "-o", so, src], check=True)
            C = self.C
            lib = C.CDLL(so)
            lib.plugin_probe_mul_relin.restype = C.c_double
            lib.plugin_probe_mul_relin.argtypes = [C.c_void_p] * 8 + [C.c_int, C.c_int, C.POINTER(C.c_long)]
            self._probe = lib
        except Exception:
            self._probe = None
        return self._probe

    def per_handle_native(self, threads, pairs):
        """seconds for `pairs` x (Evaluator_Multiply + Evaluator_Relinearize) from `threads` native threads, or None"""
        lib = self._native_probe()
        if lib is None:
            return None
        C = self.C
        fn = lambda name: C.cast(getattr(self.S.lib, name), C.c_void_p)
        err = C.c_long(0)
        secs = lib.plugin_probe_mul_relin(fn("Evaluator_Multiply"), fn("Evaluator_Relinearize"), self.O.ev, self._arr(self.pa[:pairs]),
                                          self._arr(self.pb[:pairs]), self._arr(self.pm[:pairs]), self._arr(self.pr[:pairs]), self.rlk,
                                          pairs, threads, C.byref(err))
        if err.value:
            raise RuntimeError("plugin call failed: HRESULT 0x%08x" % (err.value & 0xFFFFFFFF))
        return secs

    def per_handle_run(self, threads, pairs):
        S, O = self.S, self.O
        errs = []

        def work(tid):
            try:
                for i in range(tid, pairs, threads):
                    S.call("Evaluator_Multiply", O.ev, self.pa[i], self.pb[i], self.pm[i], None)
                    S.call("Evaluator_Relinearize", O.ev, self.pm[i], self.rlk, self.pr[i], None)
            except Exception as ex:
                errs.append(ex)

        ts = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        if errs:
            raise errs[0]

    def per_handle_check(self, out_dev, pairs):
        import torch
        ok = True
        for i in (0, pairs // 2, pairs - 1):
            w = self.O.ct_words(self.pr[i])
            ok = ok and bool(torch.equal(torch.from_numpy(w.view(self.np.int64)), out_dev[i].cpu()))
        return ok


def dump_outputs(directory, out, batch):
    """The words of a fixed, seeded sample of the batch's results as float64 (exact: every residue is below 2^53), with
    the batch indices they came from, so that two builds can be compared on identical inputs."""
    import numpy as np
    import torch
    items = np.sort(np.random.default_rng(0).choice(batch, size=min(DUMP_ITEMS, batch), replace=False))
    words = out[torch.from_numpy(items).to(out.device)].cpu().numpy()
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "mul_relin_out.npy"), words.astype(np.float64))
    np.save(os.path.join(directory, "mul_relin_out_items.npy"), items.astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--quick", action="store_true", help="device-resident loop + rooflines only (for runs under ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help=f"write a fixed sample of {DUMP_ITEMS} multiply+relinearize results of the last timed step to DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    from sunscreen_b200.lib import B200Context

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the B200 backend has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_node = None if os.environ.get("B200_BENCH_NO_NUMA") else bind_to_gpu_numa(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    ctx = B200Context(N_POLY, MODULI, PLAIN, device=local)
    k = ctx.k()
    n = N_POLY
    B = args.batch
    g = torch.Generator(device=dev)
    g.manual_seed(1234 + rank)

    def rand_rows(shape_prefix, mods):
        out = torch.empty(shape_prefix + (len(mods), n), dtype=torch.int64, device=dev)
        for i, m in enumerate(mods):
            out[..., i, :] = torch.randint(0, m, shape_prefix + (n,), generator=g, device=dev, dtype=torch.int64)
        return out

    a = rand_rows((B, 2), MODULI[:k])
    b = rand_rows((B, 2), MODULI[:k])
    rlk = rand_rows((k, 2), MODULI)
    out = torch.zeros((B, 2, k, n), dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    def step():
        ctx.multiply_relin(a, b, rlk, out, B, stream=stream)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()  # nvidia-smi needs ~0.2 s to come up: start it before the warm-up
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    # keep the GPU under the same load until the sampler is producing lines, then time
    t_wait = time.time()
    while rank == 0 and not sampler.samples and time.time() - t_wait < 3.0:
        step()
        torch.cuda.synchronize()
    sampler.mark = len(sampler.samples)
    l0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = ctx.launch_count() - l0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out, B)
    if dist is not None:
        tms = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms = float(tms.item())
    clocks = sampler.stop() if rank == 0 else None
    value = world * B * args.steps / (ms / 1000.0)

    ct_bytes = 2 * k * n * 8
    e2e_value = slab_value = ph_value = ph1_value = None
    if args.quick:
        quick_line = {"metric": "ciphertext mul+relin/sec", "value": value, "unit": "ops/s", "n_gpus": world, "steps": args.steps,
                      "ms_per_step": ms / args.steps, "gpu_launches": int(launches), "quick": True}
    else:
        # ---- e2e legs (host buffers; H2D + compute + D2H inside the timed region) ----
        ct_bytes = 2 * k * n * 8
        ah = torch.empty((B, 2, k, n), dtype=torch.int64).pin_memory()
        bh = torch.empty((B, 2, k, n), dtype=torch.int64).pin_memory()
        oh = torch.empty((B, 2, k, n), dtype=torch.int64).pin_memory()
        ah.copy_(a)
        bh.copy_(b)
        e2e_steps = max(2, min(args.steps, 5))

        def wall_max(seconds):
            if dist is None:
                return seconds
            ts = torch.tensor([seconds], device=dev, dtype=torch.float64)
            dist.all_reduce(ts, op=dist.ReduceOp.MAX)
            return float(ts.item())

        # the link's own ceiling for this box: one pinned 1 GiB copy each way (the e2e legs move 1 MiB in + 0.5 MiB out per op)
        link = {}
        for name, dst_t, src_t in (("h2d", a, ah), ("d2h", oh, out)):
            dst_t.copy_(src_t, non_blocking=True)
            barrier()  # every rank copies at the same time: GPUs that share a host link / PCIe switch share its bandwidth
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            for _ in range(2):
                dst_t.copy_(src_t, non_blocking=True)
            c1.record()
            torch.cuda.synchronize()
            link[name + "_gbs"] = 2 * dst_t.numel() * 8 / (c0.elapsed_time(c1) / 1000.0) / 1e9
            if dist is not None:
                tot = torch.tensor([link[name + "_gbs"]], device=dev, dtype=torch.float64)
                dist.all_reduce(tot, op=dist.ReduceOp.SUM)
                link[name + "_all_ranks_concurrent_gbs"] = float(tot.item())
        # both directions at once (what the e2e legs do), every rank at once
        s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
        barrier()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        with torch.cuda.stream(s_in):
            ev[0].record()
            for _ in range(2):
                a.copy_(ah, non_blocking=True)
            ev[1].record()
        with torch.cuda.stream(s_out):
            ev[2].record()
            for _ in range(2):
                oh.copy_(out, non_blocking=True)
            ev[3].record()
        torch.cuda.synchronize()
        link["bidir_h2d_gbs"] = 2 * a.numel() * 8 / (ev[0].elapsed_time(ev[1]) / 1000.0) / 1e9
        link["bidir_d2h_gbs"] = 2 * out.numel() * 8 / (ev[2].elapsed_time(ev[3]) / 1000.0) / 1e9
        ah.copy_(a)  # (a was only overwritten with its own contents; keep the pinned copy authoritative)
        # ceiling of the e2e legs (2 ct in, 1 ct out per op): each direction at its own rate with every rank copying, and both
        # together within what the host sustains when every rank moves data BOTH ways at once (on the 8-GPU node that sum is
        # ~49 GB/s per GPU against 54 + 40 one way: the host side, not the links, bounds the scaling of `e2e`)
        link["bound_ops_per_s"] = min(link["h2d_gbs"] * 1e9 / (2 * ct_bytes), link["d2h_gbs"] * 1e9 / ct_bytes,
                                      (link["bidir_h2d_gbs"] + link["bidir_d2h_gbs"]) * 1e9 / (3 * ct_bytes))

        # (a) layer-1 host-slab entry point
        ctx.multiply_relin_host(ah, bh, rlk, oh, B)  # warm
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            ctx.multiply_relin_host(ah, bh, rlk, oh, B)
        torch.cuda.synchronize()
        slab_s = wall_max(time.perf_counter() - t0)
        slab_value = world * B * e2e_steps / slab_s
        slab_same = bool(torch.equal(oh.to(dev), out))
        pack_num = 6 if (max(MODULI[:k]) < 2 ** 48 and os.environ.get("B200_HOST_PACK", "0") not in ("", "0")) else 8

        # (b) the plugin calls (SEAL-named C ABI): handles, batch seam, bulk word access
        os.environ["B200_DEVICE"] = str(local)  # the SEAL-named layer creates its own device context: same GPU as this rank
        plug = PluginLegs(ctx, local, k, n, rlk)
        oh.zero_()
        assert B % plug.chunk == 0, "batch must be a multiple of the e2e chunk"
        # the caller's host layout: per chunk, its first operands followed by its second operands (one transfer per chunk)
        abh = torch.empty((B // plug.chunk, 2, plug.chunk, 2, k, n), dtype=torch.int64).pin_memory()
        abh[:, 0].copy_(ah.view(B // plug.chunk, plug.chunk, 2, k, n))
        abh[:, 1].copy_(bh.view(B // plug.chunk, plug.chunk, 2, k, n))
        plug.batch_step(abh, oh, B)  # warm (allocates the handles' device buffers)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            plug.batch_step(abh, oh, B)
        plug_s = wall_max(time.perf_counter() - t0)
        e2e_value = world * B * e2e_steps / plug_s
        same = bool(torch.equal(oh.to(dev), out))
        # (c) per-handle calls from 8 threads, handles device-resident
        ph_threads = int(os.environ.get("B200_BENCH_PH_THREADS", "8"))
        ph_pairs = min(B, 1024)
        plug.per_handle_prepare(ah, bh, ph_pairs)
        plug.per_handle_run(ph_threads, ph_pairs)  # warm
        barrier()
        native = plug.per_handle_native(ph_threads, ph_pairs) is not None  # also warms the native harness
        ph_scaling = {}
        if native:
            barrier()
            for tcount in (1, 2, 4, 8, 16):
                for _ in range(3):  # warm: the batch shapes this thread count produces get their graphs instantiated here
                    plug.per_handle_native(tcount, ph_pairs)
                ph_scaling[str(tcount)] = ph_pairs / min(plug.per_handle_native(tcount, ph_pairs) for _ in range(3))
            barrier()
            plug.per_handle_native(ph_threads, ph_pairs)
            ph_s = wall_max(min(plug.per_handle_native(ph_threads, ph_pairs) for _ in range(3)))
            ph1_value = ph_scaling["1"]
        else:
            t0 = time.perf_counter()
            plug.per_handle_run(ph_threads, ph_pairs)
            ph_s = wall_max(time.perf_counter() - t0)
            t0 = time.perf_counter()
            plug.per_handle_run(1, min(ph_pairs, 64))
            ph1_value = min(ph_pairs, 64) / (time.perf_counter() - t0)
        ph_value = world * ph_pairs / ph_s
        ph_same = plug.per_handle_check(out, ph_pairs)

    # ---- north-star multi-GPU split (N > 1): rank 0 holds the whole batch, NCCL scatter -> compute -> NCCL gather ----
    sharded = None
    if dist is not None:
        Bt = B  # total pairs held by rank 0 (strong scaling: fixed total work)
        per = Bt // world
        a_loc = torch.empty((per, 2, k, n), dtype=torch.int64, device=dev)
        b_loc = torch.empty_like(a_loc)
        o_loc = torch.zeros_like(a_loc)
        gathered = [torch.empty_like(o_loc) for _ in range(world)] if rank == 0 else None
        a_chunks = list(a[: per * world].chunk(world)) if rank == 0 else None  # rank 0's own batch is the job
        b_chunks = list(b[: per * world].chunk(world)) if rank == 0 else None
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]

        def sharded_step():
            ev[0].record()
            dist.scatter(a_loc, a_chunks, src=0)
            dist.scatter(b_loc, b_chunks, src=0)
            ev[1].record()
            ctx.multiply_relin(a_loc, b_loc, rlk_shared, o_loc, per, stream=stream)
            ev[2].record()
            dist.gather(o_loc, gathered, dst=0)
            ev[3].record()

        # every rank needs rank 0's relinearization key (replicated once, outside the timed region)
        rlk_shared = rlk.clone()
        dist.broadcast(rlk_shared, src=0)
        for _ in range(2):
            sharded_step()
        barrier()
        reps_s = max(2, min(args.steps, 5))
        phase = torch.zeros(4, dtype=torch.float64, device=dev)
        for _ in range(reps_s):
            barrier()
            sharded_step()
            torch.cuda.synchronize()
            phase += torch.tensor([ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[2].elapsed_time(ev[3]),
                                   ev[0].elapsed_time(ev[3])], dtype=torch.float64, device=dev)
        phase /= reps_s
        dist.all_reduce(phase, op=dist.ReduceOp.MAX)
        ok = None
        if rank == 0:
            whole = torch.cat(gathered)
            ok = bool(torch.equal(whole, out[: per * world]))  # `out` = the same pairs computed on one GPU (timed loop above)
        sc_ms, comp_ms, ga_ms, tot_ms = (float(x) for x in phase.tolist())
        moved_out = (world - 1) * per * 2 * ct_bytes  # bytes leaving rank 0 in the scatter
        moved_in = (world - 1) * per * ct_bytes
        sharded = {"scaling": "strong", "total_pairs": per * world, "scatter_ms": sc_ms, "compute_ms": comp_ms, "gather_ms": ga_ms,
                   "total_ms": tot_ms, "ops_per_s": per * world / (tot_ms / 1000.0),
                   "ops_per_s_compute_only": per * world / (comp_ms / 1000.0),
                   "scatter_gbs_out_of_rank0": moved_out / (sc_ms / 1000.0) / 1e9 if sc_ms else None,
                   "gather_gbs_into_rank0": moved_in / (ga_ms / 1000.0) / 1e9 if ga_ms else None,
                   "equals_one_gpu_words": ok, "timing": "CUDA events per phase, max over ranks, mean of %d steps" % reps_s,
                   "collectives": "torch.distributed scatter x2 / gather (NCCL over NVLink), none inside the compute"}

    # ---- roofline of the dominant kernel: batched forward NTT, 4096 polys x 4 residues (1 GiB slab > L2) ----
    roof = None
    roof_ks = None
    cpu = None
    if rank == 0:
        peak, peak_src = peaks()
        slab = rand_rows((NTT_POLYS,), MODULI[:k])
        for _ in range(3):
            ctx.ntt_forward(slab, NTT_POLYS, stream=stream)
            ctx.ntt_inverse(slab, NTT_POLYS, stream=stream)
        torch.cuda.synchronize()
        reps = 10
        ef0, ef1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        fwd_ms = 0.0
        inv_ms = 0.0
        for _ in range(reps):
            ef0.record()
            ctx.ntt_forward(slab, NTT_POLYS, stream=stream)
            ef1.record()
            torch.cuda.synchronize()
            fwd_ms += ef0.elapsed_time(ef1)
            ef0.record()
            ctx.ntt_inverse(slab, NTT_POLYS, stream=stream)
            ef1.record()
            torch.cuda.synchronize()
            inv_ms += ef0.elapsed_time(ef1)
        fwd_ms /= reps
        inv_ms /= reps
        alg_bytes = 16 * n * NTT_POLYS * k  # SURVEY.md 8(d): 16*n bytes per residue NTT
        achieved = alg_bytes / (fwd_ms / 1000.0) / 1e9
        traffic = None
        tf = os.path.join(ROOT, "profiles", "ntt_traffic.json")
        if os.path.exists(tf):
            try:
                traffic = json.load(open(tf)).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        roof = {"bound": "hbm", "kernel": "ntt_fp_kernel<13, fwd, 256> (4096 polys x 4 residues, n=8192; FP64 butterflies)", "achieved": achieved,
                "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "algorithmic_bytes_per_launch": alg_bytes, "fwd_ms": fwd_ms, "inv_ms": inv_ms,
                "inverse_achieved": alg_bytes / (inv_ms / 1000.0) / 1e9,
                "mul_relin_algorithmic_gbs": (8 * n * k * 6) * value / world / 1e9}
        del slab
        # key switch (relinearize 3 -> 2 over the batch): digit NTTs + inner product against the key + inverse NTTs + mod-down.
        # algorithmic bytes (SURVEY.md 8(d)): 8nk*5 per item + the key once per batch
        c3 = rand_rows((B, 3), MODULI[:k])
        o2 = torch.zeros((B, 2, k, n), dtype=torch.int64, device=dev)
        for _ in range(3):
            ctx.relinearize(c3, rlk, o2, B, stream=stream)
        torch.cuda.synchronize()
        ks_ms = 0.0
        for _ in range(reps):
            ef0.record()
            ctx.relinearize(c3, rlk, o2, B, stream=stream)
            ef1.record()
            torch.cuda.synchronize()
            ks_ms += ef0.elapsed_time(ef1)
        ks_ms /= reps
        ks_bytes = 8 * n * k * 5 * B + 16 * n * k * (k + 1)
        roof_ks = {"bound": "hbm", "kernel": "relinearize = ntt_fp_kernel<fwd> (k(k+1) digit rows) + ksmac + ntt_fp_kernel<inv> + ksmoddown",
                   "achieved": ks_bytes / (ks_ms / 1000.0) / 1e9, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                   "frac": ks_bytes / (ks_ms / 1000.0) / 1e9 / peak, "ms_per_batch": ks_ms, "batch": B,
                   "algorithmic_bytes_per_launch": ks_bytes, "ops_per_s": B / (ks_ms / 1000.0),
                   "note": "the key switch is bound by its 30 transforms per item (FP64 pipe), not by HBM: see DESIGN.md"}
        del c3, o2
        if not args.no_cpu and world == 1:  # the CPU baseline is an N=1 leg (the reference arm covers every N)
            try:
                try:
                    os.sched_setaffinity(0, range(os.cpu_count() or 1))
                except Exception:
                    pass
                quota = cpu_quota()
                cores = os.cpu_count() or 1
                iters = 32 if (quota["effective_cores"] or cores) >= 32 else 8
                rate, secs = cpu_reference_rate(cores, iters)
                rate1, secs1 = cpu_reference_rate(1, 16)
                cpu = {"value": rate, "unit": "ops/s", "cores": cores, "kind": "reference",
                       "sample": f"{cores} threads x {iters} multiply+relinearize_inplace (uniform-random words), {secs:.2f}s",
                       "single_thread_ops_per_s": rate1,
                       # a CPU-quota'd lease shows up here: threads >> the cores' worth of time the box grants
                       "box": quota, "parallel_speedup_over_one_thread": rate / rate1 if rate1 else None,
                       "build": "unmodified reference sources, -O3, Intel HEXL off (not buildable offline), one MemoryPool per thread",
                       "full_node_reference": "the same arm on an 8-GPU lease (96-core cgroup quota, 128 threads): 3654 ops/s (profiles/r2_bench_reference_arm_fullnode.json)"}
            except Exception as ex:  # reference .so missing on this box
                cpu = {"value": None, "unit": "ops/s", "cores": os.cpu_count(), "kind": "reference",
                       "sample": f"unavailable: {ex}"}

    if rank == 0 and args.quick:
        quick_line.update({"roofline": roof, "roofline_keyswitch": roof_ks, "sharded": sharded, "clocks": clocks})
        print(json.dumps(quick_line))
    elif rank == 0:
        line = {
            "metric": "ciphertext mul+relin/sec", "value": value, "unit": "ops/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": "Evaluator::multiply + relinearize, n=8192, BFVDefault 218-bit chain (k=4 + special), "
                                   f"batch={B} ct pairs per GPU", "batch_per_gpu": B,
                       "parallelism": f"batch sharded over {world} GPU(s), no data-path collective",
                       "l2": "inputs (1 GiB per GPU) exceed the 126 MB L2; no explicit flush"},
            "clocks": clocks, "gpu_launches": int(launches),
            "e2e": {"value": e2e_value, "unit": "ops/s",
                    "path": "pinned host words -> B200_Ciphertext_SetWordsBatch -> B200_Evaluator_MultiplyRelinBatch -> "
                            "B200_Ciphertext_GetWordsBatch -> pinned host words (SEAL-named plugin ABI, include/b200_sealc.h)",
                    "h2d_bytes_per_step": 2 * B * ct_bytes, "d2h_bytes_per_step": B * ct_bytes,
                    "threads": plug.threads, "chunk_pairs": plug.chunk, "steps": e2e_steps, "matches_device_path": same,
                    "host_numa_node": numa_node, "pcie_gbs": 3 * B * ct_bytes * e2e_steps / plug_s / 1e9,
                    "roofline": {"bound": "pcie", "h2d_peak_gbs": link["h2d_gbs"], "d2h_peak_gbs": link["d2h_gbs"],
                                 "bidirectional_h2d_gbs": link["bidir_h2d_gbs"], "bidirectional_d2h_gbs": link["bidir_d2h_gbs"],
                                 "bound_ops_per_s_per_gpu": link["bound_ops_per_s"],
                                 "h2d_all_ranks_concurrent_gbs": link.get("h2d_all_ranks_concurrent_gbs"),
                                 "d2h_all_ranks_concurrent_gbs": link.get("d2h_all_ranks_concurrent_gbs"),
                                 "frac": e2e_value / world / link["bound_ops_per_s"],
                                 "note": "1 MiB in + 0.5 MiB out per multiply+relinearize: the end-to-end rate is the host link's, not the kernels'; the peaks are measured with every rank copying at once; bound = min(H2D alone / 1 MiB, D2H alone / 0.5 MiB, (H2D + D2H with both directions busy) / 1.5 MiB)"}},
            "e2e_host_slab": {"value": slab_value, "unit": "ops/s", "path": "b200_multiply_relin_host (layer-1 C ABI, include/b200_bfv.h)",
                              "h2d_bytes_per_step": 2 * B * ct_bytes * pack_num // 8, "d2h_bytes_per_step": B * ct_bytes * pack_num // 8,
                              "transfer": "6-byte packed residues" if pack_num == 6 else "8-byte words",
                              "matches_device_path": slab_same},
            "plugin_per_handle": {"value": ph_value, "unit": "ops/s", "threads": ph_threads, "pairs": ph_pairs,
                                  "path": "Evaluator_Multiply + Evaluator_Relinearize per handle (device-resident handles; what "
                                          "unmodified sunscreen_runtime issues, run.rs:243,279)",
                                  "one_thread_ops_per_s": ph1_value, "matches_device_path": ph_same,
                                  "driver": "native threads (tools/plugin_probe.cpp)" if native else "python threads (ctypes)",
                                  "ops_per_s_by_threads": ph_scaling or None,
                                  "combining": "concurrent calls of one kind run as one batched launch sequence (sealc_api.cpp: combine_submit)"},
            "roofline": roof, "roofline_keyswitch": roof_ks, "cpu_baseline": cpu, "sharded": sharded,
        }
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
