#!/usr/bin/env python
"""bench.py -- BASELINE.json configs[1]: Take + Cast(float64->float32) + Add over 1B rows per
GPU, null_probability 0.1, as three CallFunction-equivalent calls through the C-ABI:

    out = add(cast(take(values, indices), float32), other)

One "step" = one pass of that pipeline over one synthetic batch.
  value : rows/s, inputs already resident in HBM (device-timed with CUDA events, max over ranks)
  e2e   : rows/s through the same public calls starting from pinned HOST buffers, H2D of all
          inputs and D2H of the result column inside the timed region
  roofline : the dominant kernel (take_kernel, random int64 indices into float64), algorithmic
          bytes (SURVEY.md section 8d: 24.25 B/row) / its CUDA-event time, against the measured copy peak
  configs  : (N = 1) the other BASELINE.json configs at full size -- c1 filter, c3 group-by (fused and
          Grouper + aggregators), c4 sort_indices (wide / narrow keys), c5 utf8 filter + dictionary take --
          each {ms, alg_bytes, frac, parity_checksum_ok}
  multi_gpu: configs[2] and configs[3] with the row range sharded over the N ranks (STRONG scaling: the
          total is fixed at --rows): local pass -> one exchange (b2_comm_*: NCCL all-to-all-v over NVLink,
          csrc/comm.cu) -> owner-side merge, CUDA-event timed, max over ranks, with checksums that are
          identical at every N and are verified against invariants derived from the inputs
  cpu_baseline / --impl reference : the reference's own CPU kernels (oracle/_ref/ref_bench: a C++ harness
          linked against the installed libarrow_compute.so.2400, the same kernels as /root/reference for
          this path) on the host cores.
Multi-GPU (config 2): rows shard by range, `values` replicated per GPU (SURVEY section 8e), no collective on
the data path => weak scaling, one process per GPU.
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

ALG_TAKE, ALG_CAST, ALG_ADD = 24.25, 12.25, 12.375  # bytes/row, SURVEY section 8d
ALG_PIPELINE = ALG_TAKE + ALG_CAST + ALG_ADD          # 48.875
NULL_P = 0.1
SEED = 0x0FF1CE
REF_BENCH = os.path.join(ROOT, "oracle", "_ref", "ref_bench")


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], threading.Event()
        # NVML is initialised HERE, before the timed region: nvmlInit can take longer than the whole ~150 ms region, which
        # once left a run with a single sample
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = (pynvml, pynvml.nvmlDeviceGetHandleByIndex(index))
        except Exception:
            self._nvml = None

    def run(self):
        # NVML in-process (same counters nvidia-smi prints, but every 10 ms: the device-resident timed region
        # is < 200 ms long); the nvidia-smi subprocess loop is the fallback
        try:
            self._nvml_loop()
        except Exception:
            self._smi_loop()

    def _nvml_loop(self):
        if self._nvml is None:
            raise RuntimeError("NVML unavailable")
        pynvml, h = self._nvml
        mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
        reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
        bits = [0x8, 0x40, 0x20, 0x4]  # hw_slowdown, hw_thermal_slowdown, sw_thermal_slowdown, sw_power_cap (nvml.h)
        while not self.stop_flag.is_set():
            sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
            r = int(reasons(h))
            self.samples.append([str(sm), str(mx)] + ["Active" if r & b else "Not Active" for b in bits])
            self.stop_flag.wait(0.01)

    def _smi_loop(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        sm = sorted(int(s[0]) for s in self.samples if s and s[0].isdigit())
        mx = [int(s[1]) for s in self.samples if len(s) > 1 and s[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for s in self.samples for n, v in zip(names, s[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's own CPU kernels on the host cores
# ------------------------------------------------------------------------------------------------
def host_info():
    model = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    avail = 0
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable"):
                avail = int(line.split()[1]) * 1024
    except Exception:
        pass
    return model, os.cpu_count() or 1, avail


def ref_bench(op, rows, steps, warmup, threads, groups=None, timeout=900):
    """Runs oracle/_ref/ref_bench (C++, linked against libarrow_compute.so.2400) and returns its JSON."""
    if not os.path.exists(REF_BENCH):
        raise RuntimeError(f"{REF_BENCH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
    cmd = [REF_BENCH, op, str(int(rows)), str(int(steps)), str(int(warmup)), str(int(threads))]
    if groups:
        cmd.append(str(int(groups)))
    def all_cpus():  # the GPU arm pinned this process to its GPU's NUMA node: the CPU arm gets every host thread back
        try:
            os.sched_setaffinity(0, range(os.cpu_count() or 1))
        except Exception:
            pass
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, preexec_fn=all_cpus)
    if out.returncode != 0:
        raise RuntimeError(f"ref_bench failed: {out.stderr[-500:]}")
    return json.loads(out.stdout.strip().splitlines()[-1])


def reference_rows(requested):
    """The CPU arm runs the SAME row count as the GPU arm when host RAM allows (the pipeline needs
    ~40 B/row of host memory), otherwise the largest power-of-two sample that fits (>= 2^28 wanted)."""
    _, _, avail = host_info()
    rows = requested
    while rows * 44 > 0.6 * avail and rows > (1 << 22):
        rows //= 2
    return rows


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    model, cores, avail = host_info()
    rows = reference_rows(args.rows)
    r = ref_bench("pipeline", rows, args.steps, args.warmup, cores)
    rate = r["rows_per_s_mean"]
    line = {
        "impl": "reference", "metric": "rows/sec", "value": rate, "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["mean_s"] * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64->f32", "data": "synthetic",
        "config": {"workload": "Take(float64,int64 idx)+Cast(float64->float32)+Add(float32), null_probability=0.1, 1B rows/GPU"
                   if rows == 1_000_000_000 else f"Take+Cast(f64->f32)+Add, null_probability=0.1, {rows} rows",
                   "rows_per_step": rows, "same_rows_as_gpu_arm": rows == args.rows,
                   "note": "reference CPU kernels (libarrow_compute.so.2400) through arrow::compute::CallFunction, one row-range slice per host thread"},
        "cpu_baseline": {"value": rate, "unit": "rows/s", "cores": cores, "kind": "reference", "cpu_model": model,
                         "best_rows_per_s": r["rows_per_s_best"],
                         "sample": f"{rows} rows/step x {args.steps} steps (+{args.warmup} warm-up), oracle/_ref/ref_bench pipeline, "
                                   f"arrow {r['arrow_version']}, {cores} row-range threads"},
        "e2e": {"value": rate, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_leg(args):
    """rank 0, N = 1: the reference pipeline on all host cores (same rows as the GPU arm when RAM allows,
    2 timed passes) and on one thread (2^26-row sample) -- a bounded ~10-30 s of CPU work."""
    model, cores, _ = host_info()
    rows = reference_rows(args.rows)
    out = {"unit": "rows/s", "cores": cores, "kind": "reference", "cpu_model": model}
    try:
        allc = ref_bench("pipeline", rows, 2, 1, cores)
        one = ref_bench("pipeline", min(rows, 1 << 26), 1, 1, 1)
        out.update({"value": allc["rows_per_s_best"], "single_thread_value": one["rows_per_s_best"],
                    "sample": f"all cores: {rows} rows x best of 2 (+1 warm-up); single thread: {min(rows, 1 << 26)} rows x 1 (+1 warm-up); "
                              f"oracle/_ref/ref_bench pipeline, arrow {allc['arrow_version']}"})
    except Exception as e:  # the baseline is a reported number, not a gate: never lose the GPU line over it
        out.update({"value": None, "error": str(e)[:300], "sample": "ref_bench failed"})
    return out


# ------------------------------------------------------------------------------------------------
# helpers (torch is plumbing here: synthetic inputs, events, verification arithmetic)
# ------------------------------------------------------------------------------------------------
def pack_bits(torch, valid):
    """bool[n] (n % 8 == 0) -> LSB-first bitmap bytes"""
    w = torch.tensor([1, 2, 4, 8, 16, 32, 64, 128], dtype=torch.uint8, device=valid.device)
    return (valid.view(-1, 8).to(torch.uint8) * w).sum(dim=1, dtype=torch.uint8)


def make_validity(torch, n, gen, null_p=NULL_P):
    out = torch.empty((n + 7) // 8 + 64, dtype=torch.uint8, device="cuda")
    out.zero_()
    chunk = 1 << 27
    nulls = 0
    for lo in range(0, n, chunk):
        m = min(chunk, n - lo)
        m8 = (m + 7) // 8 * 8
        v = torch.rand(m8, device="cuda", generator=gen) >= null_p
        if m8 != m:
            v[m:] = False
        nulls += int(m - v[:m].sum().item())
        out[lo // 8: lo // 8 + m8 // 8] = pack_bits(torch, v)
        del v
    return out, nulls


def make_mask(torch, n, gen, sel):
    m8 = (n + 7) // 8 * 8
    bits = torch.zeros(m8 // 8 + 64, dtype=torch.uint8, device="cuda")
    chunk = 1 << 27
    for lo in range(0, m8, chunk):
        m = min(chunk, m8 - lo)
        bits[lo // 8:(lo + m) // 8] = pack_bits(torch, torch.rand(m, device="cuda", generator=gen) < sel)
    return bits


def make_word_column(torch, gen, m, vocab):
    """m strings drawn from `vocab` distinct words of 8..16 bytes (large_utf8 layout: int64 offsets + bytes); word k = the 5
    base-26 digits of k followed by a k-dependent tail, so a key string decodes back to k.  Returns (k per row, offsets, bytes, total)"""
    I64 = torch.int64
    kid = torch.randint(0, vocab, (m,), dtype=I64, device="cuda", generator=gen)
    lens = 8 + (kid * 7) % 9
    offs = torch.zeros(m + 1, dtype=I64, device="cuda")
    torch.cumsum(lens, 0, out=offs[1:])
    total = int(offs[-1].item())
    data = torch.empty(total + 64, dtype=torch.uint8, device="cuda")
    cs = 1 << 24
    for lo in range(0, m, cs):
        hi = min(m, lo + cs)
        ln = lens[lo:hi]
        b0, b1 = int(offs[lo].item()), int(offs[hi].item())
        kk = torch.repeat_interleave(kid[lo:hi], ln)
        j = torch.arange(b0, b1, device="cuda", dtype=I64) - torch.repeat_interleave(offs[lo:hi], ln)
        head = (kk // torch.pow(26, 4 - j.clamp(max=4))) % 26
        digit = torch.where(j < 5, head, (kk * 31 + j * 7) % 26)
        data[b0:b1] = (97 + digit).to(torch.uint8)
        del kk, j, head, digit, ln
    return kid, offs, data, total


def unpack_bits(torch, bits, n):
    """LSB-first bitmap bytes -> bool[n] (verification only)"""
    sh = torch.arange(8, device=bits.device, dtype=torch.uint8)
    return ((bits[: (n + 7) // 8].unsqueeze(1) >> sh) & 1).reshape(-1)[:n].bool()


def mix64(torch, x):
    """murmur3 fmix64 on int64 tensors (wrap-around arithmetic; logical shifts emulated)"""
    def lsr(v, s):
        return (v >> s) & ((1 << (64 - s)) - 1)
    x = x ^ lsr(x, 33)
    x = x * -49064778989728563            # 0xff51afd7ed558ccd
    x = x ^ lsr(x, 33)
    x = x * -4265267296055464877          # 0xc4ceb9fe1a85ec53
    return x ^ lsr(x, 33)


def bind_to_gpu_numa(local):
    """Pin this rank's CPU threads (and therefore its first-touch / pinned allocations) to the NUMA node
    its GPU hangs off: 8 ranks pulling 20 GB/step of pinned H2D through the wrong socket cost the e2e leg
    30 % at N = 8 in round 1.  Best effort, silent when sysfs does not say."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        dom, rest = bus.split(":", 1)
        path = f"/sys/bus/pci/devices/{dom[-4:].lower()}:{rest.lower()}/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.extend(range(int(a), int(b or a) + 1))
        allowed = set(os.sched_getaffinity(0)) & set(cpus)
        if allowed:
            os.sched_setaffinity(0, allowed)
        return node
    except Exception:
        return None


class Env:
    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.args = torch, dist, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.numa = bind_to_gpu_numa(self.local)
        torch.cuda.set_device(self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        from arrow_b200 import Context, _cabi
        self.ctx = Context.get(self.local)
        # a real (non-NULL) stream: the C-ABI treats stream 0 as "use the context's own stream", and
        # torch.cuda.Event only times the stream it is recorded on
        self.stream = torch.cuda.Stream()
        torch.cuda.set_stream(self.stream)
        assert self.stream.cuda_stream != 0
        self.ctx.stream = self.stream.cuda_stream  # all C-ABI calls are ordered on torch's current stream
        self.lib = _cabi.lib()

    def sync_all(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, ms):
        if self.world == 1:
            return ms
        t = self.torch.tensor([ms], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, ints):
        t = self.torch.tensor([int(x) for x in ints], dtype=self.torch.int64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return [int(x) for x in t.tolist()]

    def timed(self, fn, reps, warmup=1):
        torch = self.torch
        for _ in range(warmup):
            r = fn()
            del r
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(self.stream)
        for _ in range(reps):
            r = fn()
            del r
        b.record(self.stream)
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps


# ------------------------------------------------------------------------------------------------
# configs[0,2,3,4] at full size on one GPU (the `configs` array of the bench line)
# ------------------------------------------------------------------------------------------------
def run_configs(env, n):
    import pyarrow as pa

    import arrow_b200.compute as bc
    from arrow_b200 import DeviceArray
    torch, ctx = env.torch, env.ctx
    peak, _ = measured_peaks()
    gen = torch.Generator(device="cuda")
    gen.manual_seed(SEED + 17)
    out = []
    reps = 3
    I64 = torch.int64

    def entry(name, rows, ms, alg_bytes, ok, **extra):
        gbs = alg_bytes / (ms * 1e-3) / 1e9
        e = {"name": name, "rows": rows, "ms": ms, "rows_per_s": rows / (ms * 1e-3), "alg_bytes": alg_bytes, "gbs": gbs,
             "frac": gbs / peak, "parity_checksum_ok": bool(ok)}
        e.update(extra)
        out.append(e)

    # ---- c1: Filter(int64 values null_p 0.1, bool mask s = 0.5), DROP ----
    vals_t = torch.randint(-100, 101, (n,), dtype=I64, device="cuda", generator=gen)
    vvalid_t, v_nulls = make_validity(torch, n, gen)
    values = DeviceArray.from_pointers(ctx, pa.int64(), n, vals_t.data_ptr(), validity_ptr=vvalid_t.data_ptr(), null_count=v_nulls)
    mask_bits = make_mask(torch, n, gen, 0.5)
    mask = DeviceArray.from_pointers(ctx, pa.bool_(), n, mask_bits.data_ptr())
    ms = env.timed(lambda: bc.filter(values, mask), reps)
    res = bc.filter(values, mask)
    # parity: length = popcount(mask); order-sensitive checksum of the kept values and their validity
    ok = True
    kept = 0
    chk_got = chk_want = 0
    pos = 0
    ov = unpack_bits(torch, torch.as_tensor(_view(res.buffers[0].ptr, (res.length + 7) // 8, "|u1", res), device="cuda"), res.length) \
        if res.buffers[0] is not None else None
    od = torch.as_tensor(_view(res.buffers[1].ptr, res.length, "<i8", res), device="cuda")
    chunk = 1 << 27
    for lo in range(0, n, chunk):
        m = min(chunk, n - lo)
        sel = unpack_bits(torch, mask_bits[lo // 8:], m)
        vv = unpack_bits(torch, vvalid_t[lo // 8:], m)
        k = int(sel.sum().item())
        want_v, want_ok = vals_t[lo:lo + m][sel], vv[sel]
        got_v = od[pos:pos + k]
        got_ok = ov[pos:pos + k] if ov is not None else torch.ones(k, dtype=torch.bool, device="cuda")
        w = torch.arange(pos + 1, pos + k + 1, dtype=I64, device="cuda")
        chk_want += int(((want_v * want_ok) * w).sum().item()) + int((want_ok * w).sum().item())
        chk_got += int(((got_v * got_ok) * w).sum().item()) + int((got_ok * w).sum().item())
        pos += k
        kept += k
        del sel, vv, want_v, want_ok, w
    ok = kept == res.length and (chk_got - chk_want) % (1 << 64) == 0
    entry("c1 filter int64 (values null_p 0.1, mask s=0.5, DROP)", n, ms, n * (8 + 0.125 + 0.125) + res.length * 8.125, ok,
          selectivity=res.length / n)
    del res, od, ov, mask, mask_bits, values, vals_t, vvalid_t
    ctx.trim()
    torch.cuda.empty_cache()

    # ---- c3: group-by sum + count, int64 key (10M groups), int64 value null_p 0.1 ----
    groups = 10_000_000 if n >= 100_000_000 else max(1000, n // 100)
    keys_t = torch.randint(0, groups, (n,), dtype=I64, device="cuda", generator=gen)
    vals_t = torch.randint(-100, 101, (n,), dtype=I64, device="cuda", generator=gen)
    vvalid_t, v_nulls = make_validity(torch, n, gen)
    keys = DeviceArray.from_pointers(ctx, pa.int64(), n, keys_t.data_ptr())
    vals = DeviceArray.from_pointers(ctx, pa.int64(), n, vals_t.data_ptr(), validity_ptr=vvalid_t.data_ptr(), null_count=v_nulls)

    paths = {}

    def fused():
        g = bc.GroupBySumCount(pa.int64(), pa.int64(), expected_groups=groups, ctx=ctx)
        g.consume(keys, vals)
        paths["counts"] = g.path_counts()
        return g.finalize()

    def unfused():
        return bc.group_by([keys], [("hash_sum", vals, None), ("hash_count", vals, None)], fused=False)

    # the independent answer: torch index_add_ / bincount on the same device columns
    want_cnt = torch.zeros(groups, dtype=I64, device="cuda")
    want_sum = torch.zeros(groups, dtype=I64, device="cuda")
    want_rows = torch.zeros(groups, dtype=I64, device="cuda")
    for lo in range(0, n, chunk):
        m = min(chunk, n - lo)
        vv = unpack_bits(torch, vvalid_t[lo // 8:], m).to(I64)
        kk = keys_t[lo:lo + m]
        want_cnt.index_add_(0, kk, vv)
        want_sum.index_add_(0, kk, vals_t[lo:lo + m] * vv)
        want_rows.index_add_(0, kk, torch.ones_like(vv))
        del vv
    present = want_rows > 0

    def check_groups(k, s, c):
        kt = torch.as_tensor(_view(k.buffers[1].ptr, k.length, "<i8", k), device="cuda")
        st = torch.as_tensor(_view(s.buffers[1].ptr, s.length, "<i8", s), device="cuda")
        ct = torch.as_tensor(_view(c.buffers[1].ptr, c.length, "<i8", c), device="cuda")
        if k.length != int(present.sum().item()) or k.null_count != 0:
            return False
        seen = torch.zeros(groups, dtype=torch.bool, device="cuda")
        seen[kt] = True
        if int(seen.sum().item()) != k.length:       # every key exactly once
            return False
        if not bool((ct == want_cnt[kt]).all().item()):
            return False
        nz = ct > 0
        if not bool((st[nz] == want_sum[kt][nz]).all().item()):
            return False
        return s.null_count == int((~nz).sum().item())

    ms = env.timed(fused, reps)
    k, s, c = fused()
    ng = k.length
    ok = check_groups(k, s, c)
    del k, s, c
    entry("c3 group-by hash_sum+hash_count int64 key, 10M groups (fused b2_groupby_sumcount)", n, ms, n * 16.125 + ng * 24.25, ok, groups=ng,
          paths=paths.get("counts"))
    ms = env.timed(unfused, 2)
    (ku,), (su, cu) = unfused()
    ok = check_groups(ku, su, cu)
    del ku, su, cu
    entry("c3 group-by via Grouper + 2 HashAggregators (the reference API shape)", n, ms, n * 16.125 + ng * 24.25, ok, groups=ng)
    del keys, vals, keys_t, vals_t, vvalid_t, want_cnt, want_sum, want_rows, present
    ctx.trim()
    torch.cuda.empty_cache()

    # ---- c3u: group-by sum + count with a large_utf8 KEY (north_star: hash-aggregate over utf8 columns) ----
    # n/2 strings drawn from a vocabulary of 1M words of 8..16 bytes; word k = the 5 base-26 digits of k + a k-dependent
    # tail, so the result's key strings can be decoded back to k on the device and checked against index_add_
    m = n // 2
    vocab = 1_000_000 if m >= 10_000_000 else max(100, m // 100)
    kid, offs, data, total = make_word_column(torch, gen, m, vocab)
    vals_t = torch.randint(-100, 101, (m,), dtype=I64, device="cuda", generator=gen)
    vvalid_t, v_nulls = make_validity(torch, m, gen)
    skeys = DeviceArray.from_pointers(ctx, pa.large_string(), m, offs.data_ptr(), data2_ptr=data.data_ptr())
    vals = DeviceArray.from_pointers(ctx, pa.int64(), m, vals_t.data_ptr(), validity_ptr=vvalid_t.data_ptr(), null_count=v_nulls)

    def string_group_by():
        return bc.group_by([skeys], [("hash_sum", vals, None), ("hash_count", vals, None)], fused=False)
    ms = env.timed(string_group_by, 2)
    (ku,), (su, cu) = string_group_by()
    want_cnt = torch.zeros(vocab, dtype=I64, device="cuda")
    want_sum = torch.zeros(vocab, dtype=I64, device="cuda")
    want_rows = torch.zeros(vocab, dtype=I64, device="cuda")
    for lo in range(0, m, chunk):
        hi = min(m, lo + chunk)
        vv = unpack_bits(torch, vvalid_t[lo // 8:], hi - lo).to(I64)
        want_cnt.index_add_(0, kid[lo:hi], vv)
        want_sum.index_add_(0, kid[lo:hi], vals_t[lo:hi] * vv)
        want_rows.index_add_(0, kid[lo:hi], torch.ones_like(vv))
        del vv
    ng = ku.length
    ko = torch.as_tensor(_view(ku.buffers[1].ptr, ng + 1, "<i8", ku), device="cuda")
    kb = torch.as_tensor(_view(ku.buffers[2].ptr, int(ko[-1].item()) if ng else 0, "|u1", ku), device="cuda")
    dec = torch.zeros(ng, dtype=I64, device="cuda")
    for j in range(5):
        dec = dec * 26 + (kb[ko[:-1] + j].to(I64) - 97)
    st = torch.as_tensor(_view(su.buffers[1].ptr, ng, "<i8", su), device="cuda")
    ct = torch.as_tensor(_view(cu.buffers[1].ptr, ng, "<i8", cu), device="cuda")
    ok = ng == int((want_rows > 0).sum().item()) and ku.null_count == 0
    ok = ok and int(torch.unique(dec).numel()) == ng and bool(((ko[1:] - ko[:-1]) == 8 + (dec * 7) % 9).all().item())
    ok = ok and bool((ct == want_cnt[dec]).all().item())
    nz = ct > 0
    ok = ok and bool((st[nz] == want_sum[dec][nz]).all().item()) and su.null_count == int((~nz).sum().item())
    L = total / m
    entry("c3 group-by hash_sum+hash_count, large_utf8 key (1M distinct words of 8-16 B; string Grouper + 2 HashAggregators)", m, ms,
          m * (8 + L + 8.125) + ng * (8 + L + 16.25), ok, groups=ng, mean_len=L)
    del ku, su, cu, ko, kb, dec, st, ct, skeys, vals, kid, offs, data, vals_t, vvalid_t, want_cnt, want_sum, want_rows
    ctx.trim()
    torch.cuda.empty_cache()

    # ---- c4: SortIndices int64 + validity ----
    m = n
    for name, lo_v, hi_v in (("wide [-2^62,2^62)", -2**62, 2**62), ("narrow [0,4095]", 0, 4096)):
        keys_t = torch.randint(lo_v, hi_v, (m,), dtype=I64, device="cuda", generator=gen)
        kvalid_t, k_nulls = make_validity(torch, m, gen)
        keys = DeviceArray.from_pointers(ctx, pa.int64(), m, keys_t.data_ptr(), validity_ptr=kvalid_t.data_ptr(), null_count=k_nulls)
        ms = env.timed(lambda: bc.array_sort_indices(keys), 2)
        idx = bc.array_sort_indices(keys)
        it = torch.as_tensor(_view(idx.buffers[1].ptr, m, "<i8", idx), device="cuda")
        nv = m - k_nulls
        # stable permutation, keys non-decreasing with ties in index order, nulls last in index order
        ok = True
        prev_k = prev_i = None
        for lo in range(0, nv, chunk):
            hi = min(nv, lo + chunk)
            sk, si = keys_t[it[lo:hi]], it[lo:hi]
            good = (sk[1:] > sk[:-1]) | ((sk[1:] == sk[:-1]) & (si[1:] > si[:-1]))
            ok = ok and bool(good.all().item())
            if prev_k is not None:
                ok = ok and (int(sk[0]) > prev_k or (int(sk[0]) == prev_k and int(si[0]) > prev_i))
            prev_k, prev_i = int(sk[-1]), int(si[-1])
            del sk, si, good
        if k_nulls:
            ni = it[nv:]
            ok = ok and bool((ni[1:] > ni[:-1]).all().item())
            ok = ok and not bool(unpack_bits(torch, kvalid_t, m)[ni].any().item())
        ok = ok and (int(it.sum().item()) - m * (m - 1) // 2) % (1 << 64) == 0
        entry(f"c4 sort_indices int64 {name}, null_p 0.1", m, ms, m * 16.125, ok)
        del keys, keys_t, kvalid_t, idx, it
        ctx.trim()
        torch.cuda.empty_cache()

    # ---- c5: large_utf8 Filter (500M strings, 0-32 B) + dictionary-encoded Take ----
    m = n // 2
    lens = torch.randint(0, 33, (m,), dtype=I64, device="cuda", generator=gen)
    offs = torch.zeros(m + 1, dtype=I64, device="cuda")
    torch.cumsum(lens, 0, out=offs[1:])
    total = int(offs[-1].item())
    del lens
    data = torch.randint(97, 123, (total + 64,), dtype=torch.uint8, device="cuda", generator=gen)
    svalid_t, s_nulls = make_validity(torch, m, gen)
    strs = DeviceArray.from_pointers(ctx, pa.large_string(), m, offs.data_ptr(), validity_ptr=svalid_t.data_ptr(), null_count=s_nulls,
                                     data2_ptr=data.data_ptr())
    mask_bits = make_mask(torch, m, gen, 0.5)
    mask = DeviceArray.from_pointers(ctx, pa.bool_(), m, mask_bits.data_ptr())
    ms = env.timed(lambda: bc.filter(strs, mask), reps)
    res = bc.filter(strs, mask)
    L = total / max(m, 1)
    # parity: kept rows, offsets = running sum of the kept lengths, validity of the kept rows, and a byte-exact
    # comparison of the whole output data buffer against torch's own compaction (16M-row slabs)
    sel = unpack_bits(torch, mask_bits, m)
    ro = torch.as_tensor(_view(res.buffers[1].ptr, res.length + 1, "<i8", res), device="cuda")
    ok = res.length == int(sel.sum().item()) and int(ro[0].item()) == 0
    rd = torch.as_tensor(_view(res.buffers[2].ptr, max(int(ro[-1].item()), 1), "|u1", res), device="cuda") if ok else None
    rv = unpack_bits(torch, torch.as_tensor(_view(res.buffers[0].ptr, (res.length + 7) // 8, "|u1", res), device="cuda"), res.length) \
        if res.buffers[0] is not None else None
    slab, k0 = 1 << 24, 0
    for r0 in range(0, m, slab):
        if not ok:
            break
        r1 = min(m, r0 + slab)
        sc = sel[r0:r1]
        row_valid = unpack_bits(torch, svalid_t[r0 // 8:], r1 - r0)
        # a null string contributes no bytes to the output (the reference appends a null = repeats the offset,
        # vector_selection_filter_internal.cc:598-856), whatever its slot spans in the input
        ln = (offs[r0 + 1:r1 + 1] - offs[r0:r1]) * row_valid
        k1 = k0 + int(sc.sum().item())
        ok = ok and bool(((ro[k0 + 1:k1 + 1] - ro[k0:k1]) == ln[sc]).all().item())
        b0, b1 = int(offs[r0].item()), int(offs[r1].item())
        want_bytes = data[b0:b1][torch.repeat_interleave(sc & row_valid, offs[r0 + 1:r1 + 1] - offs[r0:r1])]
        g0, g1 = int(ro[k0].item()), int(ro[k1].item())
        ok = ok and (g1 - g0) == want_bytes.numel() and bool(torch.equal(rd[g0:g1], want_bytes))
        want_valid = row_valid[sc]
        ok = ok and bool(((rv[k0:k1] if rv is not None else torch.ones(k1 - k0, dtype=torch.bool, device="cuda")) == want_valid).all().item())
        k0 = k1
        del sc, ln, want_bytes, want_valid, row_valid
    entry("c5 filter large_utf8 500M strings (0-32 B, null_p 0.1, s=0.5)", m, ms,
          m * (8 + L + 0.25) + res.length * (8 + L + 0.125), ok, mean_len=L)
    del res, strs, offs, data, svalid_t, mask, mask_bits, sel, ro, rd, rv
    ctx.trim()
    torch.cuda.empty_cache()
    dict_idx_t = torch.randint(0, 1_000_000, (m,), dtype=torch.int32, device="cuda", generator=gen)
    col = DeviceArray.from_pointers(ctx, pa.int32(), m, dict_idx_t.data_ptr())
    take_idx_t = torch.randint(0, m, (m,), dtype=I64, device="cuda", generator=gen)
    take_idx = DeviceArray.from_pointers(ctx, pa.int64(), m, take_idx_t.data_ptr())
    ms = env.timed(lambda: bc.take(col, take_idx), reps)
    res = bc.take(col, take_idx)
    rt = torch.as_tensor(_view(res.buffers[1].ptr, m, "<i4", res), device="cuda")
    ok = bool((rt == dict_idx_t[take_idx_t]).all().item())
    entry("c5 dictionary take (int32 index column, uniform random int64 idx)", m, ms, m * (8 + 4 + 4), ok)
    del res, rt, col, take_idx, dict_idx_t, take_idx_t
    ctx.trim()
    torch.cuda.empty_cache()
    return out


class _View:
    def __init__(self, ptr, n, typestr, owner):
        self.owner = owner
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}


def _view(ptr, n, typestr, owner):
    return _View(ptr, max(int(n), 0), typestr, owner)


DUMP_ROWS = 1 << 21  # rows of the pipeline's result written by --dump-outputs: 32 MiB of .npy files


def dump_pipeline_output(torch, out, n, out_dir, prefix=""):
    """Writes the float32 column the pipeline returns as .npy files under `out_dir`, so that two builds can be compared
    output for output: result_values (0.0 where null), result_validity (1.0 / 0.0), result_rows (the row numbers) and
    result_null_count (of the whole column).  Above DUMP_ROWS rows the column is sampled at one seeded row of each of
    DUMP_ROWS equal strata, the same rows for every run with the same --rows."""
    import numpy as np
    if n <= DUMP_ROWS:
        rows = np.arange(n, dtype=np.int64)
    else:
        stride = n // DUMP_ROWS
        rows = np.arange(DUMP_ROWS, dtype=np.int64) * stride + np.random.default_rng(SEED).integers(0, stride, DUMP_ROWS)
    r = torch.from_numpy(rows).to("cuda") + out.offset
    vals = torch.as_tensor(_view(out.buffers[1].ptr, out.offset + n, "<f4", out), device="cuda")[r]
    if out.buffers[0] is not None:
        bits = torch.as_tensor(_view(out.buffers[0].ptr, (out.offset + n + 7) // 8, "|u1", out), device="cuda")
        valid = ((bits[r >> 3] >> (r & 7).to(torch.uint8)) & 1).bool()
    else:
        valid = torch.ones(len(rows), dtype=torch.bool, device="cuda")
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"result_values": torch.where(valid, vals, 0.0).cpu().numpy(),  # a null slot's bytes are unspecified
              "result_validity": valid.to(torch.float32).cpu().numpy(),
              "result_rows": rows.astype(np.float64),
              "result_null_count": np.array([out.null_count], dtype=np.float64)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{prefix}{name}.npy"), a)


# ------------------------------------------------------------------------------------------------
# configs[2] / configs[3] sharded over the ranks (strong scaling, one exchange each)
# ------------------------------------------------------------------------------------------------
BLOCK = 1 << 20  # rows generated per seed: the global dataset is identical at every N


def run_multi_gpu(env, n_total, reps):
    import pyarrow as pa

    from arrow_b200 import DeviceArray
    from arrow_b200 import distributed as d
    torch, ctx, world, rank = env.torch, env.ctx, env.world, env.rank
    I64 = torch.int64
    ops = d.DeviceOps(ctx)
    xchg = d.B2CommExchange(ctx)
    n_blocks = (n_total + BLOCK - 1) // BLOCK
    b0, b1 = rank * n_blocks // world, (rank + 1) * n_blocks // world
    row0, row1 = b0 * BLOCK, min(b1 * BLOCK, n_total)
    n_local = row1 - row0
    groups = 10_000_000 if n_total >= 100_000_000 else max(1000, n_total // 100)
    result = {"rows_total": n_total, "scaling": "strong", "transport": "b2_comm (NCCL all-to-all-v, one NCCL group per exchange)",
              "rows_this_rank0": n_local}

    def gen_columns(kind):
        """kind 'groupby': keys uniform [0, groups), values uniform [-100, 100] null_p 0.1
           kind 'sort'   : keys uniform [-2^62, 2^62) null_p 0.1 (returned as the `keys` column + validity)"""
        keys = torch.empty(n_local, dtype=I64, device="cuda")
        vals = torch.empty(n_local, dtype=I64, device="cuda") if kind == "groupby" else None
        bits = torch.zeros(n_local // 8 + BLOCK // 8 + 64, dtype=torch.uint8, device="cuda")
        g = torch.Generator(device="cuda")
        nulls = 0
        for b in range(b0, b1):
            lo = b * BLOCK - row0
            m = min(BLOCK, n_total - b * BLOCK)
            g.manual_seed((SEED * 1000003 + b * 7 + (0 if kind == "groupby" else 3)) & 0x7FFFFFFFFFFF)
            if kind == "groupby":
                keys[lo:lo + m] = torch.randint(0, groups, (m,), dtype=I64, device="cuda", generator=g)
                vals[lo:lo + m] = torch.randint(-100, 101, (m,), dtype=I64, device="cuda", generator=g)
            else:
                keys[lo:lo + m] = torch.randint(-2**62, 2**62, (m,), dtype=I64, device="cuda", generator=g)
            v = torch.rand(BLOCK, device="cuda", generator=g) >= NULL_P
            v[m:] = False
            nulls += m - int(v.sum().item())
            bits[lo // 8: lo // 8 + BLOCK // 8] = pack_bits(torch, v)
        return keys, vals, bits, nulls

    last_reps = []

    def leg(fn):
        """CUDA-event time of `fn` (max over ranks), after one warm-up; also the exchange's own time"""
        r = fn()
        del r
        env.sync_all()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ms_list, x_list = [], []
        xbytes = 0
        for _ in range(reps):
            r = None        # the previous result goes back to the pool first: otherwise every repetition has to cudaMalloc a second set
            env.sync_all()  # of result buffers inside the timed region (measured: 11.7 / 29.4 / 44.6 ms for the same call)
            a.record(env.stream)
            r = fn()
            b.record(env.stream)
            torch.cuda.synchronize()
            ms_list.append(env.max_over_ranks(a.elapsed_time(b)))
            xm, xbytes = ops.exchange_stats() if world > 1 else (0.0, 0)
            x_list.append(env.max_over_ranks(xm))
        # median, not mean: a repetition that had to cudaMalloc (the pool was trimmed between legs) costs 2-7x and is not what the
        # exchange leg measures; every repetition is kept in `reps_ms`
        order = sorted(range(len(ms_list)), key=lambda i: ms_list[i])
        mid = order[len(order) // 2]
        last_reps[:] = [round(x, 3) for x in ms_list]
        return r, ms_list[mid], x_list[mid], xbytes

    # ---- config 3: hash-aggregate ----
    keys_t, vals_t, bits_t, v_nulls = gen_columns("groupby")
    keys = DeviceArray.from_pointers(ctx, pa.int64(), n_local, keys_t.data_ptr())
    vals = DeviceArray.from_pointers(ctx, pa.int64(), n_local, vals_t.data_ptr(), validity_ptr=bits_t.data_ptr(), null_count=v_nulls)
    # expected_groups: a shard of >= 100 rows per key sees essentially every key
    (k, s, c), ms, xms, xbytes = leg(lambda: d.group_by_sum_count(keys, vals, ops, xchg, expected_groups=groups))
    kt = torch.as_tensor(_view(k.buffers[1].ptr, k.length, "<i8", k), device="cuda")
    st = torch.as_tensor(_view(s.buffers[1].ptr, s.length, "<i8", s), device="cuda")
    ct = torch.as_tensor(_view(c.buffers[1].ptr, c.length, "<i8", c), device="cuda")
    # invariants derived from the INPUT columns (torch, independent of the kernels under test)
    valid = unpack_bits(torch, bits_t, n_local).to(I64)
    in_count, in_sum = int(valid.sum().item()), int((vals_t * valid).sum().item())
    in_keysum = int((mix64(torch, keys_t) * valid).sum().item())
    out_groups, out_count, out_sum = k.length, int(ct.sum().item()), int((st * (ct > 0)).sum().item())
    out_keysum = int((mix64(torch, kt) * ct).sum().item())
    out_distinct = int(mix64(torch, kt).sum().item())
    checksum = int((mix64(torch, kt) * (2 * st * (ct > 0) + 1) * (2 * ct + 3)).sum().item())
    tot = env.sum_over_ranks([in_count, in_sum, in_keysum, out_groups, out_count, out_sum, out_keysum, out_distinct, checksum])
    wrap = lambda x: x % (1 << 64)
    want_distinct = int(mix64(torch, torch.arange(groups, dtype=I64, device="cuda")).sum().item())
    ok = (tot[0] == tot[4] and wrap(tot[1]) == wrap(tot[5]) and wrap(tot[2]) == wrap(tot[6]) and tot[3] <= groups
          and (tot[3] != groups or wrap(tot[7]) == wrap(want_distinct)))
    result["groupby"] = {"workload": f"hash_sum+hash_count, int64 key, {groups} groups, value null_p 0.1", "ms": ms,
                         "rows_per_s": n_total / (ms * 1e-3), "alltoall_bytes_per_rank": xbytes, "alltoall_ms": xms,
                         "alltoall_share": (xms / ms) if ms else None, "groups": tot[3],
                         "alg_bytes": n_total * 16.125 + tot[3] * 24.25,
                         "frac_of_peak_x_n": (n_total * 16.125 + tot[3] * 24.25) / (ms * 1e-3) / 1e9 / (measured_peaks()[0] * world),
                         "checksum": wrap(tot[8]), "parity_checksum_ok": bool(ok), "reps_ms": list(last_reps)}
    del k, s, c, kt, st, ct, keys, vals, keys_t, vals_t, bits_t, valid
    ctx.trim()
    torch.cuda.empty_cache()

    # ---- config 4: SortIndices ----
    keys_t, _, bits_t, k_nulls = gen_columns("sort")
    keys = DeviceArray.from_pointers(ctx, pa.int64(), n_local, keys_t.data_ptr(), validity_ptr=bits_t.data_ptr(), null_count=k_nulls)
    _, ms, xms, xbytes = leg(lambda: d.sort_indices(keys, ops, xchg))
    sort_reps = list(last_reps)
    seg_fast, nulls_fast = d.sort_indices(keys, ops, xchg)                      # the timed path's own answer ...
    seg, nulls_idx, skeys = d.sort_indices(keys, ops, xchg, return_keys=True)  # ... and the variant that also returns the sorted keys
    same_answer = bool(torch.equal(seg_fast, seg)) and bool(torch.equal(nulls_fast, nulls_idx))
    del seg_fast, nulls_fast
    valid = unpack_bits(torch, bits_t, n_local)
    grow = torch.arange(row0, row1, dtype=I64, device="cuda")
    in_pair = int((mix64(torch, grow) * keys_t * valid.to(I64)).sum().item())
    out_pair = int((mix64(torch, seg) * skeys).sum().item())
    good = (skeys[1:] > skeys[:-1]) | ((skeys[1:] == skeys[:-1]) & (seg[1:] > seg[:-1]))
    local_ok = bool(good.all().item()) if skeys.numel() > 1 else True
    if nulls_idx.numel() > 1:
        local_ok = local_ok and bool((nulls_idx[1:] > nulls_idx[:-1]).all().item())
    if nulls_idx.numel():
        local_ok = local_ok and not bool(valid[nulls_idx - row0].any().item())
    # rank boundaries: (last key, last idx) of rank r must sort before (first key, first idx) of rank r+1
    edge = torch.zeros(4, dtype=I64, device="cuda")
    if skeys.numel():
        edge[0], edge[1], edge[2], edge[3] = skeys[0], seg[0], skeys[-1], seg[-1]
    edges = [torch.zeros(4, dtype=I64, device="cuda") for _ in range(world)]
    sizes = env.torch.tensor([skeys.numel()], dtype=I64, device="cuda")
    all_sizes = [torch.zeros(1, dtype=I64, device="cuda") for _ in range(world)]
    if world > 1:
        env.dist.all_gather(edges, edge)
        env.dist.all_gather(all_sizes, sizes)
    else:
        edges, all_sizes = [edge], [sizes]
    prev = None
    for e, z in zip(edges, all_sizes):
        if int(z.item()) == 0:
            continue
        e = [int(x) for x in e.tolist()]
        if prev is not None and not (e[0] > prev[0] or (e[0] == prev[0] and e[1] > prev[1])):
            local_ok = False
        prev = (e[2], e[3])
    idx_sum = int(seg.sum().item()) + int(nulls_idx.sum().item())
    checksum = int((mix64(torch, seg) * (skeys | 1)).sum().item())
    local_ok = local_ok and same_answer
    tot = env.sum_over_ranks([in_pair, out_pair, seg.numel() + nulls_idx.numel(), idx_sum, 0 if local_ok else 1, nulls_idx.numel(),
                              k_nulls, checksum])
    ok = (wrap(tot[0]) == wrap(tot[1]) and tot[2] == n_total and wrap(tot[3]) == wrap(n_total * (n_total - 1) // 2) and tot[4] == 0
          and tot[5] == tot[6])
    result["sort"] = {"workload": "sort_indices int64 uniform [-2^62, 2^62), null_p 0.1, ascending, nulls at end", "ms": ms,
                      "rows_per_s": n_total / (ms * 1e-3), "alltoall_bytes_per_rank": xbytes, "alltoall_ms": xms,
                      "alltoall_share": (xms / ms) if ms else None, "alg_bytes": n_total * 16.125,
                      "frac_of_peak_x_n": n_total * 16.125 / (ms * 1e-3) / 1e9 / (measured_peaks()[0] * world),
                      "segment_rows_rank0": int(seg.numel()), "checksum": wrap(tot[7]), "parity_checksum_ok": bool(ok),
                      "reps_ms": sort_reps}
    del seg, nulls_idx, skeys, keys, keys_t, bits_t, valid, grow
    xchg.close()
    ctx.trim()
    torch.cuda.empty_cache()
    return result


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def run_gpu(args):
    import numpy as np
    import pyarrow as pa

    env = Env(args)
    torch, dist, ctx, stream, lib = env.torch, env.dist, env.ctx, env.stream, env.lib
    world, rank, local = env.world, env.rank, env.local
    import arrow_b200.compute as bc
    from arrow_b200 import DeviceArray, PinnedBuffer

    n = args.rows
    gen = torch.Generator(device="cuda")
    gen.manual_seed(SEED + rank)
    # ---- synthetic inputs, resident in HBM (SURVEY section 8d, C2) ----
    values_t = torch.rand(n, dtype=torch.float64, device="cuda", generator=gen) * 1e6
    vvalid_t, v_nulls = make_validity(torch, n, gen)
    idx_t = torch.randint(0, n, (n,), dtype=torch.int64, device="cuda", generator=gen)
    other_t = torch.rand(n, dtype=torch.float32, device="cuda", generator=gen) * 1e6
    ovalid_t, o_nulls = make_validity(torch, n, gen)
    values = DeviceArray.from_pointers(ctx, pa.float64(), n, values_t.data_ptr(), validity_ptr=vvalid_t.data_ptr(), null_count=v_nulls)
    indices = DeviceArray.from_pointers(ctx, pa.int64(), n, idx_t.data_ptr())
    other = DeviceArray.from_pointers(ctx, pa.float32(), n, other_t.data_ptr(), validity_ptr=ovalid_t.data_ptr(), null_count=o_nulls)

    def pipeline_unfused(v, i, o):   # three CallFunction-equivalent calls
        t = bc.take(v, i)
        c = bc.cast(t, pa.float32(), safe=False)
        return bc.add(c, o)

    def pipeline(v, i, o):           # the same expression through the fused entry point (b2_take_cast_arith): one kernel
        return bc.take_cast_arith(v, i, pa.float32(), "add", o)

    if args.unfused:
        pipeline = pipeline_unfused

    sync_all, max_over_ranks = env.sync_all, env.max_over_ranks

    # ---- warm-up (also fills the pool so the timed region never calls cudaMalloc) ----
    for _ in range(args.warmup):
        out = pipeline(values, indices, other)
    out_nulls = out.null_count
    # parity of the step's result against a plain torch restatement of the same three ops (verification only)
    ot = torch.as_tensor(_view(out.buffers[1].ptr, n, "<f4", out), device="cuda")
    ovb = unpack_bits(torch, torch.as_tensor(_view(out.buffers[0].ptr, (n + 7) // 8, "|u1", out), device="cuda"), n) \
        if out.buffers[0] is not None else torch.ones(n, dtype=torch.bool, device="cuda")
    pipeline_ok = True
    chunk = 1 << 27
    vv_all = None
    for lo in range(0, n, chunk):
        m = min(chunk, n - lo)
        ii = idx_t[lo:lo + m]
        want_valid = ((vvalid_t[ii >> 3] >> (ii & 7).to(torch.uint8)) & 1).bool() & unpack_bits(torch, ovalid_t[lo // 8:], m)
        want = values_t[ii].to(torch.float32) + other_t[lo:lo + m]
        got_valid = ovb[lo:lo + m]
        pipeline_ok = pipeline_ok and bool((got_valid == want_valid).all().item())
        pipeline_ok = pipeline_ok and bool((ot[lo:lo + m][want_valid] == want[want_valid]).all().item())
        del ii, want_valid, want, got_valid
    del out, ot, ovb

    # ---- per-kernel timing (events around each call; the call = its kernel + a bitmap kernel) ----
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    k_ms = np.zeros(3)
    sync_all()
    for it in range(args.steps + 1):  # iteration 0 is a warm-up: the pool may still have to cudaMalloc the intermediates
        ev[0].record(stream)
        t = bc.take(values, indices)
        ev[1].record(stream)
        c = bc.cast(t, pa.float32(), safe=False)
        ev[2].record(stream)
        o = bc.add(c, other)
        ev[3].record(stream)
        torch.cuda.synchronize()
        if it:
            k_ms += [ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[2].elapsed_time(ev[3])]
        del t, c, o
    k_ms /= args.steps
    fused_ms = env.timed(lambda: bc.take_cast_arith(values, indices, pa.float32(), "add", other), args.steps)

    # ---- timed region: K steps, device resident ----
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    launches0 = lib.b2_launch_count()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    start.record(stream)
    for step in range(args.steps):
        out = pipeline(values, indices, other)
        if step < args.steps - 1:  # the last step's result outlives the loop for --dump-outputs
            del out
    stop.record(stream)
    sync_all()
    total_ms = max_over_ranks(start.elapsed_time(stop))
    launches = lib.b2_launch_count() - launches0
    clocks = sampler.summary() if sampler else None
    if args.dump_outputs:
        dump_pipeline_output(torch, out, n, args.dump_outputs, f"rank{rank}_" if world > 1 else "")
    del out
    ms_per_step = total_ms / args.steps
    value = n * world / (ms_per_step * 1e-3)

    # ---- sorted-index variant of take (SURVEY section 8d asks for both) ----
    inc = torch.randint(0, 3, (n,), dtype=torch.int64, device="cuda", generator=gen)
    sorted_idx_t = torch.clamp(torch.cumsum(inc, 0), max=n - 1)
    del inc
    sorted_idx = DeviceArray.from_pointers(ctx, pa.int64(), n, sorted_idx_t.data_ptr())
    take_sorted_ms = env.timed(lambda: bc.take(values, sorted_idx), args.steps)
    del sorted_idx, sorted_idx_t

    # ---- e2e: pinned host inputs -> H2D -> pipeline -> D2H of the result column ----
    e2e_rows = min(n, args.e2e_rows) if args.e2e_rows else n
    try:
        import psutil
        avail = psutil.virtual_memory().available
        need = e2e_rows * 24.5 * (world if world > 1 else 1)
        if need > 0.5 * avail:
            e2e_rows = int(0.5 * avail / (24.5 * world)) // 64 * 64
    except Exception:
        pass
    m = e2e_rows
    bm = (m + 7) // 8
    h_values, h_vvalid = PinnedBuffer(8 * m), PinnedBuffer(bm)
    h_idx, h_other, h_ovalid = PinnedBuffer(8 * m), PinnedBuffer(4 * m), PinnedBuffer(bm)
    h_out, h_outvalid = PinnedBuffer(4 * m), PinnedBuffer(bm + 8)
    idx_small = idx_t[:m] % m if m != n else idx_t
    for hb, src in ((h_values, values_t[:m]), (h_vvalid, vvalid_t[:bm]), (h_idx, idx_small), (h_other, other_t[:m]), (h_ovalid, ovalid_t[:bm])):
        ctx.d2h(hb.ptr, src.data_ptr(), hb.size)
    ctx.sync()
    del idx_small
    d_values, d_vvalid = ctx.alloc(8 * m), ctx.alloc(bm + 64)
    d_idx, d_other, d_ovalid = ctx.alloc(8 * m), ctx.alloc(4 * m), ctx.alloc(bm + 64)
    h2d_bytes = 8 * m + bm + 8 * m + 4 * m + bm
    d2h_bytes = 4 * m + bm

    # The e2e leg is chunked the way the reference chunks: `indices` / `other` travel as K chunks (a
    # ChunkedArray argument to take/add, each chunk one CallFunction-equivalent call), so the H2D copy of
    # chunk k+1, the kernels of chunk k and the D2H copy of chunk k-1 overlap on three streams.  `values`
    # (the gathered column) must be fully resident before the first chunk is gathered.
    K = max(1, args.e2e_chunks)
    copy_in, copy_out = torch.cuda.Stream(), torch.cuda.Stream()
    bounds = [min(m, (m * k // K) // 64 * 64) for k in range(K)] + [m]

    def e2e_step():
        ci, co = copy_in.cuda_stream, copy_out.cuda_stream
        ctx.h2d(d_values.ptr, h_values.ptr, h_values.size, ci)
        ctx.h2d(d_vvalid.ptr, h_vvalid.ptr, h_vvalid.size, ci)
        ev_vals = torch.cuda.Event()
        ev_vals.record(copy_in)
        ready = []
        for k in range(K):
            lo, hi = bounds[k], bounds[k + 1]
            ctx.h2d(d_idx.ptr + 8 * lo, h_idx.ptr + 8 * lo, 8 * (hi - lo), ci)
            ctx.h2d(d_other.ptr + 4 * lo, h_other.ptr + 4 * lo, 4 * (hi - lo), ci)
            ctx.h2d(d_ovalid.ptr + lo // 8, h_ovalid.ptr + lo // 8, (hi - lo + 7) // 8, ci)
            e = torch.cuda.Event()
            e.record(copy_in)
            ready.append(e)
        v = DeviceArray.from_pointers(ctx, pa.float64(), m, d_values.ptr, validity_ptr=d_vvalid.ptr, null_count=-1)
        stream.wait_event(ev_vals)
        keep, nulls = [], 0
        for k in range(K):
            lo, hi = bounds[k], bounds[k + 1]
            stream.wait_event(ready[k])
            i = DeviceArray.from_pointers(ctx, pa.int64(), hi - lo, d_idx.ptr + 8 * lo)
            o = DeviceArray.from_pointers(ctx, pa.float32(), hi - lo, d_other.ptr + 4 * lo, validity_ptr=d_ovalid.ptr + lo // 8,
                                          null_count=-1)
            r = pipeline(v, i, o)          # three C-ABI calls on `stream`
            done = torch.cuda.Event()
            done.record(stream)
            copy_out.wait_event(done)
            ctx.d2h(h_out.ptr + 4 * lo, r.buffers[1].ptr, 4 * (hi - lo), co)
            if r.buffers[0] is not None:   # chunk validity lands at its own (byte aligned: lo % 64 == 0) position
                ctx.d2h(h_outvalid.ptr + lo // 8, r.buffers[0].ptr, (hi - lo + 7) // 8, co)
            keep.append(r)                 # buffers stay alive until the D2H stream drains
            nulls += r.null_count
        copy_out.synchronize()
        return nulls

    e2e_step()
    sync_all()
    t0 = time.perf_counter()
    start.record(stream)
    e2e_steps = max(1, min(args.steps, 3))
    for _ in range(e2e_steps):
        e2e_step()
    stop.record(stream)
    sync_all()
    e2e_ms = max_over_ranks(max(start.elapsed_time(stop), (time.perf_counter() - t0) * 1e3)) / e2e_steps
    e2e_value = m * world / (e2e_ms * 1e-3)
    del h_values, h_vvalid, h_idx, h_other, h_ovalid, h_out, h_outvalid, d_values, d_vvalid, d_idx, d_other, d_ovalid

    # ---- free config 2's columns, then the other configs and the sharded legs ----
    del values, indices, other, values_t, vvalid_t, idx_t, other_t, ovalid_t
    ctx.trim()
    torch.cuda.empty_cache()
    configs = None
    if world == 1 and not args.no_configs:
        try:
            configs = run_configs(env, args.rows)
        except Exception as e:  # report, never lose the headline line
            configs = [{"error": f"{type(e).__name__}: {e}"[:400]}]
    multi = None
    if not args.no_multi:
        try:
            multi = run_multi_gpu(env, args.multi_rows or args.rows, max(1, min(args.steps, 3)))
        except Exception as e:
            multi = {"error": f"{type(e).__name__}: {e}"[:400]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peaks()
    take_gbs = ALG_TAKE * n / (k_ms[0] * 1e-3) / 1e9
    kernels = [
        {"name": "take_kernel<8,int64> (random idx)", "ms": float(k_ms[0]), "alg_bytes_per_row": ALG_TAKE, "gbs": take_gbs, "frac": take_gbs / peak},
        {"name": "take_kernel<8,int64> (monotonic idx)", "ms": float(take_sorted_ms), "alg_bytes_per_row": ALG_TAKE,
         "gbs": ALG_TAKE * n / (take_sorted_ms * 1e-3) / 1e9, "frac": ALG_TAKE * n / (take_sorted_ms * 1e-3) / 1e9 / peak},
        {"name": "map1_kernel<double,float> (cast)", "ms": float(k_ms[1]), "alg_bytes_per_row": ALG_CAST,
         "gbs": ALG_CAST * n / (k_ms[1] * 1e-3) / 1e9, "frac": ALG_CAST * n / (k_ms[1] * 1e-3) / 1e9 / peak},
        {"name": "map2_kernel<float> (add)", "ms": float(k_ms[2]), "alg_bytes_per_row": ALG_ADD,
         "gbs": ALG_ADD * n / (k_ms[2] * 1e-3) / 1e9, "frac": ALG_ADD * n / (k_ms[2] * 1e-3) / 1e9 / peak},
        {"name": "take_cast_arith_kernel<double,int64,float> (fused take+cast+add, random idx)", "ms": float(fused_ms),
         "alg_bytes_per_row": ALG_PIPELINE, "gbs": ALG_PIPELINE * n / (fused_ms * 1e-3) / 1e9,
         "frac": ALG_PIPELINE * n / (fused_ms * 1e-3) / 1e9 / peak},
    ]
    # the dominant kernel of the timed step: the fused take+cast+add kernel (or take_kernel with --unfused); its algorithmic
    # bytes are SURVEY 8d's unfused sum for the whole expression ("the honest denominator even if kernels are fused")
    traffic_key = "dram_bytes_per_row_unfused_take" if args.unfused else "dram_bytes_per_row_fused"
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "take_traffic.json")))
        traffic = tj[traffic_key] * n
    except Exception:
        traffic = None
    if args.unfused:
        roofline = {"bound": "hbm", "achieved": take_gbs, "peak": peak, "unit": "GB/s", "frac": take_gbs / peak, "traffic": traffic,
                    "kernel": "take_kernel<8,int64_t,true>", "peak_source": peak_src, "alg_bytes_per_launch": ALG_TAKE * n}
    else:
        fused_gbs = ALG_PIPELINE * n / (fused_ms * 1e-3) / 1e9
        roofline = {"bound": "hbm", "achieved": fused_gbs, "peak": peak, "unit": "GB/s", "frac": fused_gbs / peak, "traffic": traffic,
                    "kernel": "take_cast_arith_kernel<double,int64_t,float,true> (+ its take_validity_band_kernel pass: one call)",
                    "peak_source": peak_src, "alg_bytes_per_launch": ALG_PIPELINE * n,
                    "note": "time and traffic are those of the whole b2_take_cast_arith call = the gather kernel (26.9 ms under ncu) + one "
                            "validity band pass (2.9 ms). Random 8-byte gathers: DRAM moves ~127 B per gathered value and DRAM accesses, not "
                            "bytes, are the limit (42-44 G/s, profiles/gather_probe_r01.csv), so the byte roofline is not reachable; "
                            "monotonic indices run the same gather at 0.82 (profiles/take_traffic.json, take_band_sweep_r02.jsonl)"}
    cpu = cpu_baseline_leg(args) if world == 1 else {"value": None, "unit": "rows/s", "cores": os.cpu_count() or 1, "kind": "reference",
                                                      "sample": "measured at N = 1 only (rank 0)"}
    line = {
        "metric": "rows/sec", "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64->f32", "data": "synthetic",
        "config": {"workload": "Take(float64,int64 idx)+Cast(float64->float32)+Add(float32), null_probability=0.1, 1B rows/GPU"
                   if n == 1_000_000_000 else f"Take+Cast(f64->f32)+Add, null_probability=0.1, {n} rows/GPU",
                   "rows_per_gpu": n, "indices": "uniform random int64", "l2": "inputs (20 GB) are far larger than the 126 MB L2",
                   "pipeline_alg_bytes_per_row": ALG_PIPELINE, "pipeline_gbs": ALG_PIPELINE * n * world / (ms_per_step * 1e-3) / 1e9,
                   "out_null_count": int(out_nulls), "parity_checksum_ok": bool(pipeline_ok), "numa_node": env.numa,
                   "calls_per_step": "3 (take, cast, add)" if args.unfused else "1 (b2_take_cast_arith: the fused take+cast+add kernel)",
                   "unfused_ms_per_step": float(k_ms.sum())},
        "roofline": roofline,
        "kernels": kernels,
        "cpu_baseline": cpu,
        "e2e": {"value": e2e_value, "unit": "rows/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                "rows_per_gpu": m, "ms_per_step": e2e_ms, "chunks": K},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "configs": configs,
        "multi_gpu": multi,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=1_000_000_000, help="rows per GPU (config 2) / total rows (configs, multi_gpu legs)")
    ap.add_argument("--multi-rows", type=int, default=0, help="total rows of the sharded group-by / sort legs (0 = --rows)")
    ap.add_argument("--e2e-rows", type=int, default=0, help="rows per GPU for the host-buffer leg (0 = same as --rows)")
    ap.add_argument("--e2e-chunks", type=int, default=8, help="chunks of the indices/other columns in the host-buffer leg")
    ap.add_argument("--no-configs", action="store_true", help="skip the `configs` array (c1/c3/c4/c5 at full size, N = 1 only)")
    ap.add_argument("--no-multi", action="store_true", help="skip the sharded group-by / sort legs")
    ap.add_argument("--unfused", action="store_true", help="run the pipeline as three calls (take, cast, add) instead of the fused kernel")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result column of the last timed step (sampled above 2^21 rows) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl b200: the reference arm runs in oracle/_ref/ref_bench and returns timings only")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
