#!/usr/bin/env python
"""bench_configs.py -- the other BASELINE.json configs at scale (not the driver's bench line):
  c1  Filter(int64, bool mask)            1B rows, values null_p 0.1, mask non-null, s = 0.5
  c3  group-by sum+count, int64 key/value 1B rows, 10M groups (fused table and Grouper+aggregators)
  c3u group-by / dictionary_encode with a large_utf8 key   500M strings from 1M distinct words (not in the default --only list)
  join inner hash join: n/2 probe rows against 10M unique build keys (not in the default --only list)
  c4  SortIndices int64 + validity        1B rows (wide range) and narrow range [0, 4095]
  sort_utf8         SortIndices large_utf8, n/2 strings from 1M distinct words of 8-16 B (dictionary path)
  sort_utf8_unique  SortIndices large_utf8, n/5 random strings of 8-32 B (prefix refinement)
  sort_utf8_prefix  SortIndices large_utf8, n/10 strings sharing a 40-byte prefix (refinement, 7+ rounds)
                    (the three sort_utf8 configs are not in the default --only list)
  f1  dictionary_encode / value_counts of an int64 column (1M distinct values), 500M rows
  c5  large_utf8 Filter                   500M strings, 0-32 B, null_p 0.1, s = 0.5  (+ dictionary Take)
  cmp compare int64 -> bool               1B rows
Each prints one JSON line: rows/s, algorithmic GB/s (SURVEY.md section 8d byte model) and the
fraction of the measured copy peak.  Inputs are generated on the device with torch (plumbing).
Usage: python bench_configs.py [--rows N] [--only c1,c3,...] [--reps K]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import pyarrow as pa
import torch

import arrow_b200.compute as bc
from arrow_b200 import Context, DeviceArray
from bench import NULL_P, SEED, make_validity, measured_peaks


def timed(stream, fn, reps, warmup=2):
    for _ in range(warmup):
        r = fn()
        del r
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(reps):
        r = fn()
        del r
    b.record(stream)
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


class _Cai:
    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}


def _cai(ptr, n, typestr):
    return _Cai(ptr, n, typestr)


def report(name, n, ms, alg_bytes, extra=None):
    peak, _ = measured_peaks()
    gbs = alg_bytes / (ms * 1e-3) / 1e9
    line = {"config": name, "rows": n, "ms": ms, "rows_per_s": n / (ms * 1e-3), "alg_bytes": alg_bytes, "gbs": gbs,
            "frac_of_measured_peak": gbs / peak}
    if extra:
        line.update(extra)
    print(json.dumps(line), flush=True)


def card():
    """the GPU the numbers were measured on and its power limit (read only)"""
    import subprocess
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True).stdout.strip().split(", ")
    return {"gpu": q[0] if q and q[0] else torch.cuda.get_device_name(), "power_limit_w": float(q[1]) if len(q) > 1 else None}


def sort_parity(ctx, out, m, offs, data, gen):
    """the sort result is a permutation (scatter-count on the device) and 1M seeded sampled adjacent output pairs are in
    order on the host, equal neighbours in increasing row order"""
    idx = torch.as_tensor(_cai(out.buffers[1].ptr, m, "<u8"), device="cuda").to(torch.int64)
    seen = torch.zeros(m, dtype=torch.int32, device="cuda")
    seen.index_add_(0, idx, torch.ones(m, dtype=torch.int32, device="cuda"))
    ok = bool((seen == 1).all().item())
    del seen
    j = torch.randint(0, m - 1, (1 << 20,), device="cuda", generator=gen)
    a, b = idx[j], idx[j + 1]
    del idx
    host = {}
    for name, rows in (("a", a), ("b", b)):
        lo, hi = offs[rows], offs[rows + 1]
        width = int((hi - lo).max().item())
        pos = lo.unsqueeze(1) + torch.arange(width, device="cuda")
        mat = torch.where(pos < hi.unsqueeze(1), data[pos.clamp(max=data.numel() - 1)], torch.zeros((), dtype=torch.uint8, device="cuda"))
        host[name] = (mat.cpu().numpy(), (hi - lo).cpu().numpy(), rows.cpu().numpy())
    (ma, la, ra), (mb, lb, rb) = host["a"], host["b"]
    for i in range(len(ra)):
        x, y = ma[i, :la[i]].tobytes(), mb[i, :lb[i]].tobytes()
        if not (x < y or (x == y and ra[i] < rb[i])):
            return False
    return ok


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1_000_000_000)
    ap.add_argument("--only", default="c1,cmp,c3,c4,c5,f1")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--fused-only", action="store_true", help="c3: stop after the fused group-by")
    ap.add_argument("--groups", type=int, default=0, help="c3: number of distinct keys (default 10M at >= 100M rows)")
    ap.add_argument("--vocab", default="", help="sort_utf8: comma-separated numbers of distinct words (default 1M at >= 10M strings)")
    ap.add_argument("--string-paths", default="auto",
                    help="sort_utf8*: comma-separated sort paths to time on the same column: auto, dict, refine")
    args = ap.parse_args()
    only = set(args.only.split(","))
    n = args.rows
    torch.cuda.set_device(0)
    ctx = Context.get(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.stream = stream.cuda_stream
    gen = torch.Generator(device="cuda")
    gen.manual_seed(SEED)

    if "c1" in only or "cmp" in only:
        vals_t = torch.randint(-100, 101, (n,), dtype=torch.int64, device="cuda", generator=gen)
        vvalid_t, v_nulls = make_validity(torch, n, gen)
        values = DeviceArray.from_pointers(ctx, pa.int64(), n, vals_t.data_ptr(), validity_ptr=vvalid_t.data_ptr(), null_count=v_nulls)
        if "c1" in only:
            for sel in (0.5, 0.01, 0.999):
                m8 = (n + 7) // 8 * 8
                mask_bits = torch.empty(m8 // 8 + 64, dtype=torch.uint8, device="cuda")
                from bench import pack_bits
                chunk = 1 << 27
                for lo in range(0, m8, chunk):
                    m = min(chunk, m8 - lo)
                    mask_bits[lo // 8:(lo + m) // 8] = pack_bits(torch, torch.rand(m, device="cuda", generator=gen) < sel)
                mask = DeviceArray.from_pointers(ctx, pa.bool_(), n, mask_bits.data_ptr())
                ms = timed(stream, lambda: bc.filter(values, mask), args.reps)
                out_len = len(bc.filter(values, mask))
                s = out_len / n
                report(f"c1 filter int64 sel={sel}", n, ms, n * (8 + 0.125 + 0.125) + out_len * 8.125, {"selectivity": s})
                del mask, mask_bits
        if "cmp" in only:
            other_t = torch.randint(-100, 101, (n,), dtype=torch.int64, device="cuda", generator=gen)
            other = DeviceArray.from_pointers(ctx, pa.int64(), n, other_t.data_ptr())
            ms = timed(stream, lambda: bc.greater(values, other), args.reps)
            report("compare greater(int64,int64)", n, ms, n * (16 + 0.125 + 0.25))
            ms = timed(stream, lambda: bc.sum(values), args.reps)
            report("f2 sum/mean/min_max state of int64 (b2_reduce)", n, ms, n * (8 + 0.125))
            del other, other_t
        del values, vals_t, vvalid_t

    if "c3" in only:
        groups = args.groups or (10_000_000 if n >= 100_000_000 else max(1000, n // 100))
        keys_t = torch.randint(0, groups, (n,), dtype=torch.int64, device="cuda", generator=gen)
        vals_t = torch.randint(-100, 101, (n,), dtype=torch.int64, device="cuda", generator=gen)
        vvalid_t, v_nulls = make_validity(torch, n, gen)
        keys = DeviceArray.from_pointers(ctx, pa.int64(), n, keys_t.data_ptr())
        vals = DeviceArray.from_pointers(ctx, pa.int64(), n, vals_t.data_ptr(), validity_ptr=vvalid_t.data_ptr(), null_count=v_nulls)

        paths = {}

        def fused():
            g = bc.GroupBySumCount(pa.int64(), pa.int64(), expected_groups=groups, ctx=ctx)
            g.consume(keys, vals)
            paths["counts"] = g.path_counts()
            return g.finalize()
        ms = timed(stream, fused, args.reps, warmup=1)
        ng = len(fused()[0])
        report("c3 group-by sum+count (fused table)", n, ms, n * 16.125 + ng * 24.25,
               {"groups": ng, "paths": paths["counts"]})
        if args.fused_only:
            return

        def unfused():
            return bc.group_by([keys], [("hash_sum", vals, None), ("hash_count", vals, None)], fused=False)
        ms = timed(stream, unfused, max(1, args.reps - 1), warmup=1)
        report("c3 group-by sum+count (Grouper + 2 HashAggregators)", n, ms, n * 16.125 + ng * 24.25, {"groups": ng})
        del keys, vals, keys_t, vals_t, vvalid_t

    if "c3u" in only:
        # group-by with a large_utf8 key: n/2 strings from 1M distinct words of 8-16 B (bench.make_word_column)
        from bench import make_word_column
        m = n // 2
        vocab = 1_000_000 if m >= 10_000_000 else max(100, m // 100)
        kid, offs, data, total = make_word_column(torch, gen, m, vocab)
        vals_t = torch.randint(-100, 101, (m,), dtype=torch.int64, device="cuda", generator=gen)
        vvalid_t, v_nulls = make_validity(torch, m, gen)
        skeys = DeviceArray.from_pointers(ctx, pa.large_string(), m, offs.data_ptr(), data2_ptr=data.data_ptr())
        vals = DeviceArray.from_pointers(ctx, pa.int64(), m, vals_t.data_ptr(), validity_ptr=vvalid_t.data_ptr(), null_count=v_nulls)
        ms = timed(stream, lambda: bc.group_by([skeys], [("hash_sum", vals, None), ("hash_count", vals, None)], fused=False),
                   max(1, args.reps - 1), warmup=1)
        L = total / m
        report("c3u group-by sum+count, large_utf8 key (1M distinct words)", m, ms, m * (8 + L + 8.125) + vocab * (8 + L + 16.25),
               {"groups": vocab, "mean_len": L})
        ms = timed(stream, lambda: bc.dictionary_encode(skeys), max(1, args.reps - 1), warmup=1)
        report("f1 dictionary_encode large_utf8 (1M distinct words)", m, ms, m * (8 + L + 4) + vocab * (8 + L), {"mean_len": L})
        del skeys, vals, kid, offs, data, vals_t, vvalid_t

    if "join" in only:
        # inner hash join: n/2 probe rows (int64 keys, uniform over 1.25x the build keys, so 80 % match) against 10M unique build keys
        m = n // 2
        nb = 10_000_000 if m >= 100_000_000 else max(1000, m // 50)
        build_t = torch.randperm(int(nb * 1.25), device="cuda", generator=gen)[:nb].to(torch.int64)
        probe_t = torch.randint(0, int(nb * 1.25), (m,), dtype=torch.int64, device="cuda", generator=gen)
        build = DeviceArray.from_pointers(ctx, pa.int64(), nb, build_t.data_ptr())
        probe = DeviceArray.from_pointers(ctx, pa.int64(), m, probe_t.data_ptr())
        ms = timed(stream, lambda: bc.hash_join_indices([probe], [build], "inner"), max(1, args.reps - 1), warmup=1)
        li, ri = bc.hash_join_indices([probe], [build], "inner")
        pairs = len(li)
        # parity: every emitted pair has equal keys, and the pair count equals the number of probe keys present in the build side
        lt = torch.as_tensor(_cai(li.buffers[1].ptr, pairs, "<u4"), device="cuda").to(torch.int64)
        rt = torch.as_tensor(_cai(ri.buffers[1].ptr, pairs, "<u4"), device="cuda").to(torch.int64)
        present = torch.zeros(int(nb * 1.25), dtype=torch.bool, device="cuda")
        present[build_t] = True
        ok = bool((probe_t[lt] == build_t[rt]).all().item()) and pairs == int(present[probe_t].sum().item())
        report("join inner: 10M unique int64 build keys, probe keys 80 % matching", m, ms, m * 8 + nb * 8 + pairs * 8,
               {"build_rows": nb, "pairs": pairs, "parity_ok": ok})
        del build, probe, build_t, probe_t, li, ri, lt, rt, present

    if "c4" in only:
        m = min(n, (1 << 30) - 1)
        for name, lo, hi in (("wide [-2^62,2^62)", -2**62, 2**62), ("narrow [0,4095]", 0, 4096)):
            keys_t = torch.randint(lo, hi, (m,), dtype=torch.int64, device="cuda", generator=gen)
            kvalid_t, k_nulls = make_validity(torch, m, gen)
            keys = DeviceArray.from_pointers(ctx, pa.int64(), m, keys_t.data_ptr(), validity_ptr=kvalid_t.data_ptr(), null_count=k_nulls)
            ms = timed(stream, lambda: bc.array_sort_indices(keys), max(1, args.reps - 1), warmup=1)
            report(f"c4 sort_indices int64 {name}", m, ms, m * 16.125)
            del keys, keys_t, kvalid_t
            ctx.trim()

    sort_utf8 = [(c, None) for c in ("sort_utf8_unique", "sort_utf8_prefix") if c in only]
    if "sort_utf8" in only:
        m = n // 2
        vocabs = [int(v) for v in args.vocab.split(",") if v] or [1_000_000 if m >= 10_000_000 else max(100, m // 100)]
        sort_utf8 = [("sort_utf8", v) for v in vocabs] + sort_utf8
    for cfg, vocab in sort_utf8:
        if cfg == "sort_utf8":  # the c3u column: distinct words of 8-16 B
            from bench import make_word_column
            m = n // 2
            _, offs, data, total = make_word_column(torch, gen, m, vocab)
            label = f"sort_utf8 sort_indices large_utf8 ({vocab} distinct words of 8-16 B)"
        else:
            m = n // 5 if cfg == "sort_utf8_unique" else n // 10
            prefix = 0 if cfg == "sort_utf8_unique" else 40
            lens = torch.randint(8, 33, (m,), dtype=torch.int64, device="cuda", generator=gen) + prefix
            offs = torch.zeros(m + 1, dtype=torch.int64, device="cuda")
            torch.cumsum(lens, 0, out=offs[1:])
            total = int(offs[-1].item())
            data = torch.randint(97, 123, (total + 64,), dtype=torch.uint8, device="cuda", generator=gen)
            if prefix:
                starts = offs[:-1]
                for k in range(prefix):
                    data[starts + k] = 120  # 'x'
            del lens
            label = ("sort_utf8_unique sort_indices large_utf8 (random 8-32 B)" if not prefix else
                     "sort_utf8_prefix sort_indices large_utf8 (40-byte common prefix + 8-32 random B)")
        strs = DeviceArray.from_pointers(ctx, pa.large_string(), m, offs.data_ptr(), data2_ptr=data.data_ptr())
        L = total / m
        for p in args.string_paths.split(","):
            if p == "auto":
                os.environ.pop("B2_SORT_STRINGS_PATH", None)
            else:
                os.environ["B2_SORT_STRINGS_PATH"] = p
            ms = timed(stream, lambda: bc.array_sort_indices(strs), max(1, args.reps - 1), warmup=1)
            out = bc.array_sort_indices(strs)
            ok = sort_parity(ctx, out, m, offs, data, gen)
            # algorithmic bytes: offsets + characters read once, the uint64 permutation written once
            report(label, m, ms, m * (8 + L + 8), {"mean_len": L, "parity_checksum_ok": ok, "path": bc.sort_strings_path(strs),
                                                   "path_forced": p != "auto", **card()})
            del out
        os.environ.pop("B2_SORT_STRINGS_PATH", None)
        del strs, offs, data
        ctx.trim()

    if "c5" in only:
        m = n // 2
        lens = torch.randint(0, 33, (m,), dtype=torch.int64, device="cuda", generator=gen)
        offs = torch.zeros(m + 1, dtype=torch.int64, device="cuda")
        torch.cumsum(lens, 0, out=offs[1:])
        total = int(offs[-1].item())
        del lens
        data = torch.randint(97, 123, (total + 64,), dtype=torch.uint8, device="cuda", generator=gen)
        svalid_t, s_nulls = make_validity(torch, m, gen)
        strs = DeviceArray.from_pointers(ctx, pa.large_string(), m, offs.data_ptr(), validity_ptr=svalid_t.data_ptr(), null_count=s_nulls,
                                         data2_ptr=data.data_ptr())
        from bench import pack_bits
        m8 = (m + 7) // 8 * 8
        mask_bits = torch.empty(m8 // 8 + 64, dtype=torch.uint8, device="cuda")
        chunk = 1 << 27
        for lo in range(0, m8, chunk):
            c = min(chunk, m8 - lo)
            mask_bits[lo // 8:(lo + c) // 8] = pack_bits(torch, torch.rand(c, device="cuda", generator=gen) < 0.5)
        mask = DeviceArray.from_pointers(ctx, pa.bool_(), m, mask_bits.data_ptr())
        ms = timed(stream, lambda: bc.filter(strs, mask), args.reps, warmup=1)
        L = total / m
        report("c5 filter large_utf8 s=0.5", m, ms, m * (8 + L + 0.25) + 0.5 * m * (8 + L + 0.125), {"mean_len": L})
        del strs, offs, data, svalid_t, mask, mask_bits
        # dictionary-encoded Take: int32 index column, int64 take-indices
        dict_idx_t = torch.randint(0, 1_000_000, (m,), dtype=torch.int32, device="cuda", generator=gen)
        col = DeviceArray.from_pointers(ctx, pa.int32(), m, dict_idx_t.data_ptr())
        take_idx_t = torch.randint(0, m, (m,), dtype=torch.int64, device="cuda", generator=gen)
        take_idx = DeviceArray.from_pointers(ctx, pa.int64(), m, take_idx_t.data_ptr())
        ms = timed(stream, lambda: bc.take(col, take_idx), args.reps, warmup=1)
        report("c5 dictionary take (int32 index column, random int64 idx)", m, ms, m * (8 + 4 + 4))
        del col, take_idx, dict_idx_t, take_idx_t

    if "f1" in only:
        # SURVEY 8f rank 1: produce config 5's dictionary column on the device
        m = n // 2
        distinct = 1_000_000
        keys_t = torch.randint(0, distinct, (m,), dtype=torch.int64, device="cuda", generator=gen)
        kvalid_t, k_nulls = make_validity(torch, m, gen)
        col = DeviceArray.from_pointers(ctx, pa.int64(), m, keys_t.data_ptr(), validity_ptr=kvalid_t.data_ptr(), null_count=k_nulls)
        ms = timed(stream, lambda: bc.dictionary_encode(col), args.reps, warmup=1)
        nd = len(bc.unique(col))
        report("f1 dictionary_encode int64 (1M distinct, null_p 0.1)", m, ms, m * (8 + 0.125 + 4 + 0.125) + nd * 8, {"dictionary": nd})
        ms = timed(stream, lambda: bc.value_counts(col), args.reps, warmup=1)
        report("f1 value_counts int64 (1M distinct, null_p 0.1)", m, ms, m * (8 + 0.125) + nd * 16, {"dictionary": nd})


if __name__ == "__main__":
    main()
