#!/usr/bin/env python
"""bench.py — rows/sec of the hot path on synthetic TPC-DS-shaped batches (BASELINE.json metric:
"rows/sec on TPC-DS q1 hash-agg+filter at 1/2/4/8 B200; HBM GB/s vs 8 TB/s").

Headline workload (config.workload = "M2", SURVEY.md §8d): the q1-shaped FUSED FilterExec -> HashAggregateExec:
    Filter[f >= 200, f <= 399] (s = 0.2) -> SUM(v) GROUP BY k1, k2       f ~ U[0,1000), k1 ~ U[0,2^17), k2 ~ U[0,8),
    v ~ U[-1e6,1e6), all int64, `rows` rows per GPU (default 10^9), 2^20 groups; 32 B/row read once.
A step = one complete aggregation of the batch: Partial -> (murmur3 pmod N exchange when N > 1) -> Final, results pulled.
`extra` carries the other two §8d shapes, each with its own roofline: M1 (BASELINE configs[1]: SUM(v), COUNT(v) GROUP BY k,
1M groups, 16 B/row) and M0 (configs[0] shape: Filter[a < 500] -> Project[a, a + b], 24 B/row).

  value         whole-job rows/s with the input already resident in HBM (push_device)
  e2e           the same through the host-buffer C ABI (b200q_op_push of host Arrow batches, result pulled back to the host);
                .value = large pinned batches, .pageable_10k = 10,000-row pageable batches (the real FFIReaderExec shape,
                ffi_reader_exec.rs:163-194) through the library's pinned staging ring
  roofline      HBM: algorithmic bytes / CUDA-event time of the dominant kernel (measured inside the library on the op's stream)
  cpu_baseline  oracle/cpu_ref.c (restatement of the reference CPU algorithm) on this box's host cores, best thread count
  verified      every timed workload's LAST result is checked after the timed region against an independent torch
                computation (per-group sums / counts, group ownership disjoint across ranks); a mismatch exits non-zero

`--impl reference` times the CPU restatement alone on the same M2 workload (the Rust reference cannot be built here).
`--dump-outputs DIR` writes the headline's last timed result as DIR/k1.npy, k2.npy, sum_v.npy (float64, rows in key order);
the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True                     # the benchmark leaves the source tree as it found it (it may be read-only)

METRIC = "rows/sec on TPC-DS q1 hash-agg+filter at 1/2/4/8 B200; HBM GB/s vs 8 TB/s"
CARD = 1 << 20
K1_CARD, K2_CARD = 1 << 17, 1 << 3
F_LO, F_HI = 200, 399
LAUNCH_ROWS = 1 << 27                      # b200q_conf.max_launch_rows default: rows per update-kernel launch
WORKLOADS = {
    "M2": "M2: fused FilterExec[f>=200, f<=399] (s=0.2) -> HashAggregateExec SUM(v) GROUP BY k1,k2; f~U[0,1000), k1~U[0,2^17), k2~U[0,8), v~U[-1e6,1e6) int64 (SURVEY §8d M2, the q1 shape of the metric)",
    "M1": "M1: HashAggregateExec SUM(v),COUNT(v) GROUP BY k; k~U[0,2^20) int64, v~U[-1e6,1e6) int64 (BASELINE.json configs[1])",
    "M0": "M0: FilterExec[a<500] (s=0.5) -> ProjectExec[a, a+b]; a~U[0,1000), b~U[-2^31,2^31) int64 (BASELINE.json configs[0] shape)",
}
WORKLOADS["M3"] = "M3: ShuffleWriterExec 200-way hash partition (murmur3 seed 42 pmod 200 on k1) + batch_serde encode of 4 int64 columns, output kept in HBM (BASELINE.json configs[3], map side)"
WORKLOADS["M4"] = "M4: HashJoinExec store_sales x date_dim (73,049-row map side, unique key), inner, probe side 4 int64 columns, 7 output columns (BASELINE.json configs[3], join)"
ALG_BYTES_PER_ROW = {"M2": 32.0, "M1": 16.0, "M0": 24.0, "M3": 64.0, "M4": 88.0}


def env_int(name, default):
    return int(os.environ.get(name, default))


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0])); self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True); self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=10)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


# ---------------------------------------------------------------------------------------------------------------------
# plans (the reference's protobuf, built by the host mirror of the reference constructors)
# ---------------------------------------------------------------------------------------------------------------------
def build_plans(workload):
    from blaze_b200 import exprs as E, plans as PL, types as T
    if workload == "M0":
        ins = T.Schema([T.Field("a", T.int64, False), T.Field("b", T.int64, False)])
        A, B = E.Column("a"), E.Column("b")
        p = PL.ProjectExec([(A, "a"), (E.BinaryExpr(A, "Plus", B), "c")], PL.FilterExec([E.BinaryExpr(A, "Lt", E.Literal(500, T.int64))], PL.MemoryExec(ins)))
        return dict(single=p.plan_bytes(), names=["a", "b"])
    if workload == "M1":
        names = ["k", "v"]
        ins = T.Schema([T.Field(n, T.int64, False) for n in names])
        g = [E.GroupingExpr("k", E.Column("k"))]
        mk = lambda mode, ch: [E.AggExpr("sum_v", mode, PL.create_agg(E.AGG_SUM, ch, ins, T.int64)),
                               E.AggExpr("count_v", mode, PL.create_agg(E.AGG_COUNT, ch, ins, T.int64))]
        child = lambda leaf: leaf
    else:
        names = ["f", "k1", "k2", "v"]
        ins = T.Schema([T.Field(n, T.int64, False) for n in names])
        g = [E.GroupingExpr("k1", E.Column("k1")), E.GroupingExpr("k2", E.Column("k2"))]
        mk = lambda mode, ch: [E.AggExpr("sum_v", mode, PL.create_agg(E.AGG_SUM, ch, ins, T.int64))]
        preds = [E.BinaryExpr(E.Column("f"), "GtEq", E.Literal(F_LO, T.int64)), E.BinaryExpr(E.Column("f"), "LtEq", E.Literal(F_HI, T.int64))]
        child = lambda leaf: PL.FilterExec(preds, leaf)
    leaf = PL.MemoryExec(ins)
    partial = PL.AggExec(PL.HashAgg, g, mk(E.PARTIAL, [E.Column("v")]), True, child(leaf))
    final = PL.AggExec(PL.HashAgg, g, mk(E.FINAL, [E.placeholder(T.int64)]), False, partial)
    partial_col = PL.AggExec(PL.HashAgg, g, mk(E.PARTIAL, [E.Column("v")]), True, child(leaf), columnar_state=True)
    final_col = PL.AggExec(PL.HashAgg, g, mk(E.FINAL, [E.placeholder(T.int64)]), False, PL.MemoryExec(partial_col.schema()))
    return dict(single=final.plan_bytes(), partial_col=partial_col.plan_bytes(), final_col=final_col.plan_bytes(), names=names, nkeys=len(g))


def gen_columns(workload, torch, rows, dev, seed):
    gen = torch.Generator(device=dev); gen.manual_seed(seed)
    ri = lambda lo, hi: torch.randint(lo, hi, (rows,), dtype=torch.int64, device=dev, generator=gen)
    if workload == "M0":
        return [ri(0, 1000), ri(-2**31, 2**31)]
    if workload == "M1":
        return [ri(0, CARD), ri(-10**6, 10**6)]
    return [ri(0, 1000), ri(0, K1_CARD), ri(0, K2_CARD), ri(-10**6, 10**6)]


class CudaView:
    """zero-copy torch view of a device buffer returned by pull_device"""

    def __init__(self, ptr, nbytes, owner):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}
        self.owner = owner


def device_cols(dev_array, torch):
    """ArrowDeviceArray (struct of int64 columns) -> [int64 tensors] (views: keep dev_array alive)"""
    a = dev_array.array
    out = []
    for i in range(a.n_children):
        c = a.children[i].contents
        if c.length == 0:
            out.append(torch.zeros(0, dtype=torch.int64, device="cuda")); continue
        out.append(torch.as_tensor(CudaView(c.buffers[1], c.length * 8, dev_array), device="cuda").view(torch.int64))
    return out


class Runner:
    """one workload on this rank: device-resident step, host-buffer step, verification"""

    def __init__(self, workload, torch, dist, native, rank, world, local, rows, exchange):
        self.w, self.torch, self.dist, self.native = workload, torch, dist, native
        self.rank, self.world, self.local, self.rows, self.ex = rank, world, local, rows, exchange
        self.dev = torch.device("cuda", local)
        self.plans = build_plans(workload)
        self.cols = gen_columns(workload, torch, rows, self.dev, {"M0": 42, "M1": 44, "M2": 46}[workload] + 1000 * rank)
        torch.cuda.synchronize()
        self.conf = native.default_conf(agg_initial_groups=CARD)
        self.conf_col = native.default_conf(agg_initial_groups=CARD, partial_state_columnar=1)
        self.stats = {"launches": 0, "hot_ns": 0, "hot_rows": 0, "hot_launches": 0}
        self.last = None                                   # (ArrowDeviceArray, ...) of the last step, kept for verification
        self.h2d = self.d2h = 0

    def reset_stats(self):
        for k in self.stats:
            self.stats[k] = 0

    def _acc(self, m, hot=True):
        self.stats["launches"] += m["gpu_kernel_launches"]
        if hot:
            self.stats["hot_ns"] += m["hot_kernel_ns"]; self.stats["hot_rows"] += m["hot_kernel_rows"]; self.stats["hot_launches"] += m["hot_kernel_launches"]

    def _drop_last(self):
        if self.last is not None:
            for d in self.last:
                self.native.release_device_array(d)
            self.last = None

    def _input_batch(self):
        n = self.rows
        return self.native.DeviceBatch([(c.data_ptr(), 0, n) for c in self.cols], n, self.local, keepalive=tuple(self.cols))

    def _pull_all_device(self, op):
        outs = []
        while True:
            o = op.pull_device()
            if o is None:
                return outs
            outs.append(o)

    def step_device(self):
        """input resident in HBM -> result resident in HBM (kept for the verification of the last step)"""
        native = self.native
        self._drop_last()
        if os.environ.get("B200Q_BENCH_PHASES") and self.world == 1:                       # where a step's time goes (host clock, each phase synchronised)
            t = [time.perf_counter()]
            def lap(): self.torch.cuda.synchronize(); t.append(time.perf_counter())
            op = native.NativeOp(self.plans["single"], self.conf, self.local); lap()
            op.push_device(self._input_batch()); op.sync(); lap()
            op.finish(); lap()
            self.last = self._pull_all_device(op); lap()
            m = op.metrics(); self._acc(m); op.close(); lap()
            names = ["create", "push(update kernels)", "finish(emit + Final stage)", "pull", "destroy"]
            sys.stderr.write("phases[%s] " % self.w + ", ".join(f"{n}={1e3 * (b - a):.3f}ms" for n, a, b in zip(names, t, t[1:])) + f", hot_kernels={m['hot_kernel_ns'] / 1e6:.3f}ms, launches={m['gpu_kernel_launches']}\n")
            return
        if self.w == "M0" or self.world == 1:
            with native.NativeOp(self.plans["single"], self.conf, self.local) as op:
                op.push_device(self._input_batch())
                op.finish()
                self.last = self._pull_all_device(op)
                self._acc(op.metrics())
            return
        if os.environ.get("B200Q_BENCH_PHASES"):                                               # N > 1: partial op / exchange / final op (host clock, synchronised)
            t = [time.perf_counter()]
            def lap(): self.torch.cuda.synchronize(); t.append(time.perf_counter())
            part = self._partial_device(); lap()
            out, schema = part
            recv = self.ex.shuffle(schema, out, self.plans["nkeys"]); lap()
            with native.NativeOp(self.plans["final_col"], self.conf_col, self.local) as op:
                lap(); op.push_device_array(recv); lap(); op.finish(); lap(); res = op.pull_device(); self._acc(op.metrics(), hot=False); lap()
            lap()
            names = ["partial op (create..destroy)", "exchange", "final create", "final push", "final finish", "final pull", "final destroy"]
            if self.rank == 0: sys.stderr.write("phases[%s N=%d] " % (self.w, self.world) + ", ".join(f"{n}={1e3 * (b - a):.3f}ms" for n, a, b in zip(names, t, t[1:])) + "\n")
            self.last = [res]
            return
        self.last = [self._exchange_and_final(self._partial_device())]

    def _partial_device(self):
        native = self.native
        with native.NativeOp(self.plans["partial_col"], self.conf_col, self.local) as op:
            op.push_device(self._input_batch())
            op.finish()
            out = op.pull_device()
            self._acc(op.metrics())
            schema = op.output_schema()
        return out, schema

    def _exchange_and_final(self, partial):
        """Partial states -> owner rank = pmod(murmur3(keys, 42), N) (b200q_exchange_shuffle: NCCL AllToAllv) -> Final"""
        native = self.native
        out, schema = partial
        l0 = self.ex.kernel_launches()
        recv = self.ex.shuffle(schema, out, self.plans["nkeys"])
        self.stats["launches"] += self.ex.kernel_launches() - l0
        with native.NativeOp(self.plans["final_col"], self.conf_col, self.local) as op:
            op.push_device_array(recv)
            op.finish()
            res = op.pull_device()
            self._acc(op.metrics(), hot=False)
        return res

    # ---- host-buffer path (public C ABI with HOST Arrow batches)
    def step_host(self, host_batches):
        native = self.native
        n_out = 0
        if self.w == "M0" or self.world == 1:
            with native.NativeOp(self.plans["single"], self.conf, self.local) as op:
                for b in host_batches:
                    op.push(b)
                op.finish()
                while True:
                    o = op.pull()
                    if o is None:
                        break
                    n_out += o.num_rows
                m = op.metrics()
                self.h2d, self.d2h = m["h2d_bytes"], m["d2h_bytes"]
            return n_out
        with native.NativeOp(self.plans["partial_col"], self.conf_col, self.local) as op:
            for b in host_batches:
                op.push(b)
            op.finish()
            out = op.pull_device()
            schema = op.output_schema()
            self.h2d = op.metrics()["h2d_bytes"]
        recv = self.ex.shuffle(schema, out, self.plans["nkeys"])
        with native.NativeOp(self.plans["final_col"], self.conf_col, self.local) as op:
            op.push_device_array(recv)
            op.finish()
            while True:
                o = op.pull()
                if o is None:
                    break
                n_out += o.num_rows
            self.d2h = op.metrics()["d2h_bytes"]
        return n_out

    # ---- verification of the last device-resident step (outside every timed region)
    def verify(self):
        torch, dist, world = self.torch, self.dist, self.world
        res = [device_cols(d, torch) for d in (self.last or [])]
        if self.w == "M0":
            a, b = self.cols
            mask = a < 500
            exp_a = a[mask]; exp_c = exp_a + b[mask]
            got_a = torch.cat([r[0] for r in res]) if res else exp_a[:0]
            got_c = torch.cat([r[1] for r in res]) if res else exp_c[:0]
            ok = got_a.numel() == exp_a.numel() and bool(torch.equal(got_a, exp_a)) and bool(torch.equal(got_c, exp_c))
            return ok, {"out_rows": int(got_a.numel())}
        if self.w == "M1":
            k, v = self.cols
            idx, vv = k, v
            ones = torch.ones_like(v)
        else:
            f, k1, k2, v = self.cols
            mask = (f >= F_LO) & (f <= F_HI)
            idx, vv = (k1 * K2_CARD + k2)[mask], v[mask]
            ones = torch.ones_like(vv)
        exp_sum = torch.zeros(CARD, dtype=torch.int64, device=self.dev).index_add_(0, idx, vv)
        exp_cnt = torch.zeros(CARD, dtype=torch.int64, device=self.dev).index_add_(0, idx, ones)
        if world > 1:
            dist.all_reduce(exp_sum); dist.all_reduce(exp_cnt)
        cols = res[0] if res else None
        seen = torch.zeros(CARD, dtype=torch.int64, device=self.dev)
        ok = True
        n_groups = 0
        if cols is not None and cols[0].numel():
            gi = cols[0] if self.w == "M1" else cols[0] * K2_CARD + cols[1]
            n_groups = int(gi.numel())
            ok = ok and bool(((gi >= 0) & (gi < CARD)).all())
            seen.index_add_(0, gi, torch.ones_like(gi))
            gsum = cols[1] if self.w == "M1" else cols[2]
            ok = ok and bool(torch.equal(gsum, exp_sum[gi]))                          # per-group SUM, bit-exact
            if self.w == "M1":
                ok = ok and bool(torch.equal(cols[2], exp_cnt[gi]))                   # per-group COUNT
            ok = ok and bool((exp_cnt[gi] > 0).all())
        tot = torch.tensor([n_groups], dtype=torch.int64, device=self.dev)
        if world > 1:
            dist.all_reduce(seen); dist.all_reduce(tot)
        ok = ok and int(seen.max()) <= 1                                              # every group has exactly one owner
        ok = ok and int(tot.item()) == int((exp_cnt > 0).sum())                       # and no group is missing
        flag = torch.tensor([1 if ok else 0], dtype=torch.int64, device=self.dev)
        if world > 1:
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        return bool(flag.item()), {"groups": int(tot.item()), "sum_of_sums": int(exp_sum.sum().item())}

    def close(self):
        self._drop_last()
        self.cols = None


def torch_murmur3_pid(torch, k, parts):
    """pmod(murmur3_x86_32(le_bytes(int64 k), seed 42), parts) with int64 tensor arithmetic (hash/mur.rs:19-87) — independent of the library's kernel"""
    M = 0xFFFFFFFF
    def mul(a, b): return (a * b) & M
    def rotl(x, r): return ((x << r) | (x >> (32 - r))) & M
    def mix_k1(k1): return mul(rotl(mul(k1, 0xcc9e2d51), 15), 0x1b873593)
    def mix_h1(h1, k1): return (mul(rotl(h1 ^ k1, 13), 5) + 0xe6546b64) & M
    lo, hi = k & M, (k >> 32) & M
    h = mix_h1(mix_h1(torch.full_like(k, 42), mix_k1(lo)), mix_k1(hi))
    h = h ^ 8
    h = h ^ (h >> 16); h = mul(h, 0x85ebca6b); h = h ^ (h >> 13); h = mul(h, 0xc2b2ae35); h = h ^ (h >> 16)
    signed = torch.where(h >= 2**31, h - 2**32, h)
    return torch.remainder(signed, parts)


def extra_shuffle_and_join(torch, dist, native, world, local, dev, rows, steps, warmup, peak, peak_src, seed):
    """M3 (shuffle write) and M4 (hash join): device-resident steps, kernel time from the library's own CUDA events, verified"""
    from blaze_b200 import exprs as E, plans as PL, types as T
    out = []
    gen = torch.Generator(device=dev); gen.manual_seed(seed)
    ri = lambda lo, hi: torch.randint(lo, hi, (rows,), dtype=torch.int64, device=dev, generator=gen)
    ND = 73049
    cols = [ri(0, ND), ri(0, K1_CARD), ri(0, K2_CARD), ri(-10**6, 10**6)]                    # ss_sold_date_sk, k1, k2, v
    names = ["sk", "k1", "k2", "v"]
    ins = T.Schema([T.Field(n, T.int64, False) for n in names])
    batch = lambda: native.DeviceBatch([(c.data_ptr(), 0, rows) for c in cols], rows, local, keepalive=tuple(cols))
    stats = {"ns": 0, "rows": 0, "launches": 0, "all": 0}
    # ---- M3
    P = 200
    plan3 = PL.ShuffleWriterExec(PL.MemoryExec(ins), ("hash", [E.Column("k1")], P), "", "").plan_bytes()
    conf3 = native.default_conf(shuffle_output_on_device=1)
    keep = {}
    def step3():
        with native.NativeOp(plan3, conf3, local) as op:
            op.push_device(batch()); op.finish()
            m = op.metrics()
            stats["ns"] += m["hot_kernel_ns"]; stats["rows"] += m["hot_kernel_rows"]; stats["launches"] += m["hot_kernel_launches"]; stats["all"] += m["gpu_kernel_launches"]
            keep["chunks"] = [(c["rows"], c["part_rows"], c["part_off"]) for c in op.shuffle_chunks()]
    for _ in range(warmup): step3()
    for k_ in stats: stats[k_] = 0
    ms = timed(torch, dist, world, dev, step3, steps, 0)
    pid = torch_murmur3_pid(torch, cols[1], P)
    exp = torch.bincount(pid, minlength=P).cpu()
    got = torch.zeros(P, dtype=torch.int64)
    for _, pr, _ in keep["chunks"]: got += torch.tensor(pr, dtype=torch.int64)
    rec = lambda m: (1 if m < 128 else 2 if m < 16384 else 3 if m < 2**21 else 4) + 4 + 32 * m
    exp_bytes = sum(((t - 1) // 10000) * rec(10000) + rec(t - ((t - 1) // 10000) * 10000) for _, pr, _ in keep["chunks"] for t in pr if t)
    ok3 = bool(torch.equal(got, exp)) and sum(po[-1] for _, _, po in keep["chunks"]) == exp_bytes
    ach = ALG_BYTES_PER_ROW["M3"] * stats["rows"] / max(1, stats["ns"])
    out.append({"workload": WORKLOADS["M3"], "value": rows * world / (ms * 1e-3), "unit": "rows/s", "ms_per_step": ms, "steps": steps, "warmup": warmup, "rows_per_gpu": rows, "verified": ok3,
                "verification": "rows per partition == bincount of an independent torch murmur3; encoded bytes == the batch_serde size formula (contents: tests/test_gpu_shuffle_writer.py)",
                "gpu_launches": stats["all"], "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": ach / peak, "traffic": None,
                                                           "kernel": "shuffle_pids_kernel + shuffle_encode_kernel", "launches": stats["launches"], "avg_launch_ms": stats["ns"] / max(1, stats["launches"]) / 1e6,
                                                           "alg_bytes_per_row": ALG_BYTES_PER_ROW["M3"]}})
    # ---- M4
    d_sk = torch.arange(ND, dtype=torch.int64, device=dev)
    bcols = [d_sk, 1900 + d_sk // 366, (d_sk // 30) % 12 + 1]
    sd = T.Schema([T.Field(n, T.int64, False) for n in ("d_date_sk", "d_year", "d_moy")])
    build = PL.BroadcastJoinBuildHashMapExec(PL.MemoryExec(sd), [E.Column("d_date_sk")])
    join = PL.BroadcastJoinExec(PL.build_join_schema(ins, sd, PL.JOIN_INNER), PL.MemoryExec(ins), build, [(E.Column("sk"), E.Column("d_date_sk"))], PL.JOIN_INNER, PL.RIGHT_SIDE, True, "m").plan_bytes()
    for k_ in stats: stats[k_] = 0
    def step4():
        with native.NativeOp(build.plan_bytes(), None, local) as bop:                         # the map side is rebuilt every step (73,049 rows)
            bop.push_device(native.DeviceBatch([(c.data_ptr(), 0, ND) for c in bcols], ND, local, keepalive=tuple(bcols))); bop.finish()
            with native.NativeOp(join, None, local) as op:
                op.attach_build(bop)
                op.push_device(batch()); op.finish()
                n_out, ysum = 0, 0
                while True:
                    o = op.pull_device()
                    if o is None: break
                    n_out += o.array.length
                    if keep.get("check"): ysum += int(device_cols(o, torch)[5].sum().item())
                    native.release_device_array(o)
                m = op.metrics()
                stats["ns"] += m["hot_kernel_ns"]; stats["rows"] += m["hot_kernel_rows"]; stats["launches"] += m["hot_kernel_launches"]; stats["all"] += m["gpu_kernel_launches"]
                keep["join"] = (n_out, ysum)
    for _ in range(warmup): step4()
    for k_ in stats: stats[k_] = 0
    ms = timed(torch, dist, world, dev, step4, steps, 0)
    st = dict(stats); keep["check"] = True; step4()
    ok4 = keep["join"] == (rows, int((1900 + cols[0] // 366).sum().item()))
    ach = ALG_BYTES_PER_ROW["M4"] * st["rows"] / max(1, st["ns"])
    out.append({"workload": WORKLOADS["M4"], "value": rows * world / (ms * 1e-3), "unit": "rows/s", "ms_per_step": ms, "steps": steps, "warmup": warmup, "rows_per_gpu": rows, "verified": ok4,
                "verification": "output rows == probe rows (every key matches a unique map key) and SUM(d_year) over the output == SUM(1900 + sk // 366) over the probe side",
                "gpu_launches": st["all"], "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": ach / peak, "traffic": None,
                                                        "kernel": "join_probe_count_kernel + join_probe_fused_kernel (per 2^26-row probe chunk)", "launches": st["launches"],
                                                        "avg_launch_ms": st["ns"] / max(1, st["launches"]) / 1e6, "alg_bytes_per_row": ALG_BYTES_PER_ROW["M4"]}})
    return out, ok3, ok4


def timed(torch, dist, world, dev, fn, steps, warmup):
    """W untimed steps, then exactly K steps between barrier + synchronize, device-timed, max over ranks -> ms per step"""
    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(); torch.cuda.synchronize()
    for _ in range(warmup):
        fn()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.item() / steps


def load_json(path):
    try:
        return json.load(open(path))
    except Exception:
        return None


def roofline_of(workload, stats, rows, peak, peak_src):
    launches = max(1, stats["hot_launches"])
    alg = ALG_BYTES_PER_ROW[workload]
    achieved = alg * stats["hot_rows"] / max(1, stats["hot_ns"])                  # bytes/ns == GB/s
    launch_rows = min(rows, LAUNCH_ROWS)
    traffic, traffic_src = None, None
    tj = load_json(os.path.join(ROOT, "profiles", "r02_traffic.json")) or {}
    ent = tj.get(workload)
    if ent and ent.get("rows_per_launch") == launch_rows:                           # DRAM bytes of ONE launch of the same kernel at the same rows/launch
        traffic, traffic_src = ent["dram_bytes_read"] + ent["dram_bytes_write"], ent.get("source")
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "traffic_source": traffic_src, "kernel": {"M2": "agg_tile_dense_kernel<2,1,2,1>", "M1": "agg_lean_dense_kernel<2,2,1>", "M0": "filter_count_lean + filter_apply_lean (two-pass compaction)"}[workload],
            "launches": stats["hot_launches"], "avg_launch_ms": stats["hot_ns"] / launches / 1e6, "launch_rows": launch_rows,
            "alg_bytes_per_row": alg, "alg_bytes_per_launch": alg * launch_rows}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from blaze_b200 import native
    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    exchange = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        uid = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            uid.copy_(torch.frombuffer(bytearray(native.exchange_unique_id()), dtype=torch.uint8))
        dist.broadcast(uid, 0)
        exchange = native.Exchange(bytes(uid.cpu().numpy().tobytes()), rank, world, local)
    rows = env_int("B200Q_BENCH_ROWS", 1_000_000_000)
    extra_rows = env_int("B200Q_BENCH_EXTRA_ROWS", rows)
    peaks = load_json(os.path.join(ROOT, "MEASURED_PEAKS.json")) or {}
    peak_src = "measured" if "hbm_gbs" in peaks else "fallback"
    peak = float(peaks.get("hbm_gbs", 6650.0))
    failures = []

    # ---- headline: M2 -------------------------------------------------------------------------------------------
    r2 = Runner("M2", torch, dist, native, rank, world, local, rows, exchange)
    for _ in range(args.warmup):
        r2.step_device()
    r2.reset_stats()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms_per_step = timed(torch, dist, world, dev, r2.step_device, args.steps, 0)
    clocks = sampler.stop() if sampler else None
    value = rows * world / (ms_per_step * 1e-3)
    headline_stats = dict(r2.stats)
    ok, info = r2.verify()
    if not ok:
        failures.append("M2")
    verified = {"M2": dict(ok=ok, **info)}
    if args.dump_outputs:
        dump_m2_outputs(torch, dist, r2, args.dump_outputs)

    # ---- e2e: host buffers through the C ABI (M2) -------------------------------------------------------------------
    import numpy as np
    import pyarrow as pa
    numa = bind_to_gpu_numa(torch, local)                  # pinned buffers on the GPU's NUMA node (first touch)
    e2e_batch = env_int("B200Q_BENCH_E2E_BATCH_ROWS", 1 << 24)
    e2e_rows = env_int("B200Q_BENCH_E2E_ROWS", 0)
    if e2e_rows <= 0:                                      # all ranks together stay below min(48 GB, 30 % of MemAvailable) of pinned memory
        budget = min(48e9, 0.30 * mem_available_bytes())
        e2e_rows = int(min(rows, 1 << 29, max(e2e_batch, budget / (32 * world) // e2e_batch * e2e_batch)))
    host = [torch.empty(e2e_rows, dtype=torch.int64, pin_memory=True) for _ in r2.cols]
    for h, c in zip(host, r2.cols):
        h.copy_(c[:e2e_rows])
    torch.cuda.synchronize()
    schema = pa.schema([pa.field(n, pa.int64(), False) for n in r2.plans["names"]])

    def host_batches(tensors, n, step, copy=False):
        out = []
        for b in range(0, n, step):
            m = min(step, n - b)
            if copy:                                       # pageable: ordinary (unpinned) numpy memory, as a JVM-exported batch would be
                arrs = [pa.array(t.numpy()[b:b + m].copy()) for t in tensors]
            else:
                arrs = [pa.Array.from_buffers(pa.int64(), m, [None, pa.foreign_buffer(t.data_ptr() + 8 * b, 8 * m, base=t)]) for t in tensors]
            out.append(pa.RecordBatch.from_arrays(arrs, schema=schema))
        return out
    hb = host_batches(host, e2e_rows, e2e_batch)
    e2e_steps = max(1, min(args.steps, 5))
    ms_e2e = timed(torch, dist, world, dev, lambda: r2.step_host(hb), e2e_steps, max(1, min(args.warmup, 2)))
    e2e = {"value": e2e_rows * world / (ms_e2e * 1e-3), "unit": "rows/s", "h2d_bytes_per_step": r2.h2d, "d2h_bytes_per_step": r2.d2h,
           "rows_per_gpu": e2e_rows, "host_batch_rows": e2e_batch, "host_memory": "pinned", "steps": e2e_steps, "host_numa_node": numa}
    # 10,000-row pageable batches: the shape FFIReaderExec really hands over (<= BATCH_SIZE rows, ordinary heap memory)
    small_rows = int(min(e2e_rows, env_int("B200Q_BENCH_E2E_SMALL_ROWS", 1 << 26)))
    hb_small = host_batches(host, small_rows, 10000, copy=True)
    ms_small = timed(torch, dist, world, dev, lambda: r2.step_host(hb_small), max(1, min(args.steps, 3)), 1)
    e2e["pageable_10k"] = {"value": small_rows * world / (ms_small * 1e-3), "unit": "rows/s", "h2d_bytes_per_step": r2.h2d, "d2h_bytes_per_step": r2.d2h,
                           "rows_per_gpu": small_rows, "host_batch_rows": 10000, "host_memory": "pageable, staged into the library's pinned ring (staging_rows = 2^20)"}
    del hb_small

    # ---- CPU baseline on the same workload (rank 0, N = 1 only) -----------------------------------------------------
    cpu = None
    os.sched_setaffinity(0, range(os.cpu_count() or 1))
    if world == 1 and rank == 0:
        sample = int(min(e2e_rows, env_int("B200Q_BENCH_CPU_ROWS", 1 << 28)))
        cpu = cpu_baseline_m2([h.numpy()[:sample] for h in host], sample)
    del hb, host
    r2.close(); del r2
    torch.cuda.empty_cache()

    # ---- extras: M1 and M0, each timed, verified and with its own roofline ------------------------------------------
    extra = []
    ex_steps, ex_warm = max(1, min(args.steps, 10)), max(3, min(args.warmup, 3))
    for w in ("M1", "M0"):
        r = Runner(w, torch, dist, native, rank, world, local, extra_rows, exchange)
        for _ in range(ex_warm):
            r.step_device()
        r.reset_stats()
        ms = timed(torch, dist, world, dev, r.step_device, ex_steps, 0)
        ok, info = r.verify()
        if not ok:
            failures.append(w)
        verified[w] = dict(ok=ok, **info)
        extra.append({"workload": WORKLOADS[w], "value": extra_rows * world / (ms * 1e-3), "unit": "rows/s", "ms_per_step": ms, "steps": ex_steps, "warmup": ex_warm,
                      "rows_per_gpu": extra_rows, "verified": ok, "gpu_launches": r.stats["launches"], "roofline": roofline_of(w, r.stats, extra_rows, peak, peak_src)})
        r.close(); del r
        torch.cuda.empty_cache()

    x_rows = env_int("B200Q_BENCH_X_ROWS", min(extra_rows, 1 << 28))
    xs, ok3, ok4 = extra_shuffle_and_join(torch, dist, native, world, local, dev, x_rows, max(1, min(args.steps, 5)), 3, peak, peak_src, 48 + 1000 * rank)
    extra += xs
    verified["M3"], verified["M4"] = {"ok": ok3}, {"ok": ok4}
    if not ok3: failures.append("M3")
    if not ok4: failures.append("M4")
    torch.cuda.empty_cache()

    if exchange is not None:
        exchange.close()
    if world > 1:
        dist.barrier()
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": {"workload": WORKLOADS["M2"], "rows_per_gpu": rows, "groups": CARD,
                       "parallelism": f"dp{world}" + ("" if world == 1 else " + murmur3(42) pmod N ownership, in-library NCCL AllToAllv of the columnar partial states (b200q_exchange_shuffle)"),
                       "l2_policy": "input (%.1f GB/GPU) is far larger than the 126 MB L2; no flush needed" % (rows * 32 / 1e9),
                       "plan": "FilterExec fused into AggExec(Partial) -> AggExec(Final), reference protobuf + C ABI"},
            "e2e": e2e, "gpu_launches": headline_stats["launches"], "clocks": clocks,
            "roofline": roofline_of("M2", headline_stats, rows, peak, peak_src), "cpu_baseline": cpu, "verified": verified, "extra": extra,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    if failures:
        sys.stderr.write(f"bench.py: RESULT VERIFICATION FAILED for {failures}\n")
        sys.exit(3)


def dump_m2_outputs(torch, dist, runner, out_dir):
    """The M2 result of the last timed step, the columns k1, k2, sum_v the Final stage returns, merged over the ranks and
    saved as out_dir/<column>.npy.  A hash aggregate emits its groups in no fixed order, so the rows are put in key order
    (k1 * 8 + k2) to make two runs comparable row for row; float64 holds every value exactly (|sum_v| < 2^53)."""
    import numpy as np
    sums = torch.zeros(CARD, dtype=torch.int64, device=runner.dev)
    seen = torch.zeros(CARD, dtype=torch.int64, device=runner.dev)
    for cols in (device_cols(d, torch) for d in runner.last or []):
        gi = cols[0] * K2_CARD + cols[1]
        sums.index_add_(0, gi, cols[2]); seen.index_add_(0, gi, torch.ones_like(gi))
    if runner.world > 1:
        dist.all_reduce(sums); dist.all_reduce(seen)
    if runner.rank != 0:
        return
    gi = torch.nonzero(seen).squeeze(1)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in (("k1", gi // K2_CARD), ("k2", gi % K2_CARD), ("sum_v", sums[gi])):
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy().astype(np.float64))


def mem_available_bytes():
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) * 1024
    except OSError:
        pass
    return 64e9


def bind_to_gpu_numa(torch, local):
    """run this process (and first-touch its pinned buffers) on the CPU socket the GPU hangs off"""
    try:
        p = torch.cuda.get_device_properties(local)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
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


def usable_cores():
    """host threads this container may actually run: min(visible CPUs, cgroup cpu.max quota)"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def thread_candidates():
    """the restatement builds one full group table per task, so its merge grows with the task count and it does NOT scale
    to every core (profiles/r01_cpu_ref_thread_scaling.txt): time a few thread counts and report the best"""
    top = usable_cores()
    return sorted({t for t in (8, 16, 32, top) if 1 <= t <= top} or {top})


def cpu_baseline_m2(cols, sample_rows):
    from oracle import cpu_ref
    f, k1, k2, v = cols
    tried = {}
    for t in thread_candidates():
        cpu_ref.q1_time_only(f[: 1 << 22], k1[: 1 << 22], k2[: 1 << 22], v[: 1 << 22], F_LO, F_HI, t)           # warm-up
        t0 = time.perf_counter(); cpu_ref.q1_time_only(f, k1, k2, v, F_LO, F_HI, t); tried[t] = sample_rows / (time.perf_counter() - t0)
    best = max(tried, key=tried.get)
    return {"value": tried[best], "unit": "rows/s", "cores": best, "kind": "port", "cpu_model": cpu_model(), "usable_cores": usable_cores(),
            "rows_per_s_by_threads": {str(t): r for t, r in tried.items()},
            "sample": f"{sample_rows} rows of the same M2 batch; {best} reference-style tasks (Filter -> Partial agg per task, bucket by key hash, Final per partition), best of {sorted(tried)} threads (oracle/cpu_ref.c)"}


def run_reference(args):
    """The reference arm: the restatement of the reference's own CPU algorithm (oracle/cpu_ref.c) on the host cores, on the
    same M2 workload.  (The Rust reference cannot be built or installed in this image: no cargo/rustc, no network.)"""
    rank = env_int("RANK", 0)
    if rank != 0:
        return
    import numpy as np
    from oracle import cpu_ref
    rows = env_int("B200Q_BENCH_REF_ROWS", 1 << 28)
    rng = np.random.default_rng(46)
    f = rng.integers(0, 1000, rows, dtype=np.int64); k1 = rng.integers(0, K1_CARD, rows, dtype=np.int64)
    k2 = rng.integers(0, K2_CARD, rows, dtype=np.int64); v = rng.integers(-10**6, 10**6, rows, dtype=np.int64)
    probe = min(rows, 1 << 26)
    rates = {}
    for t in thread_candidates():                                     # pick the thread count on a bounded probe, then time every step with it
        cpu_ref.q1_time_only(f[: 1 << 22], k1[: 1 << 22], k2[: 1 << 22], v[: 1 << 22], F_LO, F_HI, t)
        t0 = time.perf_counter(); cpu_ref.q1_time_only(f[:probe], k1[:probe], k2[:probe], v[:probe], F_LO, F_HI, t); rates[t] = probe / (time.perf_counter() - t0)
    threads = max(rates, key=rates.get)
    for _ in range(args.warmup):
        cpu_ref.q1_time_only(f, k1, k2, v, F_LO, F_HI, threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_ref.q1_time_only(f, k1, k2, v, F_LO, F_HI, threads)
    dt = (time.perf_counter() - t0) / args.steps
    val = rows / dt
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "rows/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": WORKLOADS["M2"], "rows_per_step": rows, "groups": CARD},
        "cpu_baseline": {"value": val, "unit": "rows/s", "cores": threads, "kind": "port", "cpu_model": cpu_model(), "usable_cores": usable_cores(),
                         "probe_rows_per_s_by_threads": {str(t): r for t, r in rates.items()},
                         "sample": f"{rows} rows per step, {threads} reference-style tasks (best of {sorted(rates)} on a {probe}-row probe) + final merge (oracle/cpu_ref.c)"},
        "e2e": {"value": val, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the headline's last timed result to DIR/<column>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
