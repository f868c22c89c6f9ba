#!/usr/bin/env python
"""Headline benchmark: aggregations/sec of the Byzantine-robust aggregation hot path.

Workload (BASELINE.json configs[1]):  Krum, N=100 clients, D=11.2M fp32 (f = int(0.24*N) = 24, the
reference default main.py:106), synthetic seeded gradients.

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's own CPU code (or its port) on host cores

A "step" is one complete aggregation `defences.krum(G, N, f)`: pairwise squared distances (tcgen05
Gram kernel) -> [cross-GPU sum of the N x N table when D is sharded] -> distances -> Krum score/argmin ->
index to the host -> view of the winning row.  Multi-GPU runs shard the FIXED D = 11.2M over the ranks
("strong" scaling: one aggregation gets faster), with the single exchange step of the path.

One JSON line on stdout (rank 0).  `value`: inputs resident in HBM.  `e2e`: the same aggregation from
HOST buffers through the C-ABI host entry point (H2D inside the timed region).  `parity`: the timed
result checked against the plain-C float64 oracle in the same run (the run FAILS on a mismatch).
`extra`: the other BASELINE.json configurations (C3 trimmed mean bf16, N=1000 x D=25M Krum / Bulyan /
ALIE on one GPU, or their per-GPU shards under --gpus 8), each with its own roofline and parity.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_CLIENTS, DIM, F_BYZ = 100, 11_200_000, 24
METRIC = "aggregations/sec (Krum, N=100 clients x D=11.2M fp32 params)"
UNIT = "aggregations/s"
RULES = {"Krum", "TrimmedMean", "Bulyan", "NoDefense", "ALIE"}


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"hbm": float(p["hbm_gbs"]), "tf_burst": float(p.get("bf16_tflops", 1590.0)),
                "tf_sustained": float(p.get("bf16_tflops_sustained", 1400.0)),
                "src": "measured (MEASURED_PEAKS.json)"}
    except Exception:
        return {"hbm": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons (B200_PROFILING.md's clocks line, its 200 ms period) sampled while the step
    loop runs.  Round 1 polled every 20 ms; a 2-GPU A/B (profiles/r02_clock_sampler_ab.json) showed that a query landing
    inside a 10-20 ms timed region stalls kernel launches: 0.528 ms/step with the sampler off or at 200 ms, 0.535 or
    0.682 ms at 20 ms - the "sporadic slow run" of the round-1 scaling table.  So: the timed region starts right after
    a sample arrived (the next query is 200 ms away), and when the region is shorter than two periods the same step
    loop keeps running, untimed, until two more samples are in (`run_config`), so the clocks are read under the
    measured load without a query inside the measurement."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index
        self.period_ms = int(os.environ.get("AFL_BENCH_CLOCKS_MS", "200"))

    def start(self):
        if self.period_ms <= 0:
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", str(self.period_ms)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
            t0 = time.time()
            while not self.rows and time.time() - t0 < 3.0:      # first sample before the timed region starts
                time.sleep(0.002)
        except Exception:
            self.proc = None

    def align(self):
        """Return right after the next sample arrived, so that the following period is free of queries."""
        if self.proc is None:
            return
        n0, t0 = len(self.rows), time.time()
        while len(self.rows) == n0 and time.time() - t0 < 1.0:
            time.sleep(0.001)
        self.first = len(self.rows)                              # samples from here on are taken under the step loop

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows[getattr(self, "first", 0):]:
            c = [x.strip() for x in r.split(",")]
            if len(c) < 8:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], c[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def synth_shard(n, c0, c1, device, seed=1234, dtype="f32"):
    """Heterogeneous-client gradients (SURVEY 8d 'Dist B'), generated by fixed 2^20-column blocks so
    that sharded and unsharded runs see the same matrix column for column."""
    import torch
    blk = 1 << 20
    ld = (c1 - c0 + 31) // 32 * 32
    tdt = torch.float32 if dtype == "f32" else torch.bfloat16
    G = torch.empty((n, ld), dtype=tdt, device=device)[:, :c1 - c0]
    gs = torch.Generator(device=device).manual_seed(seed)
    scale = torch.exp(0.25 * torch.randn(n, 1, generator=gs, device=device))
    b = c0 // blk
    while b * blk < c1:
        lo, hi = max(b * blk, c0), min((b + 1) * blk, c1)
        g = torch.Generator(device=device).manual_seed(seed + 1 + b)
        mu = 0.1 * torch.randn(blk, generator=g, device=device)
        off = lo - b * blk
        rows = 250                                            # bound the fp32 temporary at large N
        for r0 in range(0, n, rows):
            r1 = min(n, r0 + rows)
            eps = torch.randn(r1 - r0, blk, generator=g, device=device)
            G[r0:r1, lo - c0:hi - c0] = (mu[None, off:off + hi - lo] + scale[r0:r1] * eps[:, off:off + hi - lo]).to(tdt)
            del eps
        b += 1
    return G


# ------------------------------------------------------------------------------------------------
# CPU legs: the reference's own code when it is present on this host, else its NumPy port
# ------------------------------------------------------------------------------------------------
def load_reference():
    """The UNMODIFIED reference `defences` / `malicious` modules, if a checkout is on this host."""
    import importlib.util
    for base in (os.environ.get("AFL_REFERENCE_DIR"), "/root/reference", os.path.join(ROOT, "baseline", "_ref")):
        if base and os.path.isfile(os.path.join(base, "defences.py")):
            try:
                mods = {}
                for name in ("defences", "malicious"):
                    spec = importlib.util.spec_from_file_location(f"_afl_ref_{name}", os.path.join(base, f"{name}.py"))
                    m = importlib.util.module_from_spec(spec); spec.loader.exec_module(m); mods[name] = m
                return mods, base
            except Exception:
                continue
    return None, None


def cpu_sample_dim(rule, n, d, budget=5.0):
    """D' of the CPU sample: FIXED per (rule, N) so that every CPU figure of one record is taken on the same
    shape (the reference's cost is linear in D at fixed N; ~4 ns per element per pair, ~0.35 us per value
    of a trimmed-mean column)."""
    if rule in ("Krum", "Bulyan"):
        pairs = max(1, n * (n - 1) // 2)
        want = budget / (pairs * 4.0e-9)
        d_s = 1 << max(12, min(20, int(want).bit_length() - 1))
        return int(min(d, d_s))
    if rule == "TrimmedMean":
        return int(min(d, max(256, int(budget / (n * 0.35e-6)))))
    return int(min(d, 1 << 20))


def cpu_inputs(n, d_s, seed):
    import numpy as np
    rng = np.random.default_rng(seed)
    mu = (0.1 * rng.standard_normal(d_s)).astype(np.float32)
    scale = np.exp(0.25 * rng.standard_normal((n, 1))).astype(np.float32)
    return mu[None, :] + scale * rng.standard_normal((n, d_s), dtype=np.float32)      # Dist B, like synth_shard


def cpu_reference_leg(rule, n, d, f, seed=1234, z=1.5, budget=5.0):
    """Times the reference's CPU path on a bounded sample of the workload (full N, reduced D') and scales
    linearly in D; the D-independent selection part is timed at full N and added un-scaled."""
    import numpy as np
    from oracle import ref_numpy as orc
    ref, ref_dir = load_reference()
    kind = "reference" if ref else "port"
    d_s = cpu_sample_dim(rule, n, d, budget)
    G = cpu_inputs(n, d_s, seed)
    tm_cols = int(min(d_s, max(64, int(0.6 * budget / (max(n - 2 * f, 1) * 0.35e-6)))))
    note = ""
    if rule in ("Krum", "Bulyan"):
        t0 = time.perf_counter()
        table = ref["defences"]._krum_create_distances(G) if ref else orc.pairwise_distances_f32(G)
        t_pairs = time.perf_counter() - t0
        theta = n - 2 * f
        if rule == "Krum":
            t0 = time.perf_counter()
            if ref:
                ref["defences"].krum(G, n, f, distances=table, return_index=True)
            else:
                orc.krum_select(table, orc.visit_order(n), n, f)
            t_sel = time.perf_counter() - t0
        else:
            # defences.py:61-68: theta rounds of krum-with-removal; the first `rounds` are timed and the rest is
            # extrapolated with the (n - r)^2 log(n - r) cost of a round (all rounds when that takes < ~20 s)
            rounds = theta if n <= 300 else max(2, min(theta, int(2.0 * budget / (2.2e-7 * n * n))))
            t0 = time.perf_counter()
            if ref:
                sel = []
                for r in range(rounds):
                    idx = ref["defences"].krum(G, n - r, f, table, True)
                    sel.append(idx); table.pop(idx)
                    for u in table:
                        table[u].pop(idx)
            else:
                alive = orc.visit_order(n); sel = []
                for r in range(rounds):
                    idx = orc.krum_select(table, alive, n - r, f); sel.append(idx); alive.remove(idx)
            t_sel = time.perf_counter() - t0
            w = lambda r: (n - r) ** 2 * max(1.0, __import__("math").log2(max(n - r, 2)))
            t_sel *= sum(w(r) for r in range(theta)) / sum(w(r) for r in range(rounds))
            note = f"; selection: {rounds} of {theta} rounds timed, rest extrapolated"
            rows = (sel + [i for i in range(n) if i not in sel])[:theta]
            Gs = np.ascontiguousarray(G[rows][:, :tm_cols])
            t0 = time.perf_counter()
            (ref["defences"].trimmed_mean if ref else orc.trimmed_mean)(Gs, theta, 2 * f)
            t_tm = time.perf_counter() - t0
        total = t_pairs * (d / d_s) + t_sel + (t_tm * (d / tm_cols) if rule == "Bulyan" else 0.0)
        sample = (f"all {n * (n - 1) // 2} pairs at D'={d_s} of D={d} (x{d / d_s:.1f}) + selection at full N{note}" +
                  (f" + stage-2 trimmed mean on {tm_cols} columns" if rule == "Bulyan" else ""))
    elif rule == "TrimmedMean":
        t0 = time.perf_counter()
        (ref["defences"].trimmed_mean if ref else orc.trimmed_mean)(G, n, f)
        total = (time.perf_counter() - t0) * (d / d_s)
        sample = f"{d_s} of {d} columns (x{d / d_s:.1f})"
    elif rule == "ALIE":
        class U:                                              # the duck-typed client of malicious.py:10-27
            def __init__(self, g): self.grads = g; self.original_params = None; self.learning_rate = None
        users = [U(G[i].copy()) for i in range(f)]
        t0 = time.perf_counter()
        if ref:
            ref["malicious"].DriftAttack(z).attack(users)
        else:
            orc.alie_attack([u.grads for u in users], z)
        total = (time.perf_counter() - t0) * (d / d_s)
        sample = f"{f} malicious rows x {d_s} of {d} columns (x{d / d_s:.1f})"
    else:
        t0 = time.perf_counter()
        (ref["defences"].no_defense(G, n, f) if ref else orc.no_defense(G))
        total = (time.perf_counter() - t0) * (d / d_s)
        sample = f"{d_s} of {d} columns (x{d / d_s:.1f})"
    info = {"value": 1.0 / total, "unit": UNIT, "cores": 1, "kind": kind,
            "sample": sample + ("; unmodified reference modules from " + ref_dir if ref else "; NumPy port of the reference (oracle/ref_numpy.py)") +
                      ", single Python thread + NumPy/OpenBLAS as the reference runs",
            "seconds_per_aggregation": total, "host_cpus": os.cpu_count(), "sample_dim": d_s}
    return info


def c_port_leg(rule, n, d, f):
    """Second, stronger CPU figure: plain-C restatement on all host threads (never substituted for the above)."""
    import numpy as np
    try:
        from oracle import c_oracle as co
        d_c = int(min(d, 1 << 20)) if rule in ("Krum", "Bulyan") and n <= 200 else int(min(d, 1 << 17))
        Gc = cpu_inputs(n, d_c, 99)
        t0 = time.perf_counter()
        if rule in ("Krum", "Bulyan"):
            co.pairwise_sqdist(Gc)
        elif rule == "TrimmedMean":
            co.trimmed_mean(Gc, f)
        elif rule == "ALIE":
            co.alie(Gc[:f], 1.5)
        else:
            co.mean(Gc)
        tc = (time.perf_counter() - t0) * (d / d_c)
        return {"value": 1.0 / tc, "unit": UNIT, "cores": co.threads(),
                "sample": f"D'={d_c} of {d}, dominant stage only, float64 accumulation"}
    except Exception as e:  # pragma: no cover
        return {"error": str(e)[:200]}


def run_reference(args, rank):
    if rank != 0:
        return
    t_all = time.perf_counter()
    vals = []
    for s in range(args.warmup + args.steps):
        info = cpu_reference_leg(args.rule, args.n, args.d, args.f, seed=1234 + s, budget=args.ref_budget)
        if s >= args.warmup:
            vals.append(info)
    v = statistics.median(x["value"] for x in vals)
    last = vals[-1]
    line = {"impl": "reference",
            "metric": METRIC if (args.rule, args.n, args.d) == ("Krum", N_CLIENTS, DIM)
            else f"aggregations/sec ({args.rule}, N={args.n} x D={args.d} {args.dtype})",
            "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000.0 / v, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args.rule, args.n, args.d, args.f, args.dtype, args.gpus)},
            "cpu_baseline": {**{k: last[k] for k in ("unit", "cores", "kind", "sample")}, "value": v},
            "cpu_c_port_all_threads": c_port_leg(args.rule, args.n, args.d, args.f),
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.perf_counter() - t_all}
    print(json.dumps(line), flush=True)


def workload_name(rule, n, d, f, dtype, world):
    return f"{rule} N={n} D={d} f={f} {dtype}, D sharded over {world} GPU(s)"


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class Ctx:
    pass


def parity_check(cx, rule, G, n, d, f, out, z=1.5):
    """The timed result against the float64 C oracle (oracle/oracle.c) in the same run.  Full matrix when it
    is small enough for the host (<= 6 GB, single GPU); otherwise the first `cols` columns of the same
    device-resident matrix are pushed through the same kernels and compared, plus a column sample of the
    coordinate-wise outputs at full size."""
    import numpy as np
    import torch
    from oracle import c_oracle as co
    res = {"oracle": "oracle/oracle.c (float64 arbiter, all host threads)"}
    agg, world = cx.agg, cx.world
    es = G.element_size()
    if rule in ("TrimmedMean", "NoDefense", "ALIE"):
        cols = torch.arange(0, G.shape[1], max(1, G.shape[1] // 1536), device=G.device)[:1536]
        Gs = (G[n - f:] if rule == "ALIE" else G)[:, cols].float().cpu().numpy()
        got = out[cols].float().cpu().numpy().astype(np.float64)
        if rule == "TrimmedMean":
            ref = co.trimmed_mean(Gs, f)
        elif rule == "ALIE":
            ref = co.alie(Gs, z)[0]
        else:
            ref = co.mean(Gs)
        scale = float(np.abs(Gs).mean()) + 1e-30
        err = np.abs(got - ref) / (np.abs(ref) + 1e-6 * scale / 1e-5)
        res.update({"checked": f"{len(cols)} columns of rank 0's shard vs the oracle", "max_rel_err": float(err.max()),
                    "tolerance": 1e-5, "match": bool(err.max() <= 1e-5)})
        return res
    full = world == 1 and n * d * es <= 6e9
    if full:
        Gc, gpu_idx_or_sel = G, out
        res["checked"] = f"selected indices on the full {n} x {d} matrix"
    else:
        cols = min(G.shape[1], max(32768, (1 << 22) // n // 32 * 32))
        Gc = G[:, :cols]
        res["checked"] = (f"selected indices on the first {cols} columns of every rank's shard of the timed matrix "
                          f"(the full {n} x {d} matrix does not fit the host oracle)")
        if rule == "Krum":
            gpu_idx_or_sel = agg.krum(Gc, n, f, return_index=True)
        else:
            gpu_idx_or_sel = agg.bulyan(Gc, n, f, return_selection=True)
    host = Gc.float().cpu().numpy()
    if world > 1:
        import torch.distributed as dist
        parts = [None] * world
        dist.all_gather_object(parts, host)
        host = np.concatenate(parts, axis=1)
    if cx.rank != 0:
        return None
    t64 = np.sqrt(co.pairwise_sqdist(np.ascontiguousarray(host)))
    if rule == "Krum":
        want, margin = co.krum_select(t64, n, f, with_margin=True)
        got = int(gpu_idx_or_sel)
        res.update({"index": got, "oracle_index": want, "margin": margin,
                    "match": bool(got == want or 0.0 < margin <= 1e-5)})
    else:
        o, sel = gpu_idx_or_sel
        sel = sel.cpu().tolist()
        want, margins = co.bulyan_select(t64, n, f, with_margins=True)
        first_close = next((i for i, m in enumerate(margins) if 0.0 < m <= 1e-5), len(margins))
        ok_sel = sel[:first_close] == want[:first_close]
        cs = np.arange(0, host.shape[1], max(1, host.shape[1] // 1024))[:1024] if cx.world == 1 else np.arange(min(1024, Gc.shape[1]))
        ref = co.trimmed_mean(np.ascontiguousarray(host[:, cs]), 2 * f, rows=sel)
        got = o[torch.from_numpy(cs).to(o.device)].cpu().numpy().astype(np.float64)
        scale = float(np.abs(host[:, cs]).mean())
        err = float((np.abs(got - ref) / (np.abs(ref) + 0.1 * scale)).max())
        res.update({"rounds": len(sel), "rounds_required_exact": first_close, "min_positive_margin": min([m for m in margins if m > 0] or [0.0]),
                    "selection_match": bool(ok_sel), "stage2_max_rel_err": err, "match": bool(ok_sel and err <= 1e-5)})
    return res


DUMP_BYTES = 64_000_000


def last_step_outputs(cx, rule, G, out, d):
    """What a caller of the timed path receives from its last step, on every rank: the per-column outputs gathered
    to full length D (float32 device tensors), and the selected indices."""
    import torch
    if rule == "Krum":
        cols, picks = {"aggregate": G[out]}, {"krum_index": torch.tensor([out])}       # defences.krum returns the row G[idx]
    elif rule == "Bulyan":
        cols, picks = {"aggregate": out[0]}, {"bulyan_selection": out[1]}
    else:
        cols, picks = {"crafted" if rule == "ALIE" else "aggregate": out}, {}
    cols = {k: cx.agg.gather_output(v.float(), d) for k, v in cols.items()}
    return cols, picks


def write_outputs(dirname, cols, picks, budget=DUMP_BYTES):
    """Writes DIR/<name>.npy: the per-column outputs `cols` (equal-length vectors) as float32, the indices `picks` as
    float64, `budget` bytes in all.  When the vectors do not fit, each is cut to the same seeded sample of columns (the
    same columns for the same D in every run), and the sampled column numbers go to DIR/columns.npy."""
    import numpy as np
    import torch
    os.makedirs(dirname, exist_ok=True)
    picks = {name: torch.as_tensor(v).cpu().numpy().astype(np.float64) for name, v in picks.items()}
    room = budget - sum(v.nbytes for v in picks.values()) - 128 * (len(cols) + len(picks) + 1)   # 128: .npy header
    d = next(iter(cols.values())).numel() if cols else 0
    if 4 * d * len(cols) > room:
        pos = np.unique(np.random.default_rng(20261017).integers(0, d, room // (4 * len(cols) + 8)))
        picks["columns"] = pos.astype(np.float64)
        cols = {name: v[torch.from_numpy(pos).to(v.device)] for name, v in cols.items()}
    for name, v in cols.items():
        np.save(os.path.join(dirname, f"{name}.npy"), v.float().cpu().numpy())
    for name, v in picks.items():
        np.save(os.path.join(dirname, f"{name}.npy"), v)


def run_config(cx, rule, n, d, f, dtype, steps, warmup, want_e2e=False, e2e_steps=3, z=1.5, check=True, dump_dir=None):
    """One benchmark configuration on the current process group: returns the fields of a bench record.  `dump_dir`:
    rank 0 writes the outputs of the last timed step there (`write_outputs`)."""
    import torch
    import torch.distributed as dist
    from attacking_federate_learning_b200 import _native as nat, defences as D
    from attacking_federate_learning_b200.sharded import shard_bounds
    world, rank, device, agg = cx.world, cx.rank, cx.device, cx.agg
    c0, c1 = shard_bounds(d, world, rank)
    G = synth_shard(n, c0, c1, device, dtype=dtype)
    es = G.element_size()
    d_local = c1 - c0

    def step():
        if rule == "Krum":
            return agg.krum(G, n, f, return_index=True)       # index -> host; the row itself is a view G[idx]
        if rule == "Bulyan":
            return agg.bulyan(G, n, f, return_selection=True)
        if rule == "TrimmedMean":
            return agg.trimmed_mean(G, n, f)
        if rule == "ALIE":
            return agg.alie(G, f, z, write_rows=True, source_rows=G[n - f:])   # reads f rows, writes the crafted vector into rows 0..f-1
        return agg.no_defense(G)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(warmup, 3)):
        out = step()
    barrier()
    nat.profile_enable(2)             # CUDA events around the dominant kernel only (one pair per step), inside the timed region
    launches0 = nat.launch_count()
    sampler = ClockSampler(cx.local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if rank == 0:
        sampler.align()               # the next nvidia-smi query is one period (200 ms) away
    barrier()
    e0.record()
    for _ in range(steps):
        out = step()
    e1.record()
    barrier()
    ms_total = torch.tensor([e0.elapsed_time(e1)], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms_total, op=dist.ReduceOp.MAX)
    ms_step = float(ms_total.item()) / steps
    launches = nat.launch_count() - launches0
    nat.profile_enable(False)
    if dump_dir:
        cols, picks = last_step_outputs(cx, rule, G, out, d)
        if rank == 0:
            write_outputs(dump_dir, cols, picks)
        del cols, picks
    # clocks under load: keep the same step loop running (untimed, same count on every rank) until two sampler periods
    # have passed since the timed region began
    need_ms = 2.2 * sampler.period_ms - float(ms_total.item())
    if need_ms > 0 and sampler.period_ms > 0:
        for _ in range(min(5000, int(need_ms / max(ms_step, 1e-3)) + 1)):
            step()
        barrier()
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["sampling"] = f"nvidia-smi -lms {sampler.period_ms}, samples from the start of the timed region to the end of the same step loop"
    dom = {}
    for kname in ("gram_bf16x2", "gram_pair", "gram_tcgen05", "sqdist_simt", "trimmed_mean", "mean", "alie"):
        k_ms, k_cnt = nat.profile_read(kname)
        if k_cnt:
            dom[kname] = (k_ms / k_cnt, k_cnt)
    # Breakdown of the small kernels: a SECOND, short loop with every in-library bracket on (a few host microseconds
    # per kernel that the timed loop above does not pay).
    nat.profile_enable(1)
    for _ in range(max(3, min(steps, 10))):
        step()
    barrier()
    nat.profile_enable(False)
    # per-kernel device times of the timed region (in-library event brackets on the launching stream)
    prof = {}
    for kname in ("gram_bf16x2", "gram_pair", "gram_tcgen05", "sqdist_simt", "trimmed_mean", "mean", "alie", "bulyan_rounds",
                  "row_sort", "krum_tail", "xgpu_sum"):
        try:
            k_ms, k_cnt = nat.profile_read(kname)
        except Exception:
            continue
        if k_cnt:
            prof[kname] = (k_ms / k_cnt, k_cnt)
    prof.update(dom)                  # the dominant kernel's figure comes from the timed region itself
    order = {"Krum": ("gram_bf16x2", "gram_pair", "gram_tcgen05", "sqdist_simt"), "Bulyan": ("gram_bf16x2", "gram_pair", "gram_tcgen05", "sqdist_simt"),
             "TrimmedMean": ("trimmed_mean",), "NoDefense": ("mean",), "ALIE": ("alie",)}[rule]
    kname = next((k for k in order if k in prof), order[0])
    kt = torch.tensor([prof.get(kname, (0.0, 0))[0]], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(kt, op=dist.ReduceOp.MAX)
    k_avg_ms = float(kt.item())
    k_cnt = prof.get(kname, (0.0, 0))[1]

    rec = {"ms_per_step": ms_step, "value": 1000.0 / ms_step, "launches": int(launches), "clocks": clocks}
    peaks = load_peaks()
    theta = n - 2 * f
    if rule in ("Krum", "Bulyan"):
        algo_bytes = n * d_local * es                              # SURVEY 8(d): the Gram reads the matrix once
    elif rule == "ALIE":
        algo_bytes = f * d_local * es + f * d_local * 4 + d_local * 4   # read f rows, write f crafted rows + the vector
    else:
        algo_bytes = n * d_local * es + d_local * 4
    achieved = algo_bytes / (k_avg_ms * 1e-3) / 1e9 if k_avg_ms > 0 else None
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            traffic = json.load(fh).get(f"{rule}:{n}x{d}:{dtype}:{world}")
    except Exception:
        pass
    rec["roofline"] = {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peaks["hbm"], "unit": "GB/s",
                       "frac": (achieved / peaks["hbm"]) if achieved else None, "traffic": traffic,
                       "peak_source": peaks["src"] + " hbm_gbs", "algorithmic_bytes_per_launch": algo_bytes,
                       "kernel_ms_avg": k_avg_ms, "kernel_launches_timed": k_cnt,
                       "kernel_share_of_step": k_avg_ms / ms_step if ms_step else None}
    if rule in ("Krum", "Bulyan") and k_avg_ms > 0:
        flops = 2.0 * n * n * d_local
        tf = flops / (k_avg_ms * 1e-3) / 1e12
        rec["roofline_tensor"] = {"bound": "tensor", "kernel": kname, "achieved": tf, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                                  "frac": tf / peaks["tf_sustained"], "flops_per_launch": flops,
                                  "note": "algorithmic 2*N^2*D_local fp32-equivalent flops (SURVEY 8d); the kernel issues bf16 "
                                          "tensor-core products for three split terms on the lower-triangular tile pairs only",
                                  "peak_source": peaks["src"] + " bf16_tflops_sustained"}
        rec["bound_by"] = "hbm" if rec["roofline"]["frac"] >= rec["roofline_tensor"]["frac"] else "tensor"
    rec["breakdown_us"] = {k: round(v[0] * 1e3, 2) for k, v in prof.items()}
    rec["breakdown_us"]["step_total"] = round(ms_step * 1e3, 2)
    if rule == "Bulyan":
        rec["algorithmic_bytes_per_step"] = n * d_local * es + theta * d_local * es + d_local * 4

    # ---------------- parity of the timed result, same run ----------------
    if check:
        try:
            par = parity_check(cx, rule, G, n, d, f, out, z)
        except Exception as ex:  # pragma: no cover
            par = {"match": False, "error": repr(ex)[:300]} if rank == 0 else None
        rec["parity"] = par

    # ---------------- e2e: host buffers through the reference-facing call ----------------
    if want_e2e:
        e2e = None
        try:
            if e2e_steps <= 0:
                raise RuntimeError('skipped (--e2e-steps 0)')
            host = torch.empty((n, d_local), dtype=torch.float32).pin_memory()
            host.copy_(G.float())
            h2d = n * d * 4
            if world == 1 and dtype == "f32" and rule != "ALIE":
                call = {"Krum": D.krum, "Bulyan": D.bulyan, "TrimmedMean": D.trimmed_mean, "NoDefense": D.no_defense}[rule]

                def timed(Gh):
                    call(Gh, n, f)                                 # warm-up (allocates the staging buffers once)
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    for _ in range(e2e_steps):
                        call(Gh, n, f)
                    torch.cuda.synchronize()
                    return (time.perf_counter() - t0) / e2e_steps
                dt = timed(host.numpy())
                d2h = 4 if rule == "Krum" else d * 4
                e2e = {"value": 1.0 / dt, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                       "ms_per_step": dt * 1e3, "steps": e2e_steps,
                       "path": "afl_defend_host (C ABI, pinned host matrix, H2D slabs overlapped with kernels)"}
                try:                                               # what server.py:35's np.empty buffer gives: pageable memory
                    import numpy as np
                    pageable = np.empty((n, d_local), np.float32); pageable[:] = host.numpy()
                    dtp = timed(pageable)
                    e2e["pageable_host"] = {"value": 1.0 / dtp, "ms_per_step": dtp * 1e3,
                                            "note": "same call on an ordinary np.empty matrix (as server.py:35 allocates it)"}
                    del pageable
                except Exception as ex:  # pragma: no cover
                    e2e["pageable_host"] = {"error": str(ex)[:200]}
            else:
                stage = torch.empty_like(G)

                def e2e_step():
                    stage.copy_(host if dtype == "f32" else host.bfloat16(), non_blocking=True)
                    if rule == "Krum":
                        return agg.krum(stage, n, f, return_index=True)
                    o = {"Bulyan": agg.bulyan, "TrimmedMean": agg.trimmed_mean, "NoDefense": lambda a, b, c: agg.no_defense(a),
                         "ALIE": lambda a, b, c: agg.alie(a, c, z, write_rows=True, source_rows=a[n - c:])}[rule](stage, n, f)
                    return o.cpu()
                e2e_step(); barrier()
                t0 = time.perf_counter()
                for _ in range(e2e_steps):
                    e2e_step()
                barrier()
                tt = torch.tensor([(time.perf_counter() - t0) / e2e_steps], device=device, dtype=torch.float64)
                if world > 1:
                    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                dt = float(tt.item())
                e2e = {"value": 1.0 / dt, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4 * world if rule == "Krum" else d * 4,
                       "ms_per_step": dt * 1e3, "steps": e2e_steps, "path": "per-rank pinned shard -> device copy + device path"}
            del host
        except Exception as ex:  # pragma: no cover
            e2e = {"value": None, "unit": UNIT, "error": str(ex)[:300]}
        rec["e2e"] = e2e
    del G
    torch.cuda.empty_cache()
    return rec


def extra_configs(world, free_gb):
    """The other BASELINE.json configurations (SURVEY 8: C3, C4, C5).  N=1000 x D=25M fp32 is 100 GB and fits one
    B200; under --gpus 8 the same configurations run as their per-GPU shards."""
    ex = [("TrimmedMean", 1000, 10_000_000, 240, "bf16", "C3"),
          ("Bulyan", 500, 25_000_000, 100, "f32", "C4"),
          ("Krum", 1000, 25_000_000, 240, "f32", "C5-krum"),
          ("Bulyan", 1000, 25_000_000, 240, "f32", "C5-bulyan"),
          ("ALIE", 1000, 25_000_000, 240, "f32", "C5-alie")]
    out = []
    for rule, n, d, f, dt, tag in ex:
        gb = n * d * (4 if dt == "f32" else 2) / world / 1e9
        while gb > free_gb - 12:                                  # largest D that fits, stated in the record
            d = d // 2
            gb /= 2
        out.append((rule, n, d, f, dt, tag))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rule", default="Krum", choices=sorted(RULES))
    ap.add_argument("--n", "--clients", dest="n", type=int, default=N_CLIENTS)      # --clients/--dim/--byzantine: the spelling
    ap.add_argument("--d", "--dim", dest="d", type=int, default=DIM)                 # that survives torchrun's own parser
    ap.add_argument("--f", "--byzantine", dest="f", type=int, default=None)
    ap.add_argument("--dtype", default="f32", choices=["f32", "bf16"])
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--ref-budget", type=float, default=5.0,
                    help="seconds of CPU work per reference step that size the FIXED sample D' (same in every CPU leg)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--extras", default="auto", choices=["auto", "on", "off"],
                    help="append the C3/C4/C5 configurations (auto: only for the default headline workload)")
    ap.add_argument("--extra-steps", type=int, default=3)
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (at most 64 MB; inputs are seeded, so "
                         "two builds run with the same arguments can be compared output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps: at least one timed step")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed; the reference arm times a reduced CPU sample")
    if args.f is None:
        args.f = int(0.24 * args.n)
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    from attacking_federate_learning_b200 import _native as nat
    from attacking_federate_learning_b200.sharded import ShardedAggregator, shard_bounds

    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    nat.lib()
    cx = Ctx()
    cx.world, cx.rank, cx.local_rank, cx.device = world, rank, local_rank, device
    cx.agg = ShardedAggregator()
    n, d, f, rule = args.n, args.d, args.f, args.rule
    headline = (rule, n, d, args.dtype) == ("Krum", N_CLIENTS, DIM, "f32")

    rec = run_config(cx, rule, n, d, f, args.dtype, args.steps, args.warmup, want_e2e=True, e2e_steps=args.e2e_steps,
                     check=not args.no_parity, dump_dir=args.dump_outputs)
    extras = []
    if args.extras == "on" or (args.extras == "auto" and headline):
        free_gb = torch.cuda.mem_get_info(device)[0] / 1e9
        for (xr, xn, xd, xf, xdt, tag) in extra_configs(world, free_gb):
            t0 = time.perf_counter()
            try:
                xrec = run_config(cx, xr, xn, xd, xf, xdt, args.extra_steps, 3, want_e2e=False, check=not args.no_parity)
                item = {"tag": tag, "metric": f"aggregations/sec ({xr}, N={xn} x D={xd} {xdt})", "unit": UNIT,
                        "workload": workload_name(xr, xn, xd, xf, xdt, world), "value": xrec["value"], "ms_per_step": xrec["ms_per_step"],
                        "steps": args.extra_steps, "roofline": xrec["roofline"], "breakdown_us": xrec["breakdown_us"],
                        "parity": xrec.get("parity"), "gpu_launches": xrec["launches"], "clocks": xrec["clocks"]}
                for k in ("roofline_tensor", "bound_by", "algorithmic_bytes_per_step"):
                    if k in xrec:
                        item[k] = xrec[k]
                if rank == 0 and world == 1 and not args.no_cpu_baseline:
                    try:
                        item["cpu_baseline"] = cpu_reference_leg(xr, xn, xd, xf)
                        item["speedup_vs_cpu_reference"] = item["value"] / item["cpu_baseline"]["value"]
                    except Exception as ex:  # pragma: no cover
                        item["cpu_baseline"] = {"error": str(ex)[:200]}
                item["wall_s"] = round(time.perf_counter() - t0, 1)
            except Exception as ex:  # pragma: no cover
                item = {"tag": tag, "error": repr(ex)[:400]}
                torch.cuda.empty_cache()
            extras.append(item)

    if rank != 0:
        if world > 1:
            dist.barrier(); dist.destroy_process_group()
        return

    c0, c1 = shard_bounds(d, world, 0)
    d_local = c1 - c0
    es = 4 if args.dtype == "f32" else 2
    line = {
        "metric": METRIC if headline else f"aggregations/sec ({rule}, N={n} x D={d} {args.dtype})",
        "value": rec["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": rec["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": args.dtype, "data": "synthetic",
        "config": {"workload": workload_name(rule, n, d, f, args.dtype, world),      # identical string in the reference arm
                   "columns_on_rank0": d_local,
                   "l2": f"input shard {n * d_local * es / 1e6:.0f} MB >> 126 MB L2, re-streamed from HBM every step (no flush needed)",
                   "parallelism": (f"D-shard x{world}, one exchange of the {n}x{n} float64 table ({cx.agg.exchange_name()})"
                                   if world > 1 else "single GPU")},
        "roofline": rec["roofline"], "e2e": rec.get("e2e"), "gpu_launches": rec["launches"], "clocks": rec["clocks"],
        "breakdown_us": rec["breakdown_us"], "parity": rec.get("parity"),
    }
    for k in ("roofline_tensor", "bound_by"):
        if k in rec:
            line[k] = rec[k]
    if not args.no_cpu_baseline and world == 1:
        try:
            line["cpu_baseline"] = cpu_reference_leg(rule, n, d, f)
            line["cpu_baseline"]["c_port_all_threads"] = c_port_leg(rule, n, d, f)
        except Exception as ex:  # pragma: no cover
            line["cpu_baseline"] = {"error": str(ex)[:300]}
    if extras:
        line["extra"] = extras
    print(json.dumps(line), flush=True)
    bad = [p for p in [line.get("parity")] + [x.get("parity") for x in extras] if p and not p.get("match", False)]
    if world > 1:
        dist.barrier(); dist.destroy_process_group()
    if bad:
        print("PARITY FAILURE: " + json.dumps(bad), file=sys.stderr, flush=True)
        sys.exit(3)


if __name__ == "__main__":
    main()
