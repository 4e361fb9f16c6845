#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native Groth16 hot path.

Metric (BASELINE.json): G1 MSM throughput in Mpairs/s on BN254, 2^20 random scalar/point pairs per
GPU (configs[1]); one "step" = one d_msm over one resident batch.  N > 1: every rank owns its own
2^20 pairs (weak scaling), the only exchange is d_msm's all-gather of the N XYZZ partials + point sum.

  value  : pairs processed by all ranks / device time of the step (inputs resident in HBM)
  e2e    : same metric through the reference-facing call with HOST buffers
           (pinned host -> H2D of bases+scalars, MSM, D2H of the affine result) inside the timed region
  roofline: msm_accumulate_g1 (dominant kernel): 96 B/pair algorithmic bytes / its CUDA-event duration
  cpu_baseline: oracle/bn254_ref.cpp (arkworks-equivalent CPU restatement, "port") on the host cores

`--impl reference` times that CPU restatement alone (the reference itself is Rust and cannot be built
in this image: no cargo/rustc, dependencies un-vendored -- see DESIGN.md).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LOG_N = int(os.environ.get("B200ZK_BENCH_LOG_N", "20"))
METRIC = "G1 MSM throughput (BN254 Pippenger, 2^%d pairs per GPU)" % LOG_N
WORKLOAD = "BN254 G1 Pippenger MSM 2^%d random scalar/point pairs per GPU" % LOG_N     # same string in both arms
UNIT = "Mpairs/s"
ALG_BYTES_PER_PAIR = 96.0       # 32 B scalar + 64 B affine point, each read once (SURVEY 8d)


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[1]) for r in self.rows if len(r) > 2 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = set()
        for r in self.rows:
            for k, nm in enumerate(names):
                if len(r) > 5 + k and r[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dump_outputs(out_dir, point, infinity):
    """What one MSM step hands its caller: the affine G1 result (b200zk.h layout, x then y, each four little-endian u64
    Montgomery limbs) as sixteen 32-bit words in float64, which holds them exactly, and the infinity flag."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    words = np.ascontiguousarray(point, dtype="<u8").view("<u4").reshape(2, 8)
    np.save(os.path.join(out_dir, "msm_g1_affine_words.npy"), words.astype(np.float64))
    np.save(os.path.join(out_dir, "msm_g1_infinity.npy"), np.array([float(infinity)]))


def run_reference(args):
    """CPU arm: the arkworks-equivalent restatement on the host cores, rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import numpy as np  # noqa: F401
    from oracle import cref
    cref.build()
    n = 1 << LOG_N
    cores = os.cpu_count() or cref.num_threads()      # torchrun exports OMP_NUM_THREADS=1: ask for all host cores explicitly
    bases = cref.g1_generate(0xB2000002, n)
    scalars = cref.fr_generate(0xB2000002, n)
    for _ in range(max(args.warmup, 1) if args.warmup else 0):
        cref.msm_g1(bases, scalars, cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = cref.msm_g1(bases, scalars, cores)
    dt = (time.perf_counter() - t0) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *res)
    val = n / dt / 1e6
    sample = "full 2^%d-pair G1 MSM per step, %d OpenMP threads (windows in parallel, as arkworks+rayon)" % (LOG_N, cores)
    emit({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32x8 Montgomery (256-bit modular integers)", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "note": "CPU restatement of arkworks VariableBaseMSM (oracle/bn254_ref.cpp); the Rust reference "
                           "cannot be built in this image"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


def measure_ntt(net, hbm_peak, pipe_peak):
    """BASELINE config 3: Fr radix-2 NTT, 2^22 elements resident in HBM (forward, natural order in and out)."""
    import torch
    log_n = int(os.environ.get("B200ZK_BENCH_NTT_LOG_N", "22"))
    n = 1 << log_n
    x = net.generate_fr(3, n)
    y = torch.empty_like(x)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=x.device)
    for _ in range(3):
        net.ntt_dev(x, y)
    evs = []
    for _ in range(10):
        flush.fill_(1)
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        net.ntt_dev(x, y)
        a1.record()
        evs.append((a0, a1))
    torch.cuda.synchronize()
    ts = sorted(a.elapsed_time(b) for a, b in evs)
    ms = sum(ts) / len(ts)
    back = torch.empty_like(x)
    net.ntt_dev(y, back, inverse=True)
    # products per element, as csrc/ntt.cu runs it: passes of <= 8 butterfly levels whose first level has unit twiddles (and, in a
    # pass with an even number of levels, half of the second level too: the first radix-4 unit multiplies by 1 and i only), and
    # at every pass boundary the inter-pass twiddle: 1 product where a single-level table exists (first boundary up to 2^24,
    # middle passes with <= 2^16 distinct exponents), 2 through the two-level power table otherwise
    passes = -(-log_n // 8)
    log_r = [log_n // passes + (1 if i < log_n % passes else 0) for i in range(passes)]
    per_elem, log_l = (log_n - passes) / 2.0 - 0.25 * sum(1 for r in log_r if r % 2 == 0), 0
    bigtab = int(os.environ.get("B200ZK_NTT_BIGTAB", "24"))
    for i in range(passes - 1):
        single = (i == 0 and log_n <= bigtab) or (i > 0 and log_n - log_l <= 16)
        per_elem += 1.0 if single else 2.0
        log_l += log_r[i]
    products = n * per_elem
    return {"metric": "Fr NTT 2^%d (BN254 scalar field)" % log_n, "ms": ms, "ms_min": ts[0], "gelem_s": n / ms / 1e6,
            "roofline": {"bound": "hbm", "achieved": 64.0 * n / ms / 1e6, "peak": hbm_peak, "unit": "GB/s",
                         "frac": 64.0 * n / ms / 1e6 / hbm_peak, "algorithmic_bytes_per_element": 64,
                         "pipe": {"achieved": products / ms / 1e6, "peak": pipe_peak, "unit": "G modular products/s",
                                  "frac": products / ms / 1e6 / pipe_peak,
                                  "products_per_element": per_elem,
                                  "how": "n x ((log n - passes) / 2 butterfly products - 1/4 per pass with an even number of levels + 1 "
                                         "(single-level table) or 2 (two-level) twiddle products per pass boundary)"}},
            "round_trip_exact": bool((back == x).all()),
            "timing": "CUDA events per transform, L2 flushed between transforms, 10 runs after 3 warm-ups"}


def measure_prove(net, args, with_cpu):
    """Secondary metric of BASELINE.json: Groth16 prove ms, BN254, 2^20 constraints (m = n_vars = 2^20, dummy CRS
    built like groth16/examples/local_groth_bench.rs:21-52; witness and QAP evaluations resident in HBM)."""
    import numpy as np
    import torch
    from distributed_groth16_b200.groth16 import ProvingKey, prove
    log_m = int(os.environ.get("B200ZK_BENCH_PROVE_LOG_M", "20"))
    m = 1 << log_m
    n_vars, n_inputs = m, 2
    aq, b1 = net.generate_g1(101, n_vars), net.generate_g1(102, n_vars)
    b2 = net.generate_g2(103, n_vars)
    lq, hq = net.generate_g1(104, n_vars - n_inputs), net.generate_g1(105, m)
    vk = np.concatenate([net.generate_g1(106, 3).cpu().numpy().view(np.uint64).reshape(-1),
                         net.generate_g2(107, 2).cpu().numpy().view(np.uint64).reshape(-1)])
    z = net.generate_fr(108, n_vars)
    from distributed_groth16_b200._constants import FR_ONE_MONT
    z[0] = torch.from_numpy(np.array(FR_ONE_MONT, dtype=np.uint64).view(np.int64)).to(z.device)
    a, b, c = (net.generate_fr(sd, m) for sd in (109, 110, 111))
    pk = ProvingKey.from_device(net, aq, b1, b2, lq, hq, n_inputs, vk)
    times = []
    proof = None
    for _ in range(2 + 5):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        proof = prove.create_proof_dev(pk, z, a, b, c)         # returns after the 128 proof bytes are on the host
        times.append((time.perf_counter() - t0) * 1e3)
    times = sorted(times[2:])
    res = {"metric": "Groth16 prove (BN254, 2^%d constraints, r = s = 0)" % log_m, "ms": times[len(times) // 2],
           "ms_min": times[0], "unit": "ms", "higher_is_better": False, "n_vars": n_vars, "domain": m,
           "msm_sizes": {"g1": [n_vars - 1, n_vars - n_inputs, m], "g2": [n_vars - 1]},
           "pk_table_gb": pk.table_bytes / 2**30,
           "timing": "host wall clock around b200zk_groth16_prove_dev (includes the D2H of the proof), 5 runs after 2 warm-ups"}
    # SURVEY 8d: 6 x 64 m (3 iNTT + 3 coset NTT) + 4 x 32 m (pointwise) + 96 (n_vars - 1) [A] + 160 (n_vars - 1) [B]
    # + 96 n_aux [L] + 96 m [H-query]; the r-dependent b_g1 MSM does not run with r = 0
    alg = 6 * 64 * m + 4 * 32 * m + 96 * (n_vars - 1) + 160 * (n_vars - 1) + 96 * (n_vars - n_inputs) + 96 * m
    peak, peak_src = _peaks()
    res["roofline"] = {"bound": "hbm", "achieved": alg / (res["ms"] * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                       "frac": alg / (res["ms"] * 1e-3) / 1e9 / peak, "algorithmic_bytes": alg, "peak_source": peak_src,
                       "note": "whole proof (h pipeline + 4 MSMs + assembly); multiplier-pipe bound like its kernels"}
    if with_cpu:
        from oracle import cref
        ncores = os.cpu_count() or 1
        h2 = lambda t: t.cpu().numpy().view(np.uint64)
        t0 = time.perf_counter()
        hh = cref.h_circom(h2(a), h2(b), h2(c), ncores)
        exp = cref.groth16_prove(h2(aq), h2(b1), h2(b2), h2(lq), h2(hq), vk, n_inputs, h2(z), hh, np.zeros(4, np.uint64),
                                 np.zeros(4, np.uint64), nthreads=ncores)
        res["cpu_baseline"] = {"ms": (time.perf_counter() - t0) * 1e3, "cores": ncores, "kind": "port",
                               "sample": "one full prove (h + 4 MSMs) with the CPU restatement"}
        res["bit_exact_vs_cpu"] = bool(exp == proof)
    pk.free()
    return res


def measure_prove_sha256(net, with_cpu):
    """BASELINE config 4: the reference's own workload (groth16/examples/sha256.rs:158-169 "Arkworks Proof" timer;
    zk-cli/README.md:42): sha256 circuit, m = 2^15, r = s = 0.  The key is made by the product's GPU setup from a toxic waste;
    with the CPU baseline enabled the toxic waste and generators are the ones the reference's seed [42; 32] yields
    (oracle/ark_rand.py), so the GPU proof must be the reference's committed proof.bin byte for byte."""
    import numpy as np
    from distributed_groth16_b200.groth16 import circom, setup
    gold_dir = os.path.join(ROOT, "tests", "golden")
    d = np.load(os.path.join(gold_dir, "sha256_circuit.npz"))
    n_wires, n_pub, n_cons = (int(x) for x in d["dims"])
    n_inputs = n_pub + 1
    m = 1
    while m < n_cons + n_inputs:
        m <<= 1
    coo = lambda k: (d[k + "_rows"], d[k + "_cols"], d[k + "_vals"])
    gens = {}
    toxic = (0x1234567, 0x2345678, 0x3456789, 0x456789A, 0x56789AB)
    if with_cpu:
        from oracle import ark_rand as ar, layout, reference_instance
        tw = ar.groth16_toxic_waste(reference_instance.SEED, m)
        toxic = (tw["t"], tw["alpha"], tw["beta"], tw["gamma"], tw["delta"])
        gens = dict(g1_generator=layout.g1_to_arr([tw["g1"]])[0], g2_generator=layout.g2_to_arr([tw["g2"]])[0])
    t0 = time.perf_counter()
    pk, vk, mats = setup.circuit_specific_setup(net, n_wires, n_inputs, n_cons, coo("a"), coo("b"), coo("c"), toxic, **gens)
    setup_ms = (time.perf_counter() - t0) * 1e3
    z = net.fr_convert(net.to_device(d["witness"]), to_mont=True)
    zero = np.zeros(4, dtype=np.uint64)
    ts, proof = [], None
    for _ in range(2 + 7):
        net.sync(0)
        t0 = time.perf_counter()
        proof = circom.prove_from_matrices(pk, mats, z, zero, zero)
        ts.append((time.perf_counter() - t0) * 1e3)
    ts = sorted(ts[2:])
    pk.free()
    res = {"metric": "Groth16 prove, reference sha256 circuit (BN254, %d constraints, m = 2^%d, r = s = 0)" % (n_cons, m.bit_length() - 1),
           "ms": ts[len(ts) // 2], "ms_min": ts[0], "unit": "ms", "higher_is_better": False, "gpu_setup_ms": setup_ms,
           "msm_sizes": {"g1": [n_wires - 1, n_wires - n_inputs, m], "g2": [n_wires - 1]},
           "timing": "host wall clock around qap() + b200zk_groth16_prove_dev (witness resident, proof bytes on the host), 7 runs after 2"}
    if with_cpu:
        from oracle import cref, reference_instance
        gold = open(os.path.join(gold_dir, "sha256_proof.bin"), "rb").read()
        res["bytes_equal_reference_proof_bin"] = bool(proof == gold)
        cpk, cvk, cz, ca, cb, cc, _ = reference_instance.sha256_instance(cref, gold_dir)
        vk_pts = np.concatenate([cvk["alpha_g1"], cvk["beta_g1"], cvk["delta_g1"], cvk["beta_g2"], cvk["delta_g2"]])
        ncores = os.cpu_count() or 1
        t0 = time.perf_counter()
        got = cref.groth16_prove(cpk["a_query"], cpk["b_g1_query"], cpk["b_g2_query"], cpk["l_query"], cpk["h_query"], vk_pts, n_inputs,
                                 cz, cref.h_circom(ca, cb, cc, ncores), zero, zero, mirror_bg1=False, nthreads=ncores)
        res["cpu_baseline"] = {"ms": (time.perf_counter() - t0) * 1e3, "cores": ncores, "kind": "port",
                               "sample": "one full prove (h + 4 MSMs) with the CPU restatement; bytes == proof.bin: %s" % (got == gold)}
    return res


def measure_msm_sizes(net, dev, log_sizes):
    """north_star's size sweep on one GPU (the reference's own loop: dist-primitives/examples/dmsm_bench.rs:45-50): generic
    d_msm and the fixed-base-table MSM at every size, device time (CUDA events), inputs resident."""
    import torch
    out = {}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for log_n in log_sizes:
        n = 1 << log_n
        try:
            bases, scalars = net.generate_g1(0xB2000002, n), net.generate_fr(0xB2000002, n)
            part = torch.empty(16, dtype=torch.int64, device=dev)

            def timed(fn, reps):
                fn()
                evs = []
                for _ in range(reps):
                    flush.fill_(1)
                    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a0.record()
                    fn()
                    a1.record()
                    evs.append((a0, a1))
                torch.cuda.synchronize()
                t = sorted(x.elapsed_time(y) for x, y in evs)
                return t[len(t) // 2], t[0]
            reps = 5 if log_n <= 22 else 3
            ms, ms_min = timed(lambda: net.msm_dev(bases, scalars, part), reps)
            gen = net.sum_points_dev(part, 1)
            row = {"generic": {"ms": ms, "ms_min": ms_min, "mpairs_s": n / ms / 1e3,
                               "hbm_frac": 96.0 * n / (ms * 1e-3) / 1e9 / _peaks()[0]}}
            c_tab = net.msm_table_auto_window(n)
            table = net.msm_table_build(bases, c_tab)
            tms, tmin = timed(lambda: net.msm_table_dev(table, scalars, c_tab, part), reps)
            tab = net.sum_points_dev(part, 1)
            row["fixed_base"] = {"ms": tms, "ms_min": tmin, "mpairs_s": n / tms / 1e3, "window": c_tab,
                                 "table_gb": table.numel() * 8 / 2**30, "bit_exact_vs_generic": bool((tab[0] == gen[0]).all())}
            del table, bases, scalars
            torch.cuda.empty_cache()
            out["2^%d" % log_n] = row
        except Exception as e:                                 # e.g. out of memory on a smaller part: report, do not fail the line
            out["2^%d" % log_n] = {"error": str(e)[:200]}
    return out


def _cols_layout(t, ncols, world, rank):
    """device tensor (N, w) -> this rank's column layout (ncols / world, N / ncols, w)   (parallel.py)."""
    n, w = t.shape
    cg = ncols // world
    return t.reshape(n // ncols, ncols, w)[:, rank * cg:(rank + 1) * cg].permute(1, 0, 2).contiguous()


def _max_ms(times, dev):
    """median over iterations, max over ranks"""
    import torch
    import torch.distributed as dist
    t = torch.tensor(sorted(times)[len(times) // 2], device=dev, dtype=torch.float64)
    if dist.is_initialized():
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t)


def measure_multi_gpu(net, dev, rank, world, with_cpu):
    """The collectives north_star names, on the clock: four-step NTT (NCCL all-to-all vs fused peer stores), the sharded
    Groth16 prover (BASELINE config 5) and strong-scaling MSMs.  Device-event times, max over ranks."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from distributed_groth16_b200 import parallel as par
    from distributed_groth16_b200._constants import FR_ONE_MONT
    out = {}

    def ev_time(fn, reps=5, warm=2):
        for _ in range(warm):
            fn()
        ts = []
        for _ in range(reps):
            dist.barrier()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            fn()
            a1.record()
            a1.synchronize()
            ts.append(a0.elapsed_time(a1))
        return _max_ms(ts, dev)

    # ---- four-step NTT, 2^24 elements over all ranks ----------------------------------------------------------------------
    log_n = int(os.environ.get("B200ZK_BENCH_FOURSTEP_LOG_N", "24"))
    log_rows, log_cols = par.split_log(log_n)
    rows, cols = 1 << log_rows, 1 << log_cols
    cg = cols // world
    loc = net.generate_fr(0xB2000003 + rank, cg * rows).reshape(cg, rows, 4)
    be = par.GpuBackend(net)
    xch = par.P2PExchange(net, max(rows, cols) * max(rows, cols) // world)
    y_nccl = par.sharded_ntt(be, loc, log_rows, log_cols)
    y_p2p = par.sharded_ntt_p2p(net, xch, loc, log_rows, log_cols)
    same = bool((y_nccl == y_p2p).all())
    back = par.sharded_ntt_p2p(net, xch, y_p2p, log_cols, log_rows, inverse=True)
    round_trip = bool((back == loc).all())
    flags = torch.tensor([int(same), int(round_trip)], device=dev)
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    ms_nccl = ev_time(lambda: par.sharded_ntt(be, loc, log_rows, log_cols))
    ms_p2p = ev_time(lambda: par.sharded_ntt_p2p(net, xch, loc, log_rows, log_cols))
    ms_cols = ev_time(lambda: be.batched_ntt_post(loc.reshape(cg * rows, 4), log_rows, cg, False, log_base=log_n, b0=rank * cg, alpha=1))
    moved = (1 << log_n) // world * 32 * (world - 1) // world             # bytes each GPU sends (and receives)
    out["ntt_fourstep"] = {
        "log_n": log_n, "ms_nccl_all_to_all": ms_nccl, "ms_fused_p2p": ms_p2p, "ms_local_column_pass_only": ms_cols,
        "gelem_s_fused": (1 << log_n) / ms_p2p / 1e6, "bytes_sent_per_gpu": moved,
        "exchange_share_nccl": max(0.0, 1.0 - 2 * ms_cols / ms_nccl),
        "nvlink_gbs_per_gpu_if_exchange_alone": moved / max(ms_nccl - 2 * ms_cols, 1e-3) / 1e6,
        "nccl_equals_fused": bool(flags[0].item()), "inverse_round_trip_exact": bool(flags[1].item()),
        "how": "vector in the column layout of parallel.py; NCCL arm = column NTTs + all_to_all_single + row NTTs, fused arm = the "
               "column kernels' last pass stores into the owners' buffers over NVLink (no pack / all-to-all / unpack); "
               "exchange_share = 1 - 2 x (column pass alone) / whole transform"}
    del y_nccl, y_p2p, back, loc

    # ---- BASELINE config 5: sharded Groth16 prove ---------------------------------------------------------------------------
    log_m = int(os.environ.get("B200ZK_BENCH_SHARDED_LOG_M", "24"))
    m = 1 << log_m
    n_vars, n_inputs = m, 2
    n_aux = n_vars - n_inputs
    lr, lc = par.split_log(log_m)
    pcols = 1 << lc
    sl = slice(rank * n_vars // world, (rank + 1) * n_vars // world)
    sla = slice(rank * n_aux // world, (rank + 1) * n_aux // world)
    # the global dummy instance is generated on every rank (same seeds) and sliced; rank 0 keeps it for the single-GPU check
    aq, b1 = net.generate_g1(301, n_vars), net.generate_g1(302, n_vars)
    b2 = net.generate_g2(303, n_vars)
    lq, hq = net.generate_g1(304, n_aux), net.generate_g1(305, m)
    vk = np.concatenate([net.generate_g1(306, 3).cpu().numpy().view(np.uint64).reshape(-1),
                         net.generate_g2(307, 2).cpu().numpy().view(np.uint64).reshape(-1)])
    z = net.generate_fr(308, n_vars)
    z[0] = torch.from_numpy(np.array(FR_ONE_MONT, dtype=np.uint64).view(np.int64)).to(dev)
    a, b, c = (net.generate_fr(sd, m) for sd in (309, 310, 311))
    spk = par.ShardedProvingKey(net, aq[sl].contiguous(), b1[sl].contiguous(), b2[sl].contiguous(), lq[sla].contiguous(),
                                _cols_layout(hq, pcols, world, rank), n_inputs, vk)
    z_sh, zaux_sh = z[sl].contiguous(), z[n_inputs:][sla].contiguous()
    la, lb, lc_ = (_cols_layout(v, pcols, world, rank) for v in (a, b, c))
    if rank != 0:
        del aq, b1, b2, lq, hq, a, b, c, z
        torch.cuda.empty_cache()
    xch2 = par.P2PExchange(net, (1 << lr) * (1 << lr) // world)
    proofs = {}
    res = {"log_m": log_m, "fixed_base_table_gb_per_gpu": sum(t.numel() * 8 for t, _ in spk.tables.values()) / 2**30}
    for mode, x in (("nccl_all_to_all", None), ("fused_p2p", xch2)):
        ts = []
        for it in range(2 + 3):
            dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            proofs[mode] = par.sharded_prove(net, spk, z_sh, zaux_sh, la, lb, lc_, log_m, xch=x)
            torch.cuda.synchronize()
            ts.append((time.perf_counter() - t0) * 1e3)
        res["ms_" + mode] = _max_ms(ts[2:], dev)
        hs = []
        for it in range(1 + 3):
            dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            (par.sharded_h(be, la, lb, lc_, log_m) if x is None else par.sharded_h_p2p(net, x, la, lb, lc_, log_m))
            torch.cuda.synchronize()
            hs.append((time.perf_counter() - t0) * 1e3)
        res["ms_h_pipeline_" + mode] = _max_ms(hs[1:], dev)
    res["nccl_equals_fused"] = bool(proofs["nccl_all_to_all"] == proofs["fused_p2p"])
    alg = 6 * 64 * m + 4 * 32 * m + 96 * n_vars + 160 * n_vars + 96 * n_aux + 96 * m
    peak, _ = _peaks()
    res["roofline"] = {"bound": "hbm", "achieved": alg / (res["ms_fused_p2p"] * 1e-3) / 1e9, "peak": peak * world, "unit": "GB/s",
                       "frac": alg / (res["ms_fused_p2p"] * 1e-3) / 1e9 / (peak * world), "algorithmic_bytes": alg}
    res["timing"] = "host wall clock between barriers + device syncs around parallel.sharded_prove (proof bytes on every host), max over ranks"
    if rank == 0:
        try:
            from distributed_groth16_b200.groth16 import ProvingKey, prove
            pk = ProvingKey.from_device(net, aq, b1, b2, lq, hq, n_inputs, vk)
            ts = []
            for it in range(3):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                single = prove.create_proof_dev(pk, z, a, b, c)
                ts.append((time.perf_counter() - t0) * 1e3)
            res["ms_single_gpu"] = sorted(ts)[1]
            res["single_gpu_table_gb"] = pk.table_bytes / 2**30
            res["bytes_equal_single_gpu_proof"] = bool(single == proofs["fused_p2p"])
            pk.free()
        except Exception as e:
            res["single_gpu_check"] = "skipped: " + str(e)[:160]
        del aq, b1, b2, lq, hq, a, b, c, z
    torch.cuda.empty_cache()
    dist.barrier()
    out["prove_sharded"] = res
    del spk, la, lb, lc_, z_sh, zaux_sh
    torch.cuda.empty_cache()

    # ---- strong scaling: a fixed total number of pairs split over the ranks ---------------------------------------------------
    from distributed_groth16_b200.parallel import PartialExchange
    xp = PartialExchange(net)
    strong = {}
    for log_t in (24, 26):
        n_loc = (1 << log_t) // world
        bases, scalars = net.generate_g1(0xB2000002 + (rank << 24) + log_t, n_loc), net.generate_fr(0xB2000002 + rank * 7 + log_t, n_loc)
        part = torch.empty(16, dtype=torch.int64, device=dev)
        res_t = torch.empty(9, dtype=torch.int64, device=dev)

        def step():
            net.msm_dev(bases, scalars, part)
            xp.sum(part, out=res_t)
        ms = ev_time(step, reps=3, warm=1)
        strong["2^%d" % log_t] = {"pairs_per_gpu": n_loc, "ms": ms, "mpairs_s": (1 << log_t) / ms / 1e3}
        del bases, scalars
        torch.cuda.empty_cache()
    out["msm_strong"] = strong
    return out


_JSON_FD = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL's `NCCL version ...` banner comes from C
    code on fd 1): keep a private duplicate of fd 1 for the JSON line and point fd 1 at stderr for everything else."""
    global _JSON_FD
    if _JSON_FD is None:
        try:
            sys.stdout.flush()
            fd = os.dup(1)
            os.dup2(2, 1)
            _JSON_FD = fd
        except OSError:                 # no usable stderr: keep the plain stdout
            _JSON_FD = None


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, line)


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-prove", action="store_true", help="skip the secondary Groth16-prove measurements")
    ap.add_argument("--no-multi", action="store_true", help="N > 1: skip the four-step NTT / sharded prove / strong-scaling sections")
    ap.add_argument("--no-sizes", action="store_true", help="N = 1: skip the 2^22..2^26 MSM size sweep")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last timed step's result to DIR/*.npy (float64; inputs are seeded, "
                         "so runs with the same arguments can be compared output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from distributed_groth16_b200 import Net
    from distributed_groth16_b200.dist_primitives import d_msm

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus or world == 1, "launch with torchrun --nproc-per-node N for --gpus N"
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    warm = max(args.warmup, 3)
    n = 1 << LOG_N
    net = Net(local)
    net.use_torch_stream(0)
    dev = torch.device("cuda", local)
    bases = net.generate_g1(0xB2000002 + rank * 0x1000000, n)
    scalars = net.generate_fr(0xB2000002 + rank, n)
    part = torch.empty(16, dtype=torch.int64, device=dev)
    res_dev = torch.empty(9, dtype=torch.int64, device=dev)          # affine result + infinity flag (multi-GPU exchange kernel)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    xch = None
    if world > 1:
        from distributed_groth16_b200.parallel import PartialExchange
        xch = PartialExchange(net)        # peer mailboxes: d_msm's exchange is ONE kernel over NVLink stores, no NCCL call per step

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def host_result():
        r = res_dev.cpu().numpy().view(np.uint64)
        return r[:8].copy(), bool(r[8])

    def step_resident():
        net.msm_dev(bases, scalars, part)
        if world > 1:
            xch.sum(part, out=res_dev)            # publish to every peer, wait for theirs, add, normalise: stays on the device
            return None
        return net.sum_points_dev(part, 1)

    # pinned host copies for the e2e arm
    h_bases = torch.empty((n, 8), dtype=torch.int64).pin_memory()
    h_scalars = torch.empty((n, 4), dtype=torch.int64).pin_memory()
    h_bases.copy_(bases)
    h_scalars.copy_(scalars)
    hb_np, hs_np = h_bases.numpy().view(np.uint64), h_scalars.numpy().view(np.uint64)

    def step_e2e():
        if world == 1:
            return net.msm(hb_np, hs_np)                       # the C-ABI host-buffer call (b200zk_msm_g1)
        net.msm_staged(hb_np, hs_np, part)                      # H2D in parts behind the bucket kernels (b200zk_msm_staged_dev)
        xch.sum(part, out=res_dev)
        return host_result()                                   # D2H of the affine result: the step's output reaches the host

    def timed(fn, steps):
        times = []
        for _ in range(steps):
            flush.fill_(1)                                      # evict L2 between timed iterations
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            res = fn()
            b.record()
            b.synchronize()
            times.append(a.elapsed_time(b))
        return times, res

    for _ in range(warm):
        step_resident()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = net.launch_count()
    t_wall0 = time.perf_counter()
    times, res = timed(step_resident, args.steps)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = net.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *(res if world == 1 else host_result()))
    ms_step = sum(times) / len(times)
    ms_step_sorted = sorted(times)

    for _ in range(2):
        step_e2e()
    barrier()
    times_e2e, res_e2e = timed(step_e2e, max(3, min(args.steps, 10)))
    barrier()
    ms_e2e = sum(times_e2e) / len(times_e2e)
    if world > 1:
        res = host_result()
    assert (res[0] == res_e2e[0]).all()

    # steady-state throughput with the steps issued round-robin over the three stream slots, i.e. the way the
    # reference itself issues concurrent d_msm calls (MultiplexedStreamID 0..2, groth16/src/prove.rs:119-125):
    # the latency-bound tail of one MSM (bucket reduction, Horner) overlaps the bucket accumulation of the next.
    pipelined = None
    if world == 1:
        parts3 = [torch.empty(16, dtype=torch.int64, device=dev) for _ in range(3)]
        kp = max(6, args.steps)
        for _ in range(3):
            for k in range(3):
                net.msm_dev(bases, scalars, parts3[k], sid=k)
        for k in range(3):
            net.sync(k)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        outs = []
        for k in range(kp):
            if k >= 3:
                outs.append(net.sum_points_dev(parts3[k % 3], 1, sid=k % 3))      # result of step k-3 (same slot) -> host
            net.msm_dev(bases, scalars, parts3[k % 3], sid=k % 3)
        for k in range(kp, kp + 3):
            outs.append(net.sum_points_dev(parts3[k % 3], 1, sid=k % 3))
        for k in range(3):
            net.sync(k)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) * 1e3 / kp
        assert all((o[0] == res[0]).all() for o in outs)
        pipelined = {"value": n / dt / 1e3, "unit": UNIT, "ms_per_step": dt, "steps": kp,
                     "how": "steps issued round-robin on the 3 stream slots; host wall clock between device syncs; "
                            "every step's affine result is copied to the host"}

    # the same MSM over fixed-base window tables (b200zk_msm_table_*): what the proving path runs, since a proving key's
    # query vectors stay resident across proofs.  Reported beside `value`, which stays the generic d_msm (fresh bases).
    fixed_base = None
    if world == 1:
        c_tab = net.msm_table_auto_window(n)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        table = net.msm_table_build(bases, c_tab)
        e1.record()
        torch.cuda.synchronize()
        build_ms = e0.elapsed_time(e1)
        part_t = torch.empty(16, dtype=torch.int64, device=dev)
        for _ in range(3):
            net.msm_table_dev(table, scalars, c_tab, part_t)
        evs = []
        for _ in range(max(args.steps, 5)):
            flush.fill_(1)
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            net.msm_table_dev(table, scalars, c_tab, part_t)
            a1.record()
            evs.append((a0, a1))
        torch.cuda.synchronize()
        ts = sorted(x.elapsed_time(y) for x, y in evs)
        ms_t = sum(ts) / len(ts)
        got_t = net.sum_points_dev(part_t, 1)
        fixed_base = {"value": n / ms_t / 1e3, "unit": UNIT, "ms_per_step": ms_t, "ms_per_step_min": ts[0], "window": c_tab,
                      "windows": net.msm_table_windows(c_tab), "table_gb": table.numel() * 8 / 2**30, "table_build_ms": build_ms,
                      "bit_exact_vs_generic": bool((got_t[0] == res[0]).all()),
                      "how": "table[w*n+i] = 2^(c w) P_i resident in HBM; one bucket set, no Horner doublings; "
                             "CUDA events per step, L2 flushed between steps"}
        del table

    # per-kernel CUDA-event durations (separate short pass: the event pairs add launch gaps)
    net.profile(True)
    net.profile_reset()
    for _ in range(5):
        flush.fill_(1)
        step_resident()
    torch.cuda.synchronize()
    rep = net.profile_report()
    net.profile(False)

    multi = None
    gathered_inputs = None
    if world > 1:
        t = torch.tensor([ms_step, ms_e2e], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_step, ms_e2e = float(t[0]), float(t[1])
        if not args.no_cpu_baseline:
            # every rank's inputs go to rank 0, which checks the N-GPU result against the CPU restatement on the whole input
            gb = [torch.empty_like(bases) for _ in range(world)] if rank == 0 else None
            gs = [torch.empty_like(scalars) for _ in range(world)] if rank == 0 else None
            dist.gather(bases, gb, dst=0)
            dist.gather(scalars, gs, dst=0)
            if rank == 0:
                gathered_inputs = (np.concatenate([x.cpu().numpy().view(np.uint64) for x in gb]),
                                   np.concatenate([x.cpu().numpy().view(np.uint64) for x in gs]))
                del gb, gs
        del bases, scalars
        torch.cuda.empty_cache()
        if not args.no_multi:
            multi = measure_multi_gpu(net, dev, rank, world, not args.no_cpu_baseline)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = _peaks()
    # the bucket kernel runs once per window group (msm.cu, window-group pipeline): each launch processes 1/G of every
    # pair's digits, i.e. 96 n / G algorithmic bytes, in 1/G of the step's bucket time -- same GB/s either way
    acc = rep.get("msm_accumulate_g1", {"launches": 5, "ms": float("nan")})
    acc_launches_per_step = max(acc["launches"], 1) / 5.0
    acc_ms_launch = acc["ms"] / max(acc["launches"], 1)
    acc_ms = acc["ms"] / 5.0                                                  # per step, all launches
    achieved = ALG_BYTES_PER_PAIR * n / acc_launches_per_step / (acc_ms_launch * 1e-3) / 1e9
    kernel_ms = {k: round(v["ms"] / 5.0, 4) for k, v in rep.items()}
    # what actually bounds the kernel: the multiplier pipe.  A 256-bit Montgomery product = 128 32-bit wide multiply-adds
    # with carry, which issue at 32 lanes/clk/SM (tools/microbench.cu, profiles/r1_microbench_pipes.txt).
    sm_mhz = clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965.0
    pipe_peak = 32.0 * torch.cuda.get_device_properties(dev).multi_processor_count * sm_mhz * 1e6 / 128.0 / 1e9          # G products/s
    adds = n * 16.0 * (1.0 - 2.0 ** -16)                                      # 16 signed 16-bit digits per scalar (GLV: 2 x 8)
    pipe_ach = adds * 10.0 / (acc_ms * 1e-3) / 1e9                            # XYZZ mixed addition = 8M + 2S
    pipe = {"bound": "fmaheavy (32-bit multiply-add with carry)", "achieved": pipe_ach, "peak": pipe_peak,
            "unit": "G modular products/s", "frac": pipe_ach / pipe_peak,
            "how": "bucket additions (n x 16 digits) x 10 products / kernel time; peak = 32 lanes/clk/SM x SMs x SM clock / 128"}
    out = {
        "metric": METRIC, "value": world * n / ms_step / 1e3, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": warm, "ms_per_step": ms_step, "ms_per_step_median": ms_step_sorted[len(ms_step_sorted) // 2],
        "ms_per_step_min": ms_step_sorted[0], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32x8 Montgomery (256-bit modular integers)", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "pairs_per_gpu": n, "l2": "256 MiB flush write between timed iterations; inputs+workspace > L2",
                   "parallelism": "length-sharded x%d; partials exchanged by one kernel over NVLink peer mailboxes "
                                  "(b200zk_msm_exchange_sum_dev), no NCCL call in the step" % world},
        "e2e": {"value": world * n / ms_e2e / 1e3, "unit": UNIT, "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": n * 96, "d2h_bytes_per_step": 72},
        "gpu_launches": int(launches),
        "wall_s_timed_region": t_wall,
        "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": "msm_accumulate_g1", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": None, "peak_source": peak_src, "kernel_ms": acc_ms_launch,
                     "launches_per_step": acc_launches_per_step, "kernel_ms_per_step": acc_ms,
                     "algorithmic_bytes_per_launch": ALG_BYTES_PER_PAIR * n / acc_launches_per_step,
                     "note": "256-bit modular integer arithmetic: IMAD-bound by construction, HBM fraction is small",
                     "pipe": pipe},
        "kernel_ms_per_step": kernel_ms,
        "pipelined": pipelined,
        "fixed_base": fixed_base,
    }
    traffic_file = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(traffic_file):
        try:
            tj = json.load(open(traffic_file))
            out["roofline"]["traffic"] = tj.get("msm_accumulate_g1_bytes_per_launch")
            out["roofline"]["traffic_source"] = "static: ncu --set full capture recorded in profiles/traffic.json (%s), not measured in this run" % tj.get("source", "see profiles/README.md")
        except Exception:
            pass
    if not args.no_cpu_baseline:
        from oracle import cref                                  # cpu_baseline leg: the checker timed as a baseline
        cref.build()
        if world == 1:
            hb, hs = bases.cpu().numpy().view(np.uint64), scalars.cpu().numpy().view(np.uint64)
        else:
            hb, hs = gathered_inputs
        t0 = time.perf_counter()
        ncores = os.cpu_count() or cref.num_threads()
        exp, _ = cref.msm_g1(hb, hs, ncores)
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": hb.shape[0] / dt / 1e6, "unit": UNIT, "cores": ncores, "kind": "port",
                               "sample": "one full %d x 2^%d-pair G1 MSM (all ranks' inputs), arkworks-equivalent CPU restatement, "
                                         "all host threads (%.2f s)" % (world, LOG_N, dt),
                               "bit_exact_vs_gpu": bool((exp == res[0]).all())}
    if multi:
        out.update(multi)
    if world == 1:
        out["ntt"] = measure_ntt(net, peak, pipe_peak)
    if world == 1 and not args.no_prove:
        out["prove"] = measure_prove(net, args, not args.no_cpu_baseline)
        out["prove_sha256"] = measure_prove_sha256(net, not args.no_cpu_baseline)
    if world == 1 and not args.no_sizes:
        del bases, scalars
        torch.cuda.empty_cache()
        out["msm_sizes"] = measure_msm_sizes(net, dev, (22, 24, 26))
    emit(out)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
