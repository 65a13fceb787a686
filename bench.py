#!/usr/bin/env python3
"""bench.py — BLS12-381 G1 Pippenger MSM throughput (BASELINE.json configs[1]), the G1-MSM half
of the headline metric "MPN Groth16 proofs/sec ...; G1 MSM scalars/sec vs HBM roofline".

  python bench.py --gpus N --steps K --warmup W            our arm  (N>1: launched under torchrun)
  python bench.py --impl reference --gpus N --steps K ...   the CPU arm (rank 0 only)
  ... --dump-outputs DIR    also write the last timed step's result to DIR/g1_msm_sum.npy (see dump_outputs)

A step = one multi-scalar multiplication sum_i [s_i] P_i over synthetic inputs: per GPU 2^20
uniform Fr scalars (SplitMix64) and 2^20 bases P_i = [k_i] G.  At N GPUs the job is ONE MSM of
N * 2^20 terms base-sharded across the ranks (weak scaling): every rank reduces its shard to one
point, the N partial points are all-gathered over NCCL (104 B each) and folded.

  value     scalars/s, whole job, bases AND scalars resident in HBM when the timed region starts
  e2e       the same through the C-ABI call a prover makes per proof: scalars start in pinned HOST
            memory and are copied inside the timed region, the affine result lands in host memory;
            bases stay resident (they are the proving key: loaded once per circuit, like
            bellman's `Parameters`); e2e.cold also re-uploads the bases every step
  roofline  dominant kernel (bucket accumulation): 128 B/term algorithmic over its CUDA-event time
  cpu_baseline  the C oracle (bellman-equivalent multiexp) on the host cores, same inputs
Timing: CUDA events on the launching stream around every step, L2 flushed before each step,
barrier + synchronize on both sides of the region, MAX over ranks.
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

METRIC = "g1_msm_scalars_per_sec"
UNIT = "scalars/s"
LOG_N_DEFAULT = 20
ALGO_BYTES_PER_TERM = 128  # 32 B scalar + 96 B affine base (SURVEY.md §8d)
DTYPE = "u32x12 Montgomery (Fp) / u32x8 (Fr) on the GPU; u64 limbs on the CPU"


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.idx)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(int(r[1]) for r in self.rows if len(r) >= 8 and r[1].isdigit())
        mx = [int(r[2]) for r in self.rows if len(r) >= 8 and r[2].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[k] for r in self.rows if len(r) >= 8 for k in range(4) if r[4 + k].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
    """dram bytes per launch of the dominant kernel from the committed ncu --set full capture."""
    p = os.path.join(ROOT, "profiles", "msm_accumulate_ncu.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get("dram_bytes_per_launch")
        except Exception:
            return None
    return None


# ------------------------------------------------------------------------------------------------
def workload_string(log_n, world):
    """identical in both arms (the driver compares the strings)"""
    return (f"BLS12-381 G1 Pippenger MSM, {world} x 2^{log_n} random scalars/bases (BASELINE configs[1]); "
            f"one sum of {world << log_n} terms, base-sharded over {world} GPU(s)")


def rank_inputs_seeds(rank):
    """rank r owns terms [r*n, (r+1)*n) of the N*n-term job: bases stream seed, scalars stream seed"""
    return 2 + 7919 * rank, 1 + 104729 * rank


def dump_outputs(out_dir, arrays):
    """Each named array to out_dir/<name>.npy as float64, so that two builds (or the two arms) can be compared output
    for output.  The bench's result is the 104-byte affine image of the MSM sum (x | y | inf | pad), written one byte
    per element: exact in float64, and equal images mean equal points."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def run_reference(args, rank, world):
    """CPU arm: the reference's algorithm (bellman multiexp restated in C — the reference itself is
    Rust on un-vendored crates and cannot be built here) on the host cores this process may use, on
    the SAME workload as our arm at every N: one sum of N * 2^log_n terms (rank r's 2^log_n terms are
    generated from the same seeds as on the GPU side)."""
    if rank != 0:
        return
    import numpy as np
    from oracle import cref  # the only other place bench.py may execute oracle/
    n = 1 << args.log_n
    info = cref.cpu_info()
    cores = info["usable"]
    bases = np.concatenate([cref.g1_random_bases(rank_inputs_seeds(r)[0], n, cores) for r in range(world)])
    scalars = np.concatenate([cref.fr_random(rank_inputs_seeds(r)[1], n) for r in range(world)])
    total = world * n
    for _ in range(args.warmup):
        cref.msm_g1(bases, scalars, cores)
    per_step = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        result = cref.msm_g1(bases, scalars, cores)
        per_step.append(time.perf_counter() - t0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"g1_msm_sum": result})
    dt = sum(per_step) / max(len(per_step), 1)
    val = total / dt
    srt = sorted(per_step)
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
        "config": {"workload": workload_string(args.log_n, world), "terms_total": total,
                   "note": "CPU restatement of bellman 0.14 multiexp (window ceil(ln n), threads = windows x base chunks), "
                           "not bellman; full job per step"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "cpu": info,
                         "sample": f"{args.steps} x full {world} x 2^{args.log_n}-term MSM, wall clock per step",
                         "step_s_min": srt[0], "step_s_median": srt[len(srt) // 2], "step_s_max": srt[-1],
                         "value_at_min_step": total / srt[0]},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def run_ours(args, rank, local_rank, world):
    import numpy as np
    import torch
    import bazuka_b200 as B

    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = B.Context(local_rank)
    ctx.use_torch_stream()
    n = 1 << args.log_n

    # ---- synthetic inputs, generated by libbzk kernels straight into HBM -------------------------
    # rank r owns terms [r*n, (r+1)*n) of the N*n-term job: bases from stream seed 2, scalars seed 1
    d_img = torch.empty((n, 104), dtype=torch.uint8, device="cuda")
    ctx.g1_random_bases_dev(rank_inputs_seeds(rank)[0], n, d_img)
    bases = ctx.g1_bases_from_dev(d_img, n)
    # resident bases = a proving-key column: build its fixed-base table once, outside the timed region (as at key load)
    t_tab = time.perf_counter()
    table_levels = bases.precompute(args.table_levels) if args.table_levels > 1 else 1
    torch.cuda.synchronize()
    t_tab = time.perf_counter() - t_tab
    d_scalars = torch.empty((n, 4), dtype=torch.int64, device="cuda")
    ctx.fr_random_dev(rank_inputs_seeds(rank)[1], n, d_scalars)
    h_scalars = d_scalars.cpu().pin_memory()
    h_img = d_img.cpu().pin_memory() if rank == 0 else None
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    torch.cuda.synchronize()

    from bazuka_b200 import dist as bd

    def fold(partial):
        """N>1: one NCCL all-gather of the per-rank partial points (104 B each), then local adds."""
        return bd.allgather_fold(partial, "g1", device="cuda") if world > 1 else partial

    def step_resident():
        return fold(ctx.msm_g1_resident(bases, d_scalars))

    def step_e2e():
        return fold(ctx.msm_g1_resident(bases, h_scalars))

    def timed(step_fn, steps, warmup, after_warmup=None):
        for _ in range(warmup):
            step_fn()
        if after_warmup:
            after_warmup()  # e.g. reset the stage timers so lazy kernel loading is not averaged in
        if dist:
            dist.barrier()
        torch.cuda.synchronize()
        t_wall = time.perf_counter()
        total_ms = 0.0
        res = None
        for _ in range(steps):
            flush.fill_(1)  # evict L2 (outside the per-step event pair)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            res = step_fn()
            e1.record()
            e1.synchronize()
            total_ms += e0.elapsed_time(e1)
        if dist:
            dist.barrier()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t_wall
        t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
        if dist:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), wall, res

    sampler = ClockSampler(local_rank)
    launches = [0]

    def begin_region():
        ctx.set_timing(True)
        launches[0] = ctx.launch_count
        if rank == 0:
            sampler.start()

    total_ms, wall, result = timed(step_resident, args.steps, args.warmup, begin_region)
    clocks = sampler.stop() if rank == 0 else None
    launches = ctx.launch_count - launches[0]
    runs, _, stage_sum = ctx.stage_ms()
    ctx.set_timing(False)
    ms_step = total_ms / args.steps
    value = world * n / (ms_step * 1e-3)

    e2e_ms, _, result_e2e = timed(step_e2e, args.steps, max(args.warmup, 3))
    e2e_step = e2e_ms / args.steps
    assert (result_e2e == result).all(), "e2e and resident paths disagree"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"g1_msm_sum": result})

    mpn_multi = None
    if world > 1 and not args.no_mpn:
        mpn_multi = {"single_update": mpn_groth16_section(ctx, with_cpu=False, dist=dist, world=world)}
    batch = None
    if not args.no_mpn:
        # the proofs/s half of the metric on a whole update batch (all ranks: the N>1 schedules have collectives)
        from tools.mpn_batch_bench import batch_section
        shape = (16, 3, 5) if args.workload == "mpn1024" else (15, 3, 4)
        try:
            batch = batch_section(ctx, *shape, steps=args.mpn_steps, dist=dist, rank=rank, world=world, peak_gbs=measured_peak()[0])
        except Exception as e:
            batch = {"error": repr(e)}
    if rank != 0:
        if dist:
            dist.destroy_process_group()
        return

    # stage split of the timed region: averages of the CUDA-event marks over the timed steps only
    stages = {name: float(stage_sum[i] / max(runs, 1)) for i, name in enumerate(B.Context.MSM_STAGES)}
    acc_ms = stages["accumulate"]
    peak, peak_src = measured_peak()
    achieved = ALGO_BYTES_PER_TERM * n / (acc_ms * 1e-3) / 1e9 if acc_ms > 0 else None

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": DTYPE, "data": "synthetic",
        "config": {
            "workload": workload_string(args.log_n, world),
            "terms_total": world * n, "parallelism": f"base-sharded x{world}, 1 NCCL all-gather of {104 * world} B" if world > 1 else "single GPU",
            "l2": "512 MiB write before every timed step (L2 flushed); inputs 132 MB > 126 MB L2",
            "timing": "CUDA events on the launching stream per step, barrier+sync around region, max over ranks",
            "result_check": "sum folded on every rank; e2e result == resident result",
            "bases": f"resident with a fixed-base table of {table_levels} levels ({96 * table_levels * n >> 20} MiB per GPU, built once in "
                     f"{t_tab:.2f} s outside the timed region, as a proving key is at load); e2e.cold re-uploads plain bases every step",
        },
        "gpu_launches": int(launches),
        "wall_s_region": wall,
        "stages_ms": stages,
        "roofline": {
            "bound": "hbm", "kernel": "k_accumulate<Fp> (bucket accumulation, mixed XYZZ adds)",
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
            "traffic": ncu_traffic(), "peak_source": peak_src,
            "algorithmic_bytes_per_launch": ALGO_BYTES_PER_TERM * n,
            "kernel_ms": acc_ms, "frac_of_nominal_8TBs": (achieved / 8000.0) if achieved else None,
            "note": "integer-ALU bound (13 windows over the fixed-base table x ~11 Fp products per term); see DESIGN.md section 3.1-3.2 for the IMAD roofline",
        },
        "e2e": {"value": world * n / (e2e_step * 1e-3), "unit": UNIT, "ms_per_step": e2e_step,
                "h2d_bytes_per_step": 32 * n, "d2h_bytes_per_step": 16 * 192 + 104,
                "note": "scalars from pinned host memory each step; bases resident (proving key)"},
        "clocks": clocks,
    }

    if world == 1:
        # cold end-to-end: bases (104 MB) and scalars both from pinned host memory every step
        def step_cold():
            rb = ctx.g1_bases(h_img)
            out = ctx.msm_g1_resident(rb, h_scalars)
            rb.free()
            return out
        cold_ms, _, rc = timed(step_cold, max(2, min(args.steps, 5)), 1)
        assert (rc == result).all()
        cold_step = cold_ms / max(2, min(args.steps, 5))
        line["e2e"]["cold"] = {"value": n / (cold_step * 1e-3), "ms_per_step": cold_step, "h2d_bytes_per_step": 136 * n}

        # CPU baseline on this box's host cores, same inputs (bounded: one full-size MSM + one warm-up)
        try:
            from oracle import cref  # cpu_baseline leg only
            cpu = cref.cpu_info()
            cores = cpu["usable"]
            hb = h_img.numpy()
            hs = h_scalars.numpy().view(np.uint64)
            cref.msm_g1(hb[: n // 8], hs[: n // 8], cores)
            t0 = time.perf_counter()
            cpu_out = cref.msm_g1(hb, hs, cores)
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": n / dt, "unit": UNIT, "cores": cores, "kind": "port", "cpu": cpu,
                                    "sample": f"1 x full 2^{args.log_n}-term MSM ({dt:.2f} s wall), bellman-equivalent C restatement, not bellman",
                                    "matches_gpu": bool((cpu_out == result).all())}
        except Exception as e:  # the oracle is test infrastructure; its absence must not break the bench
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"unavailable: {e}"}
        if not args.no_mpn:
            line["mpn_groth16"] = {"single_update": mpn_groth16_section(ctx)}
    if mpn_multi is not None:
        line["mpn_groth16"] = mpn_multi
    if batch is not None:
        line["mpn_groth16"]["update_batch"] = batch
        po = batch.get("prove_only") or {}
        line["mpn_groth16"]["headline"] = {"metric": "mpn_groth16_proofs_per_sec", "circuit": batch.get("circuit"), "n_gpus": world,
                                           "proofs_per_s_1gpu_prove_only": po.get("proofs_per_s"),
                                           "proofs_per_s_replicas": (batch.get("replicas") or {}).get("proofs_per_s"),
                                           "ms_per_proof_sharded": (batch.get("sharded") or {}).get("ms_per_proof")}
    print(json.dumps(line), flush=True)
    if dist:
        dist.destroy_process_group()


def mpn_groth16_section(ctx, with_cpu=True, dist=None, world=1):
    """BASELINE configs[0]: one MPN state update (UpdateCircuit A=15,T=3,B=0: a signed transfer between two
    funded accounts on the production tree shape) — Groth16 prove on the GPU, the same proof on the CPU
    oracle (all host cores) and the pairing check of the GPU proof.  Secondary to the MSM headline; kept
    small (about 57 k constraints) so the default bench stays within minutes."""
    import numpy as np
    import torch
    from bazuka_b200 import groth16 as BG
    from bazuka_b200.mpn import cs as C, native as N, update as U
    out = {"circuit": "UpdateCircuit A=15 T=3 B=0 (1 tx), /root/reference/src/mpn/circuits/update_circuit.rs"}
    try:
        st, keys = U.MpnState(15, 3), []
        for i in range(2):
            pk, sk = N.eddsa_keys(b"ABC" if i == 0 else b"DEF")
            keys.append((pk, sk))
            st.set(i, U.MpnAccount(0, 0, pk, {0: U.Money(U.ZIESHA, 10 ** 12)}))
        tx = U.MpnTransaction(1, N.jj_compress(keys[0][0]), N.jj_compress(keys[1][0]), U.Money(U.ZIESHA, 1000), U.Money(U.ZIESHA, 10))
        tx.sign(keys[0][1])
        pub, trans, _ = U.update(st, [tx], 0)
        t0 = time.perf_counter()
        cs = U.UpdateCircuit(15, 3, 0, commitment=1, height=0, transitions=trans, **pub).synthesize(C.ConstraintSystem())
        ni, na, mats, inputs, aux = cs.to_csr()
        out.update({"constraints": cs.num_constraints, "aux": na, "host_synthesize_s": time.perf_counter() - t0})
        pr = BG.Prover(ctx, BG.R1CS(ni, na, *mats))
        d = torch.empty((7, 4), dtype=torch.int64, device="cuda")
        ctx.fr_random_dev(99, 7, d)
        torch.cuda.synchronize()
        rnd = d.cpu().numpy().view(np.uint64)
        pk, vk = BG.setup_gpu(ctx, pr.r1cs, rnd[:5], BG.G1_GENERATOR, BG.G2_GENERATOR)
        blob, pts = pr.prove(pk, inputs, aux, rnd[5], rnd[6])
        ts = []
        for _ in range(5):
            t0 = time.perf_counter()
            b2, _ = pr.prove(pk, inputs, aux, rnd[5], rnd[6], check_satisfied=False)
            ts.append(time.perf_counter() - t0)
        out.update({"log_m": pr.log_m, "gpu_prove_ms": min(ts) * 1e3, "gpu_proofs_per_s": 1 / min(ts),
                    "timing": "host wall clock around bzk_groth16_prove (host witness in, 387-byte proof out), best of 5"})
        # replicas: every GPU proves independent works back to back (the reference's own parallel axis:
        # independent proofs farmed to workers, /root/reference/src/mpn/mod.rs:79-107) — no communication
        reps = 20
        if dist:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            pr.prove(pk, inputs, aux, rnd[5], rnd[6], check_satisfied=False)
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if dist:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        out["replicas"] = {"n_gpus": world, "proofs": reps * world, "wall_s_max_over_ranks": float(dt.item()),
                           "proofs_per_s": reps * world / float(dt.item()), "verified": bool(BG.verify(vk, inputs[1:], pts))}
        if not with_cpu:
            return out
        from oracle import groth16_c as GC  # CPU baseline + big-integer pairing check only
        a_idx, b_idx = GC.density(ni, na, mats)
        cpk = {"log_m": pr.log_m, "vk": vk, "a_idx": a_idx, "b_idx": b_idx}
        for k in ("h", "l", "a", "b_g1", "b_g2"):
            cpk[k] = pk.device_images[k].cpu().numpy()
        GC.prove(ni, na, mats, cpk, inputs, aux, rnd[5], rnd[6])
        t0 = time.perf_counter()
        cpu_pts = GC.prove(ni, na, mats, cpk, inputs, aux, rnd[5], rnd[6])
        dt = time.perf_counter() - t0
        out.update({"cpu_prove_ms": dt * 1e3, "cpu_proofs_per_s": 1 / dt, "cpu_cores": GC.cref.usable_cpus(),
                    "proof_bytes_equal_cpu": bool((blob == GC.proof_bytes(*cpu_pts)).all()),
                    "pairing_check_accepts_gpu_proof": bool(GC.verify_py(vk, inputs[1:], pts))})
        t0 = time.perf_counter()
        ok = BG.verify(vk, inputs[1:], pts)
        out.update({"libbzk_verify_accepts": bool(ok), "libbzk_verify_ms": (time.perf_counter() - t0) * 1e3})
    except Exception as e:
        out["error"] = repr(e)
    return out


def sharded_proof_section(ctx, dist, rank, world):
    """SURVEY.md §8e schedule (S): ONE proof over all GPUs — every rank keeps a contiguous 1/N of the five base
    vectors, sums its shard (bzk_groth16_prove_partial), one NCCL all-gather of 512 B per rank, host folds and
    bzk_groth16_finalize.  Measured on a 2^20-domain synthetic MPN-like circuit; the sharded proof must equal the
    single-GPU proof byte for byte.  (tools/bench_sharded.py runs larger domains.)"""
    import numpy as np
    import torch
    from bazuka_b200 import groth16 as BG, synth
    out = {"circuit": "synthetic MPN-like, 1024 lanes x 100 rounds"}
    try:
        dev = torch.device("cuda", torch.cuda.current_device())
        ni, na, mats, inputs, aux = synth.build(1024, 100, seed=17, ops=synth.GpuOps(ctx))
        pr = BG.Prover(ctx, BG.R1CS(ni, na, *mats))
        d = torch.empty((7, 4), dtype=torch.int64, device=dev)
        ctx.fr_random_dev(99, 7, d)
        torch.cuda.synchronize()
        rnd = d.cpu().numpy().view(np.uint64)
        pk, vk = BG.setup_gpu(ctx, pr.r1cs, rnd[:5], BG.G1_GENERATOR, BG.G2_GENERATOR)
        spk = BG.shard_proving_key(ctx, pk, pr.log_m, rank, world)
        want, _ = pr.prove(pk, inputs, aux, rnd[5], rnd[6])

        def sharded():
            sums = BG.allgather_partials(pr.prove_partial(spk, inputs, aux, check_satisfied=False), device=dev)
            return BG.finalize(vk, sums, rnd[5], rnd[6])

        def timed_max(fn, reps=5):
            best = None
            for _ in range(reps):
                dist.barrier()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn()
                torch.cuda.synchronize()
                t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                best = float(t.item()) if best is None else min(best, float(t.item()))
            return best

        blob, pts = sharded()
        t_sh = timed_max(sharded)
        t_one = timed_max(lambda: pr.prove(pk, inputs, aux, rnd[5], rnd[6], check_satisfied=False))
        out.update({"constraints": pr.r1cs.num_constraints, "log_m": pr.log_m, "n_gpus": world,
                    "sharded_ms_per_proof": t_sh * 1e3, "single_gpu_ms_per_proof": t_one * 1e3, "exchange_bytes_per_rank": 512,
                    "proof_bytes_equal_single_gpu": bool((blob == want).all()), "verified": bool(BG.verify(vk, inputs[1:], pts)),
                    "timing": "wall clock between device synchronisations, max over ranks, best of 5"})
        spk.free(); pk.free(); pr.free()
    except Exception as e:
        out["error"] = repr(e)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log-n", type=int, default=LOG_N_DEFAULT)
    ap.add_argument("--table-levels", type=int, default=16, help="fixed-base table levels for the resident bases (1 = none)")
    ap.add_argument("--no-mpn", action="store_true", help="skip the MPN proof sections (single update + whole update batch)")
    ap.add_argument("--workload", default="mpn256", choices=["mpn256", "mpn1024"],
                    help="update batch proved in the mpn_groth16 section: production 256-tx batch (2^24) or BASELINE configs[3] 1024-tx (2^26)")
    ap.add_argument("--mpn-steps", type=int, default=3, help="timed update-batch proofs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the MSM sum of the last timed step to DIR/g1_msm_sum.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    rank, local_rank, world = env_int("RANK", 0), env_int("LOCAL_RANK", 0), env_int("WORLD_SIZE", 1)
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
