#!/usr/bin/env python
"""bench.py — leapfrog-steps/s of the many-chain NUTS hot path (BASELINE.json metric).

Default workload at N=1 (BASELINE.json configs[1], "C2"): 1000-dim standard MvNormal, 65 536 chains, diagonal M⁻¹,
FP64, 1×B200.  Setup (untimed): random start, initial step-size search, one dual-averaging stage so that ϵ is
adapted per chain.  A timed "step" = one pass of the hot path over the batch: `draws_per_step` NUTS transitions for
every chain (dhmc_mcmc_dev, state and outputs in HBM).  `value` = Σ tree_statistics.steps ÷ device time (CUDA events
on the library's stream, max over ranks); `e2e` repeats the same step through the host-buffer C ABI call
(dhmc_mcmc_from): positions uploaded from page-locked host memory, draws + statistics written into page-locked host
buffers, all inside the timed region.

--config selects the other BASELINE.json configurations (same JSON contract):
  C3  Neal's funnel D=10, 262 144 chains, diagonal metric adapted by the default warm-up
  C4  logistic regression N=10 000, p=256, 32 768 chains per GPU, per-chain dense (Symmetric) metric adapted in warm-up;
      likelihood and M⁻¹p on the FP64 tensor cores; roofline bound = FP64 tensor (DMMA) peak
  C5  1000-dim MvNormal with κ = 10⁴, 65 536 chains per GPU, FULL default warm-up (untimed, reported), then sampling

N>1 (torchrun): chains are sharded (rank r owns global chains r·B … (r+1)·B-1, the Philox key is the global id), no
data-path collective, weak scaling; the last draw of every chain is all-gathered once after the timed region through
the library's own NCCL communicator (dhmc_comm_init / dhmc_allgather_dev; torch.distributed only carries the 128-byte
id and the timing reductions).  NCCL_DEBUG is left exactly as the caller set it.

--impl reference: the reference's CPU path.  Julia is not in this image, so this is the oracle port (oracle/, C++
restatement of DynamicHMC.jl) on the host cores this process may use, threads pinned, 3 repetitions per step.
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
import __graft_entry__ as entry  # noqa: E402

METRIC = "leapfrog_steps_per_sec"
UNIT = "leapfrog-steps/s"
# FP64 tensor-core (DMMA m8n8k4) rate measured on this pool's B200 by benchmarks/c4_probes.cu
# (profiles/r02_c4_probes.txt): 64 FMA/clk/SM — the same as the DFMA pipe; x 148 SMs x SM clock x 2 flop
DMMA_FMA_PER_CLK_SM = 64.0


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), float(d.get("sm_max_mhz", 1965.0)), "measured"
        except Exception:
            pass
    return 6650.0, 1965.0, "fallback"


def usable_cores():
    """Cores this process may really use: affinity mask ∩ cgroup CPU quota (a 128-thread box with a 16-CPU quota
    runs 128 busy threads 8x slower — the 6x swing of the round-1 CPU arm)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    if quota:
        n = max(1, min(n, int(quota)))
    return n, quota


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
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
            pass
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(np.max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- workloads
def make_workload(pkg, name, args):
    """-> dict(model, chains, dim, draws_per_step, label, setup(eng) -> info, algo_flops/bytes per leapfrog …)"""
    if name == "C2":
        D = args.dim or 1000
        return dict(model=pkg.StandardNormal(D), dim=D, chains=args.chains or 65536, draws=args.draws_per_step or 2,
                    label=f"{D}-dim standard MvNormal, diagonal per-chain M^-1, eps adapted by dual averaging",
                    warm="search+%d dual-averaging transitions" % args.adapt_steps,
                    stages=[pkg.TuningNUTS(args.adapt_steps, pkg.DualAveraging())], bytes_per_lf=48 * D, flops_per_lf=None)
    if name == "C3":
        return dict(model=pkg.Funnel(10), dim=10, chains=args.chains or 262144, draws=args.draws_per_step or 10,
                    label="Neal's funnel D=10, diagonal per-chain M^-1 from the default warm-up",
                    warm="default_warmup_stages() (900 transitions)", stages=list(pkg.default_warmup_stages())[1:],
                    bytes_per_lf=48 * 10, flops_per_lf=None)
    if name == "C4":
        N, p = 10000, 256
        ℓ, _ = pkg.LogisticRegression.synthetic(N=N, p=p, seed=7)
        st = [pkg.TuningNUTS(args.c4_warm[0], pkg.DualAveraging()),
              pkg.TuningNUTS(args.c4_warm[1], pkg.DualAveraging(), pkg.Symmetric),
              pkg.TuningNUTS(args.c4_warm[2], pkg.DualAveraging())]
        return dict(model=ℓ, dim=p, chains=args.chains or 32768, draws=args.draws_per_step or 1,
                    label=f"logistic regression N={N} p={p}, per-chain dense (Symmetric) M^-1 adapted in warm-up, "
                          "likelihood and M^-1 p on the FP64 tensor cores",
                    warm="search + TuningNUTS(%d) + TuningNUTS(%d, Symmetric) + TuningNUTS(%d)" % tuple(args.c4_warm),
                    stages=st, bytes_per_lf=None,
                    flops_per_lf=4.0 * N * p + 2 * 2.0 * p * p)          # SURVEY §8d: likelihood 4Np + two mat-vecs 2·2p²
    if name == "C5":
        D = args.dim or 1000
        sig2 = 10.0 ** (4.0 * np.arange(D) / (D - 1))
        return dict(model=pkg.DiagNormal(np.zeros(D), sig2), dim=D, chains=args.chains or 65536, draws=args.draws_per_step or 2,
                    label=f"{D}-dim MvNormal, kappa=1e4 (sigma_i^2 = 10^(4(i-1)/{D - 1})), FULL default warm-up (900 transitions: "
                          "dual averaging + diagonal metric windows), then sampling",
                    warm="default_warmup_stages() (900 transitions)", stages=list(pkg.default_warmup_stages())[1:],
                    bytes_per_lf=56 * D, flops_per_lf=None)
    raise SystemExit(f"unknown --config {name}")


def oracle_family(po, pkg, wl):
    m = wl["model"]
    if isinstance(m, pkg.StandardNormal):
        return po.FAMILY_STD_NORMAL, None
    if isinstance(m, pkg.DiagNormal):
        return po.FAMILY_DIAG_NORMAL, m.params()
    if isinstance(m, pkg.Funnel):
        return po.FAMILY_FUNNEL, None
    return po.FAMILY_LOGISTIC, m.params()


def cpu_arm(po, fam, params, D, T, eps, seconds, reps=3):
    """Oracle port on the usable host cores: one chain per pinned thread, `reps` repetitions, median rate."""
    cores, quota = usable_cores()
    kw = dict(T=T, eps0=eps, params=params)
    st, sec = po.bench_mcmc(fam, D, cores, cores, 2, seed=2026, **kw)           # calibration
    draws = max(2, int(seconds * (st / sec) / max(st / 2, 1)))
    rates, secs, steps = [], [], []
    for r in range(reps):
        s, t = po.bench_mcmc(fam, D, cores, cores, draws, seed=2026 + r, **kw)
        rates.append(s / t); secs.append(t); steps.append(s)
    med = float(np.median(rates))
    return dict(value=med, rates=[float(x) for x in rates], seconds=float(np.sum(secs)), steps=int(np.sum(steps)),
                cores=cores, draws=draws, quota=quota)


def run_reference(args, rank, world):
    """CPU arm: oracle port, all usable host threads (pinned), same config / metric; each step = 3 repetitions of a
    bounded sample."""
    if rank != 0:
        return
    po = entry.load_oracle()
    pkg = entry.load_package()
    wl = make_workload(pkg, args.config, args)
    fam, params = oracle_family(po, pkg, wl)
    D = wl["dim"]
    eps = args.ref_eps if args.config in ("C2", "C5") else (0.05 if args.config == "C4" else 0.2)
    vals, total_t, total_s, last = [], 0.0, 0, None
    for it in range(args.warmup + args.steps):
        r = cpu_arm(po, fam, params, D, 32 if D <= 256 else 128, eps, args.ref_seconds, reps=3)
        if it >= args.warmup:
            vals.append(r["value"]); total_t += r["seconds"]; total_s += r["steps"]
        last = r
    value = float(np.median(vals))
    cores = last["cores"]
    sample = (f"{cores} chains x {last['draws']} draws x 3 repetitions per step at D={D}, fixed eps={eps}, identity metric, "
              f"one chain per pinned std::thread ({cores} threads; cgroup quota {last['quota']}); median of the repetition rates")
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total_t / max(args.steps, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "impl": "reference",
            "config": {"workload": f"{args.config}: {wl['label']} (CPU arm: bounded sample)", "dim": D, "chains": cores,
                       "draws_per_step": last["draws"]},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                             "per_core": value / cores, "cpu_model": cpu_model(), "step_values": vals},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def bind_to_gpu_numa_node(local_rank):
    """CPU affinity of this rank = the CPUs of its GPU's NUMA node (pinned buffers are then first-touched there)."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local_rank)
        bus = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for tok in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = tok.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def user_model_leg(pkg, wl, K, D, n, args, local_rank, chain_offset, draws, stats, logd, ref_steps, ref_ms):
    """The C2 step once more with ℓ supplied as a USER model header (include/models/std_normal_user.h compiled into its own
    build of the library, DESIGN.md §4.2): same seed, same setup, same number of warm-up and timed steps, so the chains are
    the shipped family's bit for bit (`same_trees`) and the two rates compare the kernels alone.  Never fails the bench:
    an error is reported in the returned dict."""
    try:
        hdr = os.path.join(ROOT, "include", "models", "std_normal_user.h")
        t0 = time.perf_counter()
        ℓ = pkg.UserLogDensity(hdr, D)
        build_s = time.perf_counter() - t0
        eng = pkg.Engine(ℓ, chains=K, seed=2026, device=local_rank, chain_offset=chain_offset,
                         threads_per_chain=args.threads_per_chain, ctas_per_sm=args.ctas_per_sm)
        try:
            eng.random_position()
            eng.find_initial_stepsize()
            for st in wl["stages"]:
                eng.warmup_stage(st)
            steps, ms = 0, 0.0
            for i in range(args.warmup + args.steps):
                eng.mcmc_dev(n, draws.data_ptr(), stats.data_ptr(), logd.data_ptr())
                if i >= args.warmup:
                    steps += eng.last_total_steps(); ms += eng.last_kernel_ms()
            launches = eng.kernel_launches()
        finally:
            eng.close()
        return {"model": ℓ.model_name(), "header": "include/models/std_normal_user.h", "library": os.path.relpath(ℓ.library_path, ROOT),
                "value": steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / args.steps,
                "relative_to_shipped_family": (steps / ms) / (ref_steps / ref_ms), "same_trees": bool(steps == ref_steps),
                "gpu_launches": int(launches), "library_lookup_seconds": build_s,
                "what": "the timed C2 step with the log density given as a model header (user formulas behind the contract of "
                        "include/dhmc_models.h, position staged in shared memory once per gradient), same chains as the shipped "
                        "STD_NORMAL kernels; device-timed like `value`, run after the timed region"}
    except Exception as e:          # auxiliary leg: report, do not lose the bench line
        return {"error": "%s: %s" % (type(e).__name__, str(e)[:300])}


def c4_probe_leg(pkg, torch, dev, local_rank, sm_max_mhz, chains=4736, warm=(20, 40, 20), draws=4):
    """The tensor-core kernel of BASELINE.json configs[3] (logistic N=10 000, p=256, per-chain dense metric) inside the default
    run, at a REDUCED chain count (4 736 = 4 waves of 148 SMs x 8 chains per CTA instead of 32 768, so that the default bench
    stays short): search + TuningNUTS(20) + TuningNUTS(40, Symmetric) + TuningNUTS(20), then `draws` timed transitions with the
    adapted dense metric.  The full-size line is `bench.py --config C4` (profiles/r02_bench_c4.json).  Never fails the bench."""
    try:
        N, p = 10000, 256
        ℓ, _ = pkg.LogisticRegression.synthetic(N=N, p=p, seed=7)
        flops = 4.0 * N * p + 2 * 2.0 * p * p
        t0 = time.perf_counter()
        eng = pkg.Engine(ℓ, chains=chains, seed=2026, device=local_rank)
        try:
            eng.random_position()
            eng.find_initial_stepsize()
            w_steps, w_ms = 0, 0.0
            stages = [pkg.TuningNUTS(warm[0], pkg.DualAveraging()), pkg.TuningNUTS(warm[1], pkg.DualAveraging(), pkg.Symmetric),
                      pkg.TuningNUTS(warm[2], pkg.DualAveraging())]
            for st in stages:
                eng.warmup_stage(st)
                w_steps += eng.last_total_steps(); w_ms += eng.last_kernel_ms()
            post = torch.empty((chains, 1, p), dtype=torch.float64, device=dev)
            stats = torch.empty((chains, 1, 56), dtype=torch.uint8, device=dev)
            logd = torch.empty((chains, 1), dtype=torch.float64, device=dev)
            steps, ms = 0, 0.0
            for i in range(1 + draws):
                eng.mcmc_dev(1, post.data_ptr(), stats.data_ptr(), logd.data_ptr())
                if i >= 1:
                    steps += eng.last_total_steps(); ms += eng.last_kernel_ms()
            summary = eng.tree_summary_dev(stats.data_ptr(), 1, ebfmi=False)
        finally:
            eng.close()
        peak_tf = DMMA_FMA_PER_CLK_SM * 2 * 148 * sm_max_mhz * 1e6 / 1e12
        rate, wrate = steps / (ms * 1e-3), w_steps / (w_ms * 1e-3)
        return {"workload": "C4 kernel probe: logistic regression N=%d p=%d, %d chains (full size: 32768), per-chain dense metric adapted by "
                            "search + TuningNUTS(%d) + TuningNUTS(%d, Symmetric) + TuningNUTS(%d); likelihood and M^-1 p on DMMA.8x8x4"
                            % ((N, p, chains) + tuple(warm)),
                "value": rate, "unit": UNIT, "tflops_fp64": rate * flops / 1e12, "frac_of_dmma_peak": rate * flops / 1e12 / peak_tf,
                "warmup_value": wrate, "warmup_tflops_fp64": wrate * flops / 1e12, "dmma_peak_tflops": peak_tf,
                "leapfrogs_per_transition": steps / (draws * chains), "a_mean": summary["a_mean"],
                "depth_counts": summary["depth_counts"], "seconds": time.perf_counter() - t0,
                "what": "device-timed like `value`, run after the timed region of the default workload; 4736 of the 32768 C4 chains, so "
                        "tail effects of the last wave weigh more than at full size"}
    except Exception as e:
        return {"error": "%s: %s" % (type(e).__name__, str(e)[:300])}


def c3_probe_leg(pkg, torch, dev, local_rank, chains=262144, draws=10):
    """BASELINE.json configs[2] at FULL size inside the default run: Neal's funnel D=10, 262 144 chains, the default warm-up
    (900 transitions, ragged tree depths), then `draws` timed transitions.  Same code as `bench.py --config C3`
    (profiles/r02_bench_c3.json).  Never fails the bench."""
    try:
        t0 = time.perf_counter()
        eng = pkg.Engine(pkg.Funnel(10), chains=chains, seed=2026, device=local_rank)
        try:
            eng.random_position()
            eng.find_initial_stepsize()
            w_steps, w_ms = 0, 0.0
            for st in list(pkg.default_warmup_stages())[1:]:
                eng.warmup_stage(st)
                w_steps += eng.last_total_steps(); w_ms += eng.last_kernel_ms()
            post = torch.empty((chains, draws, 10), dtype=torch.float64, device=dev)
            stats = torch.empty((chains, draws, 56), dtype=torch.uint8, device=dev)
            logd = torch.empty((chains, draws), dtype=torch.float64, device=dev)
            steps, ms = 0, 0.0
            for i in range(1 + 3):
                eng.mcmc_dev(draws, post.data_ptr(), stats.data_ptr(), logd.data_ptr())
                if i >= 1:
                    steps += eng.last_total_steps(); ms += eng.last_kernel_ms()
            summary = eng.tree_summary_dev(stats.data_ptr(), draws, ebfmi=False)
        finally:
            eng.close()
        return {"workload": "C3: Neal's funnel D=10, %d chains, default_warmup_stages() (900 transitions), %d draws per timed launch" % (chains, draws),
                "value": steps / (ms * 1e-3), "unit": UNIT, "warmup_value": w_steps / (w_ms * 1e-3), "warmup_kernel_seconds": w_ms * 1e-3,
                "leapfrogs_per_transition": steps / (3 * draws * chains), "a_mean": summary["a_mean"],
                "termination_counts": summary["termination_counts"], "depth_counts": summary["depth_counts"],
                "seconds": time.perf_counter() - t0,
                "what": "device-timed like `value`, run after the timed region of the default workload; latency / divergence-bound "
                        "(480 B of state per leapfrog step), so no HBM fraction is quoted"}
    except Exception as e:
        return {"error": "%s: %s" % (type(e).__name__, str(e)[:300])}


DUMP_BYTES = 60 << 20


def dump_outputs(out_dir, draws, stats, logd, stats_dtype):
    """What the last timed step handed its caller, as float64 .npy files: posterior_matrix [m, n, D], logdensities [m, n]
    and one tree_statistics_<field> [m, n] per field, for m chains: all of them, or a fixed seeded sample when all would
    exceed DUMP_BYTES; chains.npy holds their indices."""
    import torch
    K, n, D = draws.shape
    m = min(K, max(1, DUMP_BYTES // (8 * (n * (D + 8) + 1))))
    idx = np.arange(K) if m == K else np.sort(np.random.default_rng(0).choice(K, m, replace=False))
    sel = torch.from_numpy(idx).to(draws.device)
    st = stats.index_select(0, sel).cpu().numpy().view(stats_dtype)[..., 0]
    arrays = {"chains": idx, "posterior_matrix": draws.index_select(0, sel).cpu().numpy(),
              "logdensities": logd.index_select(0, sel).cpu().numpy()}
    for f in ("pi", "depth", "left", "right", "acceptance_rate", "steps", "directions"):
        arrays["tree_statistics_" + f] = st[f]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="C2", choices=["C2", "C3", "C4", "C5"])
    ap.add_argument("--dim", type=int, default=0)
    ap.add_argument("--chains", type=int, default=0, help="chains per GPU (0: the configuration's own)")
    ap.add_argument("--draws-per-step", type=int, default=0)
    ap.add_argument("--adapt-steps", type=int, default=60)
    ap.add_argument("--c4-warm", type=int, nargs=3, default=[20, 40, 20])
    ap.add_argument("--threads-per-chain", type=int, default=0)
    ap.add_argument("--ctas-per-sm", type=int, default=0)
    ap.add_argument("--ref-eps", type=float, default=0.25)
    ap.add_argument("--ref-seconds", type=float, default=1.2)
    ap.add_argument("--cpu-baseline-seconds", type=float, default=4.0)
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step (rank 0's chains) to DIR/<name>.npy, at most 64 MB")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    # stdout carries exactly one JSON line: anything native code prints to fd 1 (NCCL's INFO lines when the caller sets
    # NCCL_DEBUG — we do not touch it) is routed to stderr, where the driver can still read it
    json_fd = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(os.dup(2), "w")

    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py --impl b200 needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    numa = None if os.environ.get("DHMC_BENCH_NO_BIND") else bind_to_gpu_numa_node(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    pkg = entry.load_package()
    wl = make_workload(pkg, args.config, args)
    D, n = wl["dim"], wl["draws"]
    dev = torch.device("cuda", local_rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- setup (untimed) ----------------
    chain_offset, K = pkg.parallel.shard(world * wl["chains"], world, rank)     # weak scaling: K chains per GPU
    eng = pkg.Engine(wl["model"], chains=K, seed=2026, device=local_rank, chain_offset=chain_offset,
                     threads_per_chain=args.threads_per_chain, ctas_per_sm=args.ctas_per_sm)
    T, EPL = eng.layout()
    t_setup = time.perf_counter()
    eng.random_position()
    eng.find_initial_stepsize()
    warm_steps, warm_ms = 0, 0.0
    for st in wl["stages"]:
        eng.warmup_stage(st)
        warm_steps += eng.last_total_steps(); warm_ms += eng.last_kernel_ms()
    barrier()
    setup_s = time.perf_counter() - t_setup
    eps = eng.get_state(("eps",))["eps"]
    draws = torch.empty((K, n, D), dtype=torch.float64, device=dev)      # [D, n, K] column-major
    stats = torch.empty((K, n, 56), dtype=torch.uint8, device=dev)
    logd = torch.empty((K, n), dtype=torch.float64, device=dev)

    def step_dev():
        eng.mcmc_dev(n, draws.data_ptr(), stats.data_ptr(), logd.data_ptr())
        return eng.last_total_steps(), eng.last_kernel_ms()

    sampler = ClockSampler(local_rank)
    sampler.start()                       # nvidia-smi needs ~0.2 s to start: sample from the warm-up steps (same workload) on
    for _ in range(args.warmup):
        step_dev()
    # ---------------- timed: device-resident ----------------
    launches0 = eng.kernel_launches()
    barrier()
    t0 = time.perf_counter()
    tot_steps, dev_ms = 0, 0.0
    for _ in range(args.steps):
        s, ms = step_dev()
        tot_steps += s
        dev_ms += ms
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    launches = eng.kernel_launches() - launches0
    if args.dump_outputs and rank == 0:      # before the legs below, which reuse these buffers
        dump_outputs(args.dump_outputs, draws, stats, logd, pkg._lib.tree_stats_dtype)
    summary = eng.tree_summary_dev(stats.data_ptr(), n, ebfmi=False) if rank == 0 else None
    q_typical = None if args.skip_e2e else eng.get_state(("q",))["q"]   # posterior draws: the e2e steps start from them

    # ---------------- roofline legs ----------------
    hbm_peak, sm_max_mhz, peak_kind = peaks()
    lf_ms = lf_bytes = None
    if args.config in ("C2", "C5"):
        # standalone streaming leapfrog kernel (HBM-bound): per-chain metric => 56·D B per step
        ms_l = []
        for _ in range(6):
            eng.leapfrog(1, 1)
            ms_l.append(eng.last_kernel_ms())
        lf_ms = float(np.median(ms_l[2:]))
        lf_bytes = 56 * D * K

    # ---------------- e2e: page-locked host buffers through the C ABI ----------------
    e2e = None
    if not args.skip_e2e:
        q_host = eng.host_alloc((K, D))
        post_host = eng.host_alloc((K, n, D))
        stats_host = eng.host_alloc((K, n), dtype=pkg._lib.tree_stats_dtype)
        logd_host = eng.host_alloc((K, n))
        q_host[...] = q_typical
        del q_typical
        out = dict(posterior_matrix=post_host, tree_statistics=stats_host, logdensities=logd_host)

        def step_e2e():
            ta = time.perf_counter()
            eng.mcmc_from(q_host, n, out=out)
            tb = time.perf_counter()
            r = eng.last_total_steps()
            if os.environ.get("DHMC_BENCH_TRACE"):
                print("[bench trace] mcmc_from %.2f ms, last_total_steps %.2f ms" % (1e3 * (tb - ta), 1e3 * (time.perf_counter() - tb)), file=sys.stderr)
            return r

        for _ in range(max(2, args.warmup - 1)):
            step_e2e()
        barrier()
        t1 = time.perf_counter()
        e_steps = 0
        for _ in range(args.steps):
            e_steps += step_e2e()
        t_loop = time.perf_counter() - t1
        barrier()
        e_wall = time.perf_counter() - t1
        if os.environ.get("DHMC_BENCH_TRACE"):
            print("[bench trace] e2e loop %.1f ms, with closing barrier %.1f ms" % (1e3 * t_loop, 1e3 * e_wall), file=sys.stderr)
        e2e = (e_steps, e_wall, K * D * 8, K * n * D * 8 + K * n * 56 + K * n * 8)

    # ---------------- the same step with the log density supplied as a USER model (after timing; C2, one GPU) ----------------
    user_leg = None
    if world == 1 and args.config == "C2" and not os.environ.get("DHMC_BENCH_NO_USER_MODEL"):
        user_leg = user_model_leg(pkg, wl, K, D, n, args, local_rank, chain_offset, draws, stats, logd,
                                  tot_steps, dev_ms)

    # ---------------- the other BASELINE.json configurations inside the default run (after timing; one GPU): configs[3] on its
    # own kernel at a reduced chain count, configs[2] at full size.  DHMC_BENCH_NO_PROBES=1 skips them.
    c4_leg = c3_leg = None
    if world == 1 and args.config == "C2" and not args.chains and not args.dim and not os.environ.get("DHMC_BENCH_NO_PROBES"):
        c4_leg = c4_probe_leg(pkg, torch, dev, local_rank, peaks()[1])
        c3_leg = c3_probe_leg(pkg, torch, dev, local_rank)

    # ---------------- multi-GPU: one NCCL all-gather of the draws (library communicator), after timing ----------------
    gather = None
    if world > 1:
        ids = [pkg.Engine.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        eng.comm_init(world, rank, ids[0])
        last = draws[:, n - 1, :].contiguous()
        recv = torch.empty((world * K, D), dtype=torch.float64, device=dev)
        torch.cuda.synchronize()
        ms_g = [eng.allgather_dev(last.data_ptr(), recv.data_ptr(), K * D) for _ in range(4)]   # first call warms the communicator
        assert torch.equal(recv[rank * K:(rank + 1) * K], last)
        gather = (ms_g[0], float(np.min(ms_g[1:])))

    # ---------------- reduce over ranks ----------------
    loc = torch.tensor([dev_ms, wall, float(tot_steps), float(launches), lf_ms or 0.0,
                        e2e[1] if e2e else 0.0, float(e2e[0]) if e2e else 0.0,
                        gather[1] if gather else 0.0, warm_ms, float(warm_steps)], dtype=torch.float64, device=dev)
    mx, sm = loc.clone(), loc.clone()
    if world > 1:
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
    dev_ms_max, wall_max = mx[0].item(), mx[1].item()
    steps_all = sm[2].item()
    value = steps_all / (dev_ms_max * 1e-3)

    if rank == 0:
        ms_per_launch = dev_ms / args.steps
        steps_per_launch = tot_steps / args.steps
        packed = args.config == "C4"
        kernel = ("k_nuts<logistic, 8 chains per CTA, tensor-core likelihood + mat-vec>" if packed
                  else "k_nuts (whole NUTS transition, chain state resident on chip)")
        if wl["flops_per_lf"]:
            peak_tf = DMMA_FMA_PER_CLK_SM * 2 * 148 * sm_max_mhz * 1e6 / 1e12
            ach = steps_per_launch * wl["flops_per_lf"] / (ms_per_launch * 1e-3) / 1e12
            traffic, traffic_src = None, None
            try:   # the ncu capture ran a smaller batch; the traffic is the per-chain metric stream, i.e. proportional to the steps
                tr = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))["c4"]
                per_ms = (tr["dram_bytes_read"] + tr["dram_bytes_write"]) / tr["duration_ms"]
                traffic = per_ms * ms_per_launch
                traffic_src = ("scaled by launch duration from the committed ncu --set full capture at %d chains (profiles/r02_traffic.json: "
                               "%.0f GB in %.0f ms = %.2f TB/s, the per-chain dense metrics), not measured in this run"
                               % (tr["chains"], (tr["dram_bytes_read"] + tr["dram_bytes_write"]) / 1e9, tr["duration_ms"], per_ms / 1e9))
            except Exception:
                pass
            roof = {"bound": "tensor", "kernel": kernel, "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s",
                    "frac": ach / peak_tf, "traffic": traffic, "traffic_source": traffic_src,
                    "peak_kind": "FP64 DMMA rate measured by benchmarks/c4_probes.cu (64 FMA/clk/SM = the DFMA rate) x 148 SMs x "
                                 "%.0f MHz; MEASURED_PEAKS.json holds no FP64 figure" % sm_max_mhz,
                    "algorithmic_flops_per_launch": steps_per_launch * wl["flops_per_lf"],
                    "flops_per_leapfrog": wl["flops_per_lf"]}
            # the per-chain dense metric is a GEMV stream from HBM: 2 mat-vecs per leapfrog, each over the chain's padded
            # [D'][XS] matrix (D' = 32·⌈D/32⌉, XS = the bank-conflict-free pitch): report it against the HBM peak too
            xs_pad = ((D + 7) // 8) * 8
            while xs_pad % 16 != 4:
                xs_pad += 1
            gemv_bytes = 2 * ((D + 31) // 32 * 32) * xs_pad * 8
            gbs = steps_per_launch * gemv_bytes / (ms_per_launch * 1e-3) / 1e9
            roof["metric_gemv_stream"] = {"bytes_per_leapfrog": gemv_bytes, "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / hbm_peak,
                                          "what": "M^-1 p with the reference's PER-CHAIN metric: a GEMV per chain on DMMA.8x8x4 (the MMA's "
                                                  "n-dimension carries one vector); DHMC_METRIC_SYMMETRIC_POOLED turns it into a GEMM"}
        else:
            ach = steps_per_launch * wl["bytes_per_lf"] / (ms_per_launch * 1e-3) / 1e9
            traffic, traffic_src = None, None
            try:   # DRAM bytes per launch from the committed ncu --set full capture of this same command
                tr = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))["k_nuts"]
                if args.config == "C2" and (tr["dim"], tr["chains"], tr["draws_per_step"]) == (D, K, n):
                    traffic = tr["dram_bytes_read"] + tr["dram_bytes_write"]
                    traffic_src = "committed ncu --set full capture of this same command (profiles/r02_traffic.json), not measured in this run"
            except Exception:
                pass
            roof = {"bound": "hbm", "kernel": kernel, "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                    "frac": ach / hbm_peak, "peak_kind": peak_kind, "traffic": traffic, "traffic_source": traffic_src,
                    "achieved_is": "HBM-EQUIVALENT: leapfrog steps per launch x %d B (algorithmic bytes, SURVEY 8d) / launch time; the "
                                   "kernel keeps q, p, grad on chip across the tree, so this is not DRAM bandwidth" % wl["bytes_per_lf"],
                    "dram_frac": (traffic / (ms_per_launch * 1e-3) / 1e9 / hbm_peak) if traffic else None,
                    "algorithmic_bytes_per_launch": steps_per_launch * wl["bytes_per_lf"]}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{args.config}: {wl['label']}; {K} chains per GPU, NUTS (max_depth 10), FP64",
                       "dim": D, "chains_per_gpu": K, "draws_per_step": n, "threads_per_chain": T,
                       "elems_per_thread": EPL, "parallelism": f"chains sharded x{world}, no data-path collective",
                       "l2": "state + outputs per step = %.2f GB > 126 MB L2" % ((3 + n) * K * D * 8 / 1e9),
                       "setup": wl["warm"], "setup_seconds": setup_s,
                       "warmup_leapfrog_steps_per_sec": (sm[9].item() / (mx[8].item() * 1e-3)) if mx[8].item() > 0 else None,
                       "mean_eps": float(np.mean(eps)), "leapfrogs_per_transition": tot_steps / (args.steps * n * K),
                       "numa_node": numa},
            "draws_per_sec": world * K * n * args.steps / (dev_ms_max * 1e-3),
            "wall_ms_per_step": 1e3 * wall_max / args.steps,
            "gpu_launches": int(sm[3].item()),
            "clocks": clocks,
            "roofline": roof,
            "tree_summary": {k: summary[k] for k in ("a_mean", "termination_counts", "depth_counts")} if summary else None,
        }
        try:
            rc = json.load(open(os.path.join(ROOT, "profiles", "r02_roofline_compute.json")))[args.config]
            line["roofline_compute"] = rc
        except Exception:
            pass
        if lf_ms:
            line["roofline_leapfrog_stream"] = {"bound": "hbm", "kernel": "k_leapfrog (one leapfrog step per launch, HBM streaming)",
                                                "achieved": lf_bytes / (lf_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                                "frac": lf_bytes / (lf_ms * 1e-3) / 1e9 / hbm_peak, "peak_kind": peak_kind,
                                                "bytes_per_launch": lf_bytes, "ms": lf_ms}
        if e2e:
            line["e2e"] = {"value": sm[6].item() / mx[5].item(), "unit": UNIT,
                           "h2d_bytes_per_step": e2e[2], "d2h_bytes_per_step": e2e[3],
                           "how": "dhmc_mcmc_from with page-locked NUMA-local host buffers (node %s): positions uploaded, draws / statistics / "
                                  "log densities downloaded, both pipelined by chain chunks against the sampling of the next chunk (draws "
                                  "that do not fit in HBM would be written by the kernel directly)" % numa}
        if user_leg:
            line["user_model"] = user_leg
        if c4_leg:
            line["c4_probe"] = c4_leg
        if c3_leg:
            line["c3_probe"] = c3_leg
        if gather:
            bw = K * D * 8 * (world - 1) / (mx[7].item() * 1e-3) / 1e9
            line["allgather"] = {"ms": mx[7].item(), "first_call_ms": gather[0], "bytes_per_rank": K * D * 8,
                                 "bus_gbs": bw, "via": "dhmc_allgather_dev (library NCCL communicator)",
                                 "what": "last draw of every chain, one ncclAllGather after sampling; best of 3 after a warm-up call"}
        if world == 1:
            po = entry.load_oracle()
            fam, params = oracle_family(po, pkg, wl)
            eps_med = float(np.median(eps))
            r = cpu_arm(po, fam, params, D, T, eps_med, args.cpu_baseline_seconds, reps=3)
            line["cpu_baseline"] = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                                    "per_core": r["value"] / r["cores"], "cpu_model": cpu_model(), "rates": r["rates"],
                                    "sample": f"{r['cores']} chains x {r['draws']} draws x 3 repetitions at D={D}, eps={eps_med:.4f} "
                                              f"(median adapted), identity metric, oracle port, one chain per pinned thread "
                                              f"({r['cores']} usable cores; cgroup quota {r['quota']}); median rate"}
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
