#!/usr/bin/env python
"""Headline benchmark: timesteps/sec of 3-D Rayleigh-Benard (Fourier x Fourier x Chebyshev, RK222, fp64).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--size 256] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one full solver.step(dt): 2 IMEX stages, each = RHS evaluation (15 backward + 4 forward 3-D
transforms and the fused products), template mat-vecs, RHS combination + per-pencil LU solves, scatter.
`value` times K steps with the state resident in HBM (CUDA events, barrier + synchronize both sides, max over
ranks); `e2e` times the same K steps through the public API with the state uploaded from pinned host memory and
read back every step.  Before anything is timed a parity gate steps a tall (16 x 16 x N) problem on the same ranks against
the CPU oracle.  `--impl reference` times the UNMODIFIED reference (oracle/_ref, oracle/ref_bench.py) on a bounded sample
of the workload with all host cores (the oracle port, oracle/cpu_bench.py, if oracle/_ref was not built).
"""
import argparse, json, os, subprocess, sys, threading, time, pathlib
import numpy as np

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "timesteps/sec 3D Rayleigh-Benard 256^3 fp64"      # --size N replaces 256 (north_star: 256^3 and 512^3)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--dim", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the coefficient arrays p, b, u as DIR/<name>.npy (float64; arrays over "
                         f"{DUMP_MAX_ELEMS} elements as a fixed seeded sample of that many entries of the flattened array)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the arrays of the GPU path; --impl reference times a sample of the workload only")
    return args


DUMP_MAX_ELEMS = 1 << 21          # 16 MB of float64 per array: p, b, u stay under 64 MB together


def dump_outputs(pb, directory):
    """Write what a caller of solver.step receives -- the coefficient data field['c'] of p, b, u -- to directory/<name>.npy.
    Read from the fields' device tensors (the same memory in the same order as field['c']) without moving them to the host,
    so that the steps after the dump run as they would without it.  The sample indices depend only on the array size."""
    import torch
    out = pathlib.Path(directory)
    out.mkdir(parents=True, exist_ok=True)
    for k, name in enumerate(("p", "b", "u")):
        f = pb[name]
        if f.layout != 'c':
            raise RuntimeError(f"{name} is not in coefficient space after the step")
        flat = f.device_data().reshape(-1)
        if flat.numel() <= DUMP_MAX_ELEMS:
            arr = flat.cpu().numpy().reshape(f.local_shape('c', f.scales))
        else:
            idx = np.sort(np.random.default_rng(1000 + k).choice(flat.numel(), DUMP_MAX_ELEMS, replace=False))
            arr = flat[torch.from_numpy(idx).to(flat.device)].cpu().numpy()
        np.save(out / f"{name}.npy", np.ascontiguousarray(arr, dtype=np.float64))


def workload(args):
    N = args.size
    return dict(workload=f"3-D Rayleigh-Benard Fourier x Fourier x Chebyshev {N}^3, dealias 3/2 ({int(1.5*N)}^3 grid), "
                         f"Ra=1e6 Pr=1, RK222, fixed dt, seed-42 initial condition (SURVEY.md Appendix C)",
                N=N, dim=args.dim, timestepper="RK222", dt=1e-2 * 64.0 / N,
                l2_policy="working set (state + factors, tens of GB) exceeds the 126 MB L2 every step; no explicit flush needed")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(smax) if smax else None,
                    reasons=sorted(reasons), samples=len(sm))


def cpu_arm(args, cfg, warmup, steps, max_pencils=256):
    """CPU arm on this host: the UNMODIFIED reference (oracle/_ref, oracle/ref_bench.py) when build() made it,
    else the oracle port (oracle/cpu_bench.py).  Returns (value, cpu_baseline dict, extra)."""
    from oracle import ref_bench
    if args.dim == 3 and ref_bench.available() and not os.environ.get("DB_BENCH_PORT"):
        r = ref_bench.run(N=args.size, dt=cfg['dt'], warmup=warmup, steps=steps, max_pencils=max_pencils)
        cb = dict(value=r['steps_per_sec'], unit="steps/s", cores=r['cores'], kind="reference", sample=r['sample'],
                  spread=r['spread'], per_step=r['steps_per_sec_list'], sample_step_seconds=r['sample_step_seconds'],
                  setup_seconds=r['setup_seconds'])
        return r['steps_per_sec'], cb
    from oracle import cpu_bench
    cores = os.cpu_count() or 1
    slab = 16 if args.size >= 128 else 8
    info = cpu_bench.sampled_step(dim=args.dim, N=args.size, dt=cfg['dt'], cores=cores, slab=min(slab, args.size),
                                  n_pencils=2 * cores, reps=warmup + steps)
    vals = info['steps_per_sec_list'][warmup:]
    v = float(np.median(vals))
    return v, dict(value=v, unit="steps/s", cores=info['cores'], kind="port", sample=info['sample'])


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path on the box's host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = workload(args)
    # bounded: the sample's set-up (per-pencil matrix assembly + SuperLU factorisations, untimed as in the reference's own
    # warm-up) dominates the wall time; at most 2 warm-up and 12 timed sample steps keep the arm within a few minutes
    n_warm = max(1, min(args.warmup, 2))
    n_runs = max(3, min(args.steps, 12))
    v, cb = cpu_arm(args, cfg, n_warm, n_runs)
    line = dict(impl="reference", metric=METRIC, value=v, unit="steps/s", n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 / v, higher_is_better=True, scaling="strong", vs_baseline=None, dtype="f64", data="synthetic",
                config=dict(cfg, timed_sample_steps=n_runs, sample_warmup=n_warm), cpu_baseline=cb,
                e2e=dict(value=v, unit="steps/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0,
                note=("value = whole-256^3-step throughput of the host derived from a bounded sample (see cpu_baseline.sample): "
                      "ms_per_step is 1000 / value, not the wall time of a sample step (cpu_baseline.sample_step_seconds)"))
    print(json.dumps(line))


def parity_gate(args, world, rank):
    """Correctness gate in front of the timing (BASELINE.md section 3): a TALL problem -- the benchmark's Nz, 16 x 16 horizontal
    modes (the benchmark's pencil systems, 1/256 of them), distributed over the same ranks -- stepped 2 RK222 steps on the
    GPU(s) against the CPU oracle on rank 0.  Returns dict(max_rel, ok, ...)."""
    import torch
    import torch.distributed as dist
    import dedalus_b200 as d3
    from dedalus_b200 import examples
    N = args.size
    Nh = max(16, 2 * world)
    dt = 1e-2 * 64.0 / N
    t0 = time.time()
    pb = examples.rayleigh_benard(dim=args.dim, Nh=Nh, Nz=N, Rayleigh=1e6, mesh=(world,) if world > 1 else None)
    solver = pb['problem'].build_solver(d3.RK222)
    examples.rayleigh_benard_initial_condition(pb['b'], pb['bases'], pb['Lz'])
    u = pb['u']
    u.fill_random('g', seed=7, distribution='normal', scale=1.0)
    uc = np.array(u['c']); uc[..., N // 2:] = 0; u['c'] = uc
    b0, u0 = np.array(pb['b']['c']), np.array(pb['u']['c'])
    steps = 2
    for _ in range(steps):
        solver.step(dt)
    got = {n: np.array(pb[n]['c']) for n in ("p", "b", "u")}
    verify = float(solver.bset.last_verify)
    blocked = world > 1 and solver.rhs_plan._blocked_bwd_ok() and solver.rhs_plan._blocked_fwd_ok()
    if world > 1:
        # local coefficient blocks (axis 0 of the horizontal modes is block-distributed) -> rank 0
        def gather(a, axis):
            t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
            parts = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(parts, t)
            return np.concatenate([x.cpu().numpy() for x in parts], axis=axis)
        b0 = gather(b0, 0); u0 = gather(u0, 1)
        got = {n: gather(a, 1 if n == "u" else 0) for n, a in got.items()}
    res = None
    if rank == 0:
        from oracle import rb_oracle
        ref = rb_oracle.run(dim=args.dim, Nh=Nh, Nz=N, Ra=1e6, b0_c=b0, steps=steps, dt=dt, u0_c=u0)
        rel = {n: float(np.abs(got[n] - ref[n]).max() / np.abs(ref[n]).max()) for n in got}
        ok = all(np.allclose(got[n], ref[n], rtol=1e-8, atol=(1e-10 * np.abs(ref[n]).max() if n == "p" else 1e-12)) for n in got)
        res = dict(ok=bool(ok), max_rel=max(rel.values()), rel=rel, shape=[Nh, Nh, N], steps=steps, ranks=world,
                   blocked_transposes=bool(blocked),
                   factor_backward_error=verify, seconds=time.time() - t0,
                   what="GPU state vs CPU oracle (oracle/rb_oracle.py, pinned to the reference fixtures) after 2 RK222 steps, O(1) velocity; "
                        "np.allclose(rtol=1e-8, atol=1e-12; p: atol=1e-10 max|p|)")
    del solver, pb
    torch.cuda.empty_cache()
    return res


def main():
    global METRIC
    args = parse()
    METRIC = METRIC.replace("256^3", f"{args.size}^3")
    if args.impl == "reference":
        return run_reference(args)
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:
        sys.exit("--dump-outputs writes the arrays of a single-process run (--gpus 1)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import dedalus_b200 as d3
    from dedalus_b200 import examples
    from dedalus_b200.lib import get_lib
    cfg = workload(args)
    N, dt = args.size, cfg['dt']
    def gate():
        """Parity gate on all ranks; every rank learns the verdict (rank 0 holds the comparison)."""
        res = parity_gate(args, world, rank)
        flag = torch.tensor([1.0 if (res is None or res['ok']) else 0.0], device='cuda')
        if world > 1:
            dist.broadcast(flag, src=0)
        return res, bool(flag.item() == 1.0)

    parity, parity_ok = (None, True) if args.no_parity else gate()
    if not parity_ok and world > 1 and os.environ.get("DB_PEER_TRANSPOSE", "1") != "0":
        # safety net: the transposes-as-peer-stores path is measured at 2 and 4 GPUs; if it ever fails the gate, time the NCCL
        # all-to-all path instead (and say so in the JSON line) rather than time nothing
        os.environ["DB_PEER_TRANSPOSE"] = "0"
        first = parity
        parity, parity_ok = gate()
        if rank == 0 and parity is not None:
            parity['peer_transposes_failed_gate'] = first
    if not parity_ok:
        if rank == 0:
            print(json.dumps(dict(metric=METRIC, value=None, unit="steps/s", n_gpus=world, parity=parity,
                                  error="parity gate failed: the GPU path does not reproduce the oracle; nothing was timed")))
        if world > 1:
            dist.destroy_process_group()
        sys.exit(3)
    t_setup = time.time()
    pb = examples.rayleigh_benard(dim=args.dim, Nh=N, Nz=N, Rayleigh=1e6, mesh=(world,) if world > 1 else None)
    solver = pb['problem'].build_solver(d3.RK222)
    examples.rayleigh_benard_initial_condition(pb['b'], pb['bases'], pb['Lz'])
    lib = get_lib()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        solver.step(dt)
    barrier()
    setup_s = time.time() - t_setup
    # ---- timed region: K device-resident steps, per-launch events recorded for the roofline accounting
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    solver.prof = []
    l0 = lib.launches
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        solver.step(dt)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = lib.launches - l0
    clocks = sampler.stop() if rank == 0 else None
    prof = solver.prof
    solver.prof = None
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device='cuda')
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = args.steps / (ms * 1e-3)
    if args.dump_outputs:
        dump_outputs(pb, args.dump_outputs)
    # ---- state checksum after the timed steps (identical problem and step count at every N: the values must agree across
    #      --gpus 1/2/4/8 runs with the same --steps/--warmup; the transposes are pure permutations)
    chk = torch.stack([(v.double() ** 2).sum() for v in solver.state_views[:3]])
    if world > 1:
        dist.all_reduce(chk)
    checksum = dict(sum_sq=dict(zip(("p", "b", "u"), [float(x) for x in chk.cpu()])), steps_taken=int(solver.iteration))
    try:
        gold = json.load(open(ROOT / "tests" / "golden" / "bench_checksums.json"))
        key = f"{args.dim}d_{N}_{solver.iteration}"
        if key in gold:
            ref = gold[key]
            checksum['golden'] = ref
            checksum['matches_single_gpu'] = bool(all(abs(checksum['sum_sq'][k] - ref[k]) <= 1e-9 * abs(ref[k]) + 1e-300 for k in ref))
    except Exception:
        pass
    # ---- per-kernel accounting
    agg = {}
    for name, a, b, nbytes in prof:
        d = agg.setdefault(name, dict(ms=0.0, bytes=0, launches=0))
        d['ms'] += a.elapsed_time(b); d['bytes'] += nbytes; d['launches'] += 1
    total_kernel_ms = sum(d['ms'] for d in agg.values()) or 1.0
    kernels = {k: dict(ms_per_step=d['ms'] / args.steps, launches_per_step=d['launches'] / args.steps,
                       gbps=d['bytes'] / (d['ms'] * 1e-3) / 1e9 if d['ms'] > 0 else None,
                       share=d['ms'] / total_kernel_ms) for k, d in sorted(agg.items(), key=lambda kv: -kv[1]['ms'])}
    peaks = {}
    try:
        peaks = json.load(open(ROOT / "MEASURED_PEAKS.json"))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    dom = next(iter(kernels)) if kernels else None
    roofline = None
    if dom:
        d = agg[dom]
        ach = d['bytes'] / (d['ms'] * 1e-3) / 1e9
        roofline = dict(bound="hbm", kernel=dom, achieved=ach, peak=peak, unit="GB/s", frac=ach / peak,
                        peak_source="MEASURED_PEAKS.json hbm_gbs (sustained copy)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)",
                        algorithmic_bytes_per_launch=d['bytes'] / d['launches'], avg_launch_ms=d['ms'] / d['launches'],
                        traffic=None)
        # measured DRAM bytes per launch of this kernel class from the committed ncu capture of the same workload
        try:
            tr = json.load(open(ROOT / "profiles" / "ncu_traffic.json"))
            if world == 1 and N == 256 and args.dim == 3 and dom in tr.get("classes", {}):
                roofline['traffic'] = tr["classes"][dom]["dram_bytes_per_launch"]
                roofline['traffic_source'] = tr["classes"][dom]["capture"] + " (" + tr["how"] + ")"
        except Exception:
            pass
    # ---- end-to-end: state uploaded from pinned host memory and read back every step, through solver.step()
    e2e = None
    errors = {}
    if not args.no_e2e:
      try:
            nst = solver.state_t.numel()
            h_in = torch.empty(nst, dtype=torch.float64).pin_memory()
            h_out = torch.empty(nst, dtype=torch.float64).pin_memory()
            h_in.copy_(solver.state_t)
            barrier()
            f0 = torch.cuda.Event(enable_timing=True); f1 = torch.cuda.Event(enable_timing=True)
            ksteps = args.steps          # the same K steps as the device-resident arm
            # Every step uploads its input state from pinned host memory and downloads its result; the copies run on two
            # copy streams (PCIe is full duplex) so that step i+1's upload and step i-1's download overlap step i's kernels:
            # upload -> device staging buffer -> (D2D) state -> step -> (D2D) result staging -> download.
            main = torch.cuda.current_stream()
            s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
            d_in = [torch.empty_like(solver.state_t) for _ in range(2)]
            d_out = torch.empty_like(solver.state_t)
            in_ready = [torch.cuda.Event() for _ in range(2)]; in_free = [torch.cuda.Event() for _ in range(2)]
            out_ready, out_free = torch.cuda.Event(), torch.cuda.Event()
            torch.cuda.synchronize()
            f0.record(main)
            s_in.wait_event(f0); s_out.wait_event(f0)

            def upload(i):
                with torch.cuda.stream(s_in):
                    if i >= 2:
                        s_in.wait_event(in_free[i % 2])
                    d_in[i % 2].copy_(h_in, non_blocking=True)            # H2D: input of step i
                    in_ready[i % 2].record(s_in)

            upload(0)
            for i in range(ksteps):
                if i + 1 < ksteps:
                    upload(i + 1)
                main.wait_event(in_ready[i % 2])
                solver.state_t.copy_(d_in[i % 2])
                in_free[i % 2].record(main)
                solver.step(dt)
                if i > 0:
                    main.wait_event(out_free)
                d_out.copy_(solver.state_t)
                out_ready.record(main)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(out_ready)
                    h_out.copy_(d_out, non_blocking=True)                  # D2H: result of step i
                    out_free.record(s_out)
            main.wait_event(out_free)
            f1.record(main)
            barrier()
            ms2 = f0.elapsed_time(f1)
            if world > 1:
                t = torch.tensor([ms2], dtype=torch.float64, device='cuda')
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms2 = float(t.item())
            e2e = dict(value=ksteps / (ms2 * 1e-3), unit="steps/s", h2d_bytes_per_step=int(nst * 8 * world), d2h_bytes_per_step=int(nst * 8 * world),
                       path="solver.step(dt) with the coefficient state copied host->device from pinned memory before and device->host after every step; "
                            "the copies run on two copy streams and overlap the neighbouring steps' kernels (all inside the timed region)")
      except Exception as exc:        # the device-resident measurement above stands on its own: report it, and why this leg is absent
        e2e = None
        errors['e2e'] = repr(exc)
    # ---- CPU baseline (rank 0, N=1 only): the reference itself on the host cores, bounded sample
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            _, cpu = cpu_arm(args, cfg, 1, 4, max_pencils=64)      # short: the driver times the full arm separately (--impl reference)
        except Exception as exc:
            errors['cpu_baseline'] = repr(exc)
    if rank == 0:
        line = dict(metric=METRIC, value=value, unit="steps/s", n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3),
                    ms_per_step=ms / args.steps, higher_is_better=True, scaling="strong", vs_baseline=None, dtype="f64",
                    data="synthetic", config=dict(cfg, parallelism=f"pencil{world}" if world > 1 else "single", setup_seconds=setup_s,
                                                  pencil_systems=sum(b.S * b.R for b in solver.batches), factorisations=sum(b.S for b in solver.batches), total_modes=solver.total_modes),
                    clocks=clocks, e2e=e2e, gpu_launches=launches, roofline=roofline, kernels=kernels, cpu_baseline=cpu,
                    parity=parity, state_checksum=checksum, factor_backward_error=float(solver.bset.last_verify))
        if errors:
            line['errors'] = errors
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
