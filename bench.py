#!/usr/bin/env python
"""bench.py -- molecules/s of DiffLinker sampling (T=500 reverse steps) on B200, contract in the task statement.

A "step" is one full `sample_chain` of one synthetic batch (default workload cfg2_zinc: B=256, N=40, L=6, T=500),
i.e. 501 Dynamics.forward calls.  Arms:
  default           the native path.  `value`: inputs resident in HBM, timed with CUDA events, max over ranks.
                    `e2e`: the same through the public API from pinned HOST tensors (H2D + D2H inside the region).
  --impl reference  the reference algorithm's CPU implementation (oracle port; the Python reference cannot travel
                    to the GPU box) on the host cores, bounded sample per step.
Prints ONE JSON line (rank 0). `--dump-outputs DIR` also writes what the last timed step returned (see dump_outputs), so
that two builds can be compared output for output on identical seeded inputs.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="cfg2_zinc")
    ap.add_argument("--edge-impl", default="auto", choices=["auto", "simt", "tcgen05"])
    ap.add_argument("--T", type=int, default=None, help="override the number of reverse steps (debug only)")
    ap.add_argument("--coord-gain", type=float, default=None,
                    help="scale of coord_mlp.4 on top of the default init; default 100 (SURVEY 8c) for N <= 64, 1 above: "
                         "with 100 and hundreds of neighbours the random-weight dynamics blow up to |x| ~ 5e3 within steps")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: every rank samples its own batches (default); strong: ONE batch per step is split across the "
                         "ranks (distributed.sample_chain_sharded: same result as on one GPU)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="native arm: after the timed steps, write rank 0's results of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs applies to the native arm")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes each tensor as out_dir/<name>.npy in float32. Every workload's results fit the limit whole, so nothing is
    sampled: a larger total is refused rather than silently cut."""
    import numpy as np
    host = {name: t.detach().to(torch.float32).cpu().numpy() for name, t in arrays.items()}
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], bf16_tflops_sustained=d["bf16_tflops_sustained"],
                    source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md's clocks line, every 200 ms).
    The process is started BEFORE the warm-up steps -- NVML initialisation inside the timed region stalls command submission --
    and every sample carries nvidia-smi's own timestamp; `stop()` keeps the samples taken between `mark_begin()` and
    `mark_end()` (wall clock; both are called next to the CUDA events that bracket the timed steps)."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None
        self.t_begin = self.t_end = None

    def start(self):
        if shutil.which("nvidia-smi") is None or os.environ.get("BENCH_NO_CLOCKS"):      # the switch is for diagnosing the sampler itself
            return
        fd, self.path = tempfile.mkstemp(suffix=".csv")
        os.close(fd)
        self.out = open(self.path, "w")
        self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.gpu), "-lms", os.environ.get("BENCH_CLOCKS_MS", "200")],
                                     stdout=self.out, stderr=subprocess.DEVNULL)

    def mark_begin(self):
        self.t_begin = time.time()

    def mark_end(self):
        self.t_end = time.time()

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.out.close()
        import datetime
        sm, mx, reasons, n_all = [], [], set(), 0
        with open(self.path) as f:
            for line in f:
                parts = [p.strip() for p in line.split(",")]
                if len(parts) < 9:
                    continue
                try:
                    ts = datetime.datetime.strptime(parts[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    clk, cmax = float(parts[2]), float(parts[3])
                except ValueError:
                    continue
                n_all += 1
                if self.t_begin is not None and not (self.t_begin - 0.05 <= ts <= (self.t_end or time.time()) + 0.05):
                    continue
                sm.append(clk); mx.append(cmax)
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], parts[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        os.unlink(self.path)
        if not sm:
            return None
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm),
                "samples_outside_timed_region": n_all - len(sm)}


def cpu_reference_step(fwd, sample):
    """One bounded sample of the reference algorithm on the CPU: a single Dynamics.forward (egnn.py:374-447) over
    `sample['B']` molecules of the workload."""
    t0 = time.perf_counter()
    with torch.no_grad():
        fwd(sample["t"], sample["z"], sample["node_mask"], sample["linker_mask"], sample["edge_mask"], sample["context"])
    return time.perf_counter() - t0


def build_cpu_sample(spec, hp, nb):
    from difflinker_b200 import synthetic
    from difflinker_b200.batching import collate
    from difflinker_b200.egnn import Dynamics
    batch = collate(synthetic.make_items(spec, batch=nb))
    torch.manual_seed(0)
    dyn = Dynamics(in_node_nf=hp['in_node_nf'], n_dims=3, context_node_nf=hp['context_node_nf'], hidden_nf=128,
                   n_layers=hp['n_layers'], norm_constant=hp['norm_constant'], inv_sublayers=hp['inv_sublayers'],
                   normalization_factor=hp['normalization_factor'], graph_type='FC')
    synthetic.init_reference_like_weights(dyn)
    sd = {k: v.detach().clone() for k, v in dyn.state_dict().items()}
    g = torch.Generator().manual_seed(5)
    z = torch.cat([batch['positions'], batch['one_hot'] / 4], dim=2)
    z = z * batch['fragment_mask'] + torch.randn(z.shape, generator=g) * batch['linker_mask']
    return sd, dict(B=nb, t=torch.full((nb, 1), 0.5), z=z, node_mask=batch['atom_mask'],
                    linker_mask=batch['linker_mask'], edge_mask=batch['edge_mask'], context=batch['fragment_mask'])


def staged_reference_dynamics(hp, sd):
    """The UNMODIFIED reference `src.egnn.Dynamics` (staged by oracle/build_ref.py under oracle/_ref/), carrying the same
    weights as the oracle port's sample. None when the staging directory is absent."""
    root = os.path.join(os.path.dirname(os.path.abspath(__file__)), "oracle", "_ref")
    if not os.path.isfile(os.path.join(root, "src", "egnn.py")):
        return None
    if root not in sys.path:
        sys.path.insert(0, root)
    import importlib
    egnn = importlib.import_module("src.egnn")
    dyn = egnn.Dynamics(in_node_nf=hp['in_node_nf'], n_dims=3, context_node_nf=hp['context_node_nf'], hidden_nf=128,
                        n_layers=hp['n_layers'], norm_constant=hp['norm_constant'], inv_sublayers=hp['inv_sublayers'],
                        normalization_factor=hp['normalization_factor'])
    dyn.load_state_dict(sd, strict=True)
    return dyn.eval()


def cpu_reference_measure(spec, hp, steps, warmup):
    """Times Dynamics.forward on the host cores: the reference's own module when oracle/_ref/ is staged (kind "reference";
    its FC edge list is cached by the warm-up call, egnn.py:449-467), else the oracle port (kind "port"). torch's intra-op
    pool is slower with all 100+ hardware threads on these small ops than with a few dozen, so a quick sweep on a small
    sample picks the thread count the reference is best run with. Returns (s_per_forward, nb, threads, kind, s_port)."""
    from oracle import difflinker_oracle as orc
    cores = os.cpu_count() or 1
    ocfg = orc.OracleConfig(in_node_nf=hp['in_node_nf'], context_node_nf=hp['context_node_nf'], n_layers=hp['n_layers'],
                            inv_sublayers=hp['inv_sublayers'], norm_constant=hp['norm_constant'],
                            normalization_factor=hp['normalization_factor'])

    def port_fwd(sd):
        return lambda t, z, nm, lm, em, ctx: orc.dynamics_forward(sd, ocfg, t, z, nm, lm, em, ctx)

    sd_small, small = build_cpu_sample(spec, hp, min(spec.B, 8))
    ref_small = staged_reference_dynamics(hp, sd_small)
    fwd_small = ref_small.forward if ref_small is not None else port_fwd(sd_small)
    best_t, best = cores, None
    for th in sorted({min(cores, c) for c in (8, 16, 32, 64, cores)}):
        torch.set_num_threads(th)
        cpu_reference_step(fwd_small, small)
        dt = cpu_reference_step(fwd_small, small)
        if best is None or dt < best:
            best, best_t = dt, th
    torch.set_num_threads(best_t)
    nb = min(spec.B, 64)
    sd, sample = build_cpu_sample(spec, hp, nb)
    ref = staged_reference_dynamics(hp, sd)
    kind = "reference" if ref is not None else "port"
    fwd = ref.forward if ref is not None else port_fwd(sd)
    for _ in range(max(warmup, 1)):
        cpu_reference_step(fwd, sample)
    ts = [cpu_reference_step(fwd, sample) for _ in range(steps)]
    s_port = None
    if ref is not None:                                      # the port beside it, one call (for the record)
        cpu_reference_step(port_fwd(sd), sample)
        s_port = cpu_reference_step(port_fwd(sd), sample)
    return sum(ts) / len(ts), nb, best_t, kind, s_port


def run_reference_arm(args, spec, hp, rank, world):
    """CPU arm: rank 0 only. Each step = one Dynamics.forward over a bounded sample of the workload's molecules;
    molecules/s is extrapolated as B_sample / ((T+1) * s_per_forward) (BASELINE.md section 3)."""
    if rank != 0:
        return
    s_fwd, nb, cores, kind, s_port = cpu_reference_measure(spec, hp, args.steps, args.warmup)
    T = args.T or spec.T
    value = nb / ((T + 1) * s_fwd)
    sample_desc = f"{args.steps} Dynamics.forward calls over {nb} of {spec.B} molecules (N={spec.N}, L={spec.L}); x(T+1)={T + 1} extrapolated"
    line = {
        "impl": "reference", "metric": "molecules/sec (T=%d denoising)" % T, "value": value, "unit": "molecules/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * s_fwd,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": spec.name, "B": spec.B, "N": spec.N, "n_layers": spec.L, "T": T, "hidden_nf": 128},
        "cpu_baseline": {"value": value, "unit": "molecules/s", "cores": cores, "kind": kind, "sample": sample_desc,
                         "port_value": (nb / ((T + 1) * s_port)) if s_port else None},
        "e2e": {"value": value, "unit": "molecules/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    from difflinker_b200 import synthetic
    spec = synthetic.SPECS[args.workload]
    hp = synthetic.model_hparams(spec)
    if args.T is not None:
        hp['diffusion_steps'] = args.T

    if args.impl == "reference":
        run_reference_arm(args, spec, hp, rank, world)
        return

    import torch.distributed as dist
    from difflinker_b200 import DDPM, _native
    from difflinker_b200.batching import collate
    from difflinker_b200.distributed import broadcast_module_weights

    if not torch.cuda.is_available():
        raise SystemExit("bench.py (native arm) needs a B200; no CUDA device is visible")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    torch.manual_seed(0)
    coord_gain = args.coord_gain if args.coord_gain is not None else (100.0 if spec.N <= 64 else 1.0)
    ddpm = DDPM(**hp, edge_impl=args.edge_impl)
    synthetic.init_reference_like_weights(ddpm, coord_gain=coord_gain)
    ddpm = ddpm.to(dev)
    if world > 1:
        broadcast_module_weights(ddpm, src=0, device=dev)       # the only collective on the path
    edm = ddpm.edm
    T = edm.T
    lib = _native.load_library()

    # one distinct synthetic batch per (rank, step): weak scaling, seed = seed0 + batch id
    n_batches = args.warmup + args.steps
    host_batches = []
    for i in range(n_batches):
        data = collate(synthetic.make_items(spec, seed_offset=1 + rank * 1000 + i))
        for k, v in data.items():
            if torch.is_tensor(v):
                data[k] = v.pin_memory()
        host_batches.append(data)

    def to_device(data):
        return {k: (v.to(dev, non_blocking=True) if torch.is_tensor(v) else v) for k, v in data.items()}

    def resident_inputs(data):
        """What DDPM.sample_chain hands to EDM.sample_chain (lightning.py:405-452), precomputed on the device by the
        same code the public entry point runs (template batch, context columns, centred coordinates)."""
        from difflinker_b200.ddpm import sampler_inputs
        return sampler_inputs(ddpm, to_device(data))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------- kernel-resident arm: inputs in HBM, CUDA events --------------------------------------
    strong = args.scaling == "strong" and world > 1
    if strong:
        # every rank holds the SAME batches (seed without the rank term) and samples its slice of each
        from difflinker_b200.distributed import shard_range, slice_sampler_inputs
        host_batches = []
        for i in range(n_batches):
            data = collate(synthetic.make_items(spec, seed_offset=1 + i))
            host_batches.append({k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in data.items()})
        lo, hi = shard_range(spec.B, rank, world)
        resident = [slice_sampler_inputs(resident_inputs(b), lo, hi) for b in host_batches]
        for kw in resident:
            kw["batch_slice"] = (lo, spec.B)
    else:
        resident = [resident_inputs(b) for b in host_batches]
    torch.cuda.synchronize(dev)
    sampler = ClockSampler(local_rank)
    sampler.start()                                                      # before the warm-up: see ClockSampler
    l2_flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    for i in range(args.warmup):
        l2_flush.zero_()
        edm.sample_chain(**resident[i], keep_frames=1)
    eng = edm.dynamics.engine(local_rank)
    barrier()
    launches0 = lib.dl_launch_count(eng)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.mark_begin()
    ev0.record()
    loop_ms = []
    for i in range(args.steps):
        l2_flush.zero_()                                                 # larger than the 126 MB L2
        chain = edm.sample_chain(**resident[args.warmup + i], keep_frames=1)
        loop_ms.append(edm.last_loop_ms)
    ev1.record()
    barrier()
    sampler.mark_end()
    clocks = sampler.stop()
    launches = lib.dl_launch_count(eng) - launches0
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    mols = (1 if strong else world) * spec.B * args.steps
    value = mols / (ms_total * 1e-3)
    assert torch.isfinite(chain).all()

    # ---------------- end-to-end arm: public API from pinned host memory -----------------------------------
    e2e = None
    if not args.no_e2e:
        def e2e_step(data):
            d = to_device(data)                                          # H2D of this step's inputs
            if strong:
                from difflinker_b200.distributed import sample_chain_sharded
                ch, nm = sample_chain_sharded(ddpm, d, keep_frames=1)    # slices + one all_gather of the final frames
            else:
                ch, nm = ddpm.sample_chain(d, keep_frames=1)             # the call generate.py makes (generate.py:156)
            return ch.cpu(), nm.cpu()                                    # D2H of the step's result
        e2e_step(host_batches[0])
        barrier()
        t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
        wall0 = time.perf_counter()
        t0.record()
        for i in range(args.steps):
            l2_flush.zero_()
            ch, nm = e2e_step(host_batches[args.warmup + i])
        t1.record()
        barrier()
        wall_ms = (time.perf_counter() - wall0) * 1e3
        e2e_ms = max_over_ranks(max(t0.elapsed_time(t1), wall_ms))      # D2H is synchronous: wall covers host work
        h2d = sum(v.numel() * v.element_size() for v in host_batches[0].values() if torch.is_tensor(v))
        d2h = ch.numel() * ch.element_size() + nm.numel() * nm.element_size()
        e2e = {"value": mols / (e2e_ms * 1e-3), "unit": "molecules/s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / args.steps}

    if args.dump_outputs and rank == 0:
        # chain: EDM.sample_chain of the kernel-resident arm, (1,B,N,3+F); e2e_*: DDPM.sample_chain of the end-to-end arm
        outputs = {"chain": chain}
        if e2e is not None:
            outputs.update(e2e_chain=ch, e2e_node_mask=nm)
        dump_outputs(args.dump_outputs, outputs)

    # ---------------- roofline of the dominant kernel (GCL edge kernel) ------------------------------------
    peaks = measured_peaks()
    H = 128
    # algorithmic work of one forward, from the actual masks of the batch (ragged workloads included)
    hb = host_batches[args.warmup]
    n_b = hb['atom_mask'].reshape(spec.B, -1).sum(1).tolist()
    l_b = hb['linker_mask'].reshape(spec.B, -1).sum(1).tolist()
    if spec.pocket:
        e_b = synthetic.cutoff_edge_counts(hb, spec.graph_type)         # true edges of the cut-off graph, not n^2
    else:
        e_b = [(n * n, l * n) for n, l in zip(n_b, l_b)]
    edge_flops = sum((2 * H * H + 10 * H) * e for e, _ in e_b)           # GCL edge kernel: second Linear + first layer/mask/sum
    ms_gcl = float(lib.dl_time_edge_kernel(eng, 20))
    cut_stats = None
    if spec.pocket:
        import ctypes
        st4 = (ctypes.c_int64 * 4)()
        lib.dl_cut_graph_stats(eng, st4)
        cut_stats = {"records": st4[0], "tiles": st4[1], "edges": st4[2], "coord_records": st4[3]}
        if st4[2] > 0:                                                  # the graph the timed kernel actually walked
            edge_flops = (2 * H * H + 10 * H) * float(st4[2])
    fwd_ms = (sum(loop_ms) / len(loop_ms)) / (T + 1)
    flops_fwd = sum(synthetic.flops_alg(int(n), int(l), spec, e, ex) for n, l, (e, ex) in zip(n_b, l_b, e_b))
    bytes_fwd = spec.B * synthetic.bytes_alg(spec.N, spec)
    roofline = None
    if ms_gcl and ms_gcl > 0:
        ach = edge_flops / (ms_gcl * 1e-3) / 1e12
        traffic = None                                                  # DRAM bytes per launch from the committed ncu capture
        try:
            with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "ncu_traffic.json")) as f:
                traffic = json.load(f).get(spec.name, {}).get("edge_gcl")
        except OSError:
            pass
        roofline = {"bound": "tensor", "kernel": "edge_gcl", "achieved": ach, "peak": peaks["bf16_tflops"],
                    "unit": "TFLOP/s", "frac": ach / peaks["bf16_tflops"], "traffic": traffic,
                    "peak_source": peaks["source"], "kernel_ms": ms_gcl,
                    "kernel_share_of_step": ms_gcl * spec.L * spec.S / fwd_ms}
    forward = {"ms": fwd_ms, "flops_alg": flops_fwd, "bytes_alg": bytes_fwd,
               "compute_frac": flops_fwd / (fwd_ms * 1e-3) / 1e12 / peaks["bf16_tflops_sustained"],
               "hbm_frac": bytes_fwd / (fwd_ms * 1e-3) / 1e9 / peaks["hbm_gbs"]}

    # ---------------- parity of the benchmarked launch: one Dynamics.forward at the timed shape vs the oracle -------------
    parity = None
    if rank == 0:
        from oracle import difflinker_oracle as orc
        k = min(4, spec.B)
        hbp = host_batches[args.warmup]
        dbp = to_device(hbp)
        from difflinker_b200.ddpm import sampler_inputs
        kwp = sampler_inputs(ddpm, dbp)
        gp = torch.Generator().manual_seed(17)
        zp = torch.cat([kwp['x'].cpu(), kwp['h'].cpu() / 4], dim=2)
        zp = zp * kwp['fragment_mask'].cpu() + torch.randn(zp.shape, generator=gp) * kwp['linker_mask'].cpu()
        tp = torch.full((spec.B, 1), 0.4)
        with torch.no_grad():
            got = edm.dynamics(tp.to(dev), zp.to(dev), kwp['node_mask'], kwp['linker_mask'], kwp['edge_mask'], kwp['context']).cpu()
            ocfg = orc.OracleConfig(in_node_nf=hp['in_node_nf'], context_node_nf=hp['context_node_nf'], n_layers=hp['n_layers'],
                                    inv_sublayers=hp['inv_sublayers'], norm_constant=hp['norm_constant'],
                                    normalization_factor=hp['normalization_factor'], graph_type=hp['graph_type'])
            N = spec.N if not hasattr(kwp['x'], 'shape') else kwp['x'].shape[1]
            em = kwp['edge_mask'].cpu()
            em_k = em[:k * (em.shape[0] // spec.B)]
            sdp = {n: v.detach().cpu() for n, v in edm.dynamics.state_dict().items()}
            want = orc.dynamics_forward(sdp, ocfg, tp[:k], zp[:k], kwp['node_mask'].cpu()[:k], kwp['linker_mask'].cpu()[:k], em_k,
                                        kwp['context'].cpu()[:k])
        err = (got[:k] - want).abs().max().item() / max(want.abs().max().item(), 1e-30)
        parity = {"rel_err": err, "molecules": k, "of_batch": spec.B,
                  "what": "Dynamics.forward of the benchmarked (B,N,L) launch vs the oracle on the first molecules; tolerance 1e-4"}

    # ---------------- CPU baseline (oracle port of the reference algorithm), rank 0 at N=1 only -------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        s_fwd, nb, cores, kind, s_port = cpu_reference_measure(spec, hp, 3, 1)
        cpu = {"value": nb / ((T + 1) * s_fwd), "unit": "molecules/s", "cores": cores, "kind": kind,
               "sample": f"3 Dynamics.forward calls over {nb} of {spec.B} molecules ({cores} torch threads, best of a sweep), extrapolated x{T + 1}",
               "s_per_forward": s_fwd, "port_value": (nb / ((T + 1) * s_port)) if s_port else None}

    if rank == 0:
        line = {
            "metric": "molecules/sec (T=%d denoising)" % T, "value": value, "unit": "molecules/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps,
            "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": spec.name, "B": spec.B, "N": spec.N, "n_layers": spec.L, "T": T, "hidden_nf": 128,
                       "edge_impl": args.edge_impl, "coord_gain": coord_gain,
                       "noise": "drawn inside the kernels in the reference's torch.randn order (Philox4x32-10, dl_sample_chain_rng)",
                       "edges_per_launch": int(sum(e for e, _ in e_b)), "cut_graph_device_stats": cut_stats,
                       "l2": "flushed: a 256 MB buffer is written before every timed step (inside the timed region, ~0.05 ms); "
                             "every step also samples a fresh batch"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "forward": forward,
            "cpu_baseline": cpu, "loop_ms_device": loop_ms, "parity": parity,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
