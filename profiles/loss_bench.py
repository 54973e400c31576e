"""Throughput of the diffusion-loss evaluation (DDPM.validation_step -> EDM.forward -> dl_diffusion_loss) on one GPU.

For each shape: molecules/s of `DDPM.validation_step` over >= 50 batches (CUDA events around each call, after warm-up),
and, alternating with it in the same run, a bare `Dynamics.forward` of the same shape -- the loss step's one network call.
`native_ms` is the engine's own device time (CUDA events around its launches: q-sample, forward, loss kernel for the step;
the forward alone for the bare call), so `loss_kernels_overhead` = step native / forward native - 1 is what the q-sample and
loss kernels add. When oracle/_ref/ is staged (oracle/build_ref.py), the reference's own `src.edm.EDM.forward` is timed on
the host cores over a bounded sample. Prints one JSON line.
    python profiles/loss_bench.py [--steps 50] [--warmup 5] [--shapes cfg2_zinc,cfg2_zinc_L8,cfg3_geom,cfg4_pockets]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from difflinker_b200 import DDPM, _native, synthetic  # noqa: E402
from difflinker_b200.batching import collate  # noqa: E402

CPU_SAMPLE = {"cfg2_zinc": 8, "cfg2_zinc_L8": 8, "cfg3_geom": 8, "cfg4_pockets": 2}   # molecules in the reference's CPU sample


class MOADDataset(list):
    """Named like the reference's class: DDPM.forward builds the pocket context when train_dataset is one (lightning.py:165)."""


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = None
    return name, q or None


def timed(fn, stream):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    fn()
    b.record(stream)
    b.synchronize()
    return a.elapsed_time(b)


def reference_cpu(spec, hp, ddpm, n):
    """The reference's own EDM.forward on the host cores for `n` molecules (None without oracle/_ref/)."""
    root = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.isfile(os.path.join(root, "src", "edm.py")):
        return None
    if root not in sys.path:
        sys.path.insert(0, root)
    import importlib
    egnn, edm_mod = importlib.import_module("src.egnn"), importlib.import_module("src.edm")
    cls = egnn.DynamicsWithPockets if spec.pocket else egnn.Dynamics
    dyn = cls(in_node_nf=hp['in_node_nf'], n_dims=3, context_node_nf=hp['context_node_nf'], hidden_nf=128,
              n_layers=hp['n_layers'], norm_constant=hp['norm_constant'], inv_sublayers=hp['inv_sublayers'],
              normalization_factor=hp['normalization_factor'], graph_type=hp['graph_type'])
    ref = edm_mod.EDM(dynamics=dyn, in_node_nf=hp['in_node_nf'], n_dims=3, timesteps=hp['diffusion_steps'],
                      noise_schedule=hp['diffusion_noise_schedule'], noise_precision=hp['diffusion_noise_precision'],
                      loss_type=hp['diffusion_loss_type'], norm_values=hp['normalize_factors'])
    ref.load_state_dict({k: v.detach().cpu() for k, v in ddpm.edm.state_dict().items()}, strict=True)
    ref.eval()
    data = collate(synthetic.make_items(spec, batch=n))
    if spec.pocket:
        fo = data['fragment_only_mask']
        ctx, com = torch.cat([fo, data['fragment_mask'] - fo], dim=-1), fo
    else:
        ctx, com = data['fragment_mask'], data['fragment_mask']
    x = data['positions'] - (torch.sum(data['positions'] * com, 1, keepdim=True) / com.sum(1, keepdim=True)) * data['atom_mask']
    kw = dict(x=x, h=data['one_hot'], node_mask=data['atom_mask'], fragment_mask=data['fragment_mask'],
              linker_mask=data['linker_mask'], edge_mask=data['edge_mask'], context=ctx)
    ts = []
    with torch.no_grad():
        for _ in range(2):
            t0 = time.perf_counter()
            ref.forward(**kw)
            ts.append(time.perf_counter() - t0)
    s = min(ts)
    return dict(kind="reference", molecules=n, seconds=s, molecules_per_s=n / s, threads=torch.get_num_threads())


def run_shape(name, steps, warmup):
    spec = synthetic.SPECS[name]
    hp = synthetic.model_hparams(spec)
    torch.manual_seed(0)
    ddpm = DDPM(**hp)
    synthetic.init_reference_like_weights(ddpm)
    d = torch.device("cuda", 0)
    ddpm = ddpm.to(d)
    items = synthetic.make_items(spec)
    if spec.pocket:
        ddpm.train_dataset = MOADDataset(items)
    data = {k: (v.to(d) if torch.is_tensor(v) else v) for k, v in collate(items).items()}
    B, N = data['positions'].shape[:2]
    # the bare forward sees what the step's forward sees: a noised latent and one t per molecule
    g = torch.Generator(device=d).manual_seed(1)
    z = torch.cat([data['positions'], data['one_hot'] / 4], dim=2)
    z = z * data['fragment_mask'] + torch.randn(z.shape, device=d, generator=g) * data['linker_mask']
    t = torch.rand((B, 1), device=d, generator=g)
    fo = data.get('fragment_only_mask')
    ctx = torch.cat([fo, data['fragment_mask'] - fo], dim=-1) if spec.pocket else data['fragment_mask']
    dyn = ddpm.edm.dynamics
    lib = _native.load_library()
    stream = torch.cuda.current_stream(d)
    step = lambda: ddpm.validation_step(data)
    fwd = lambda: dyn(t, z, data['atom_mask'], data['linker_mask'], data['edge_mask'], ctx)
    for _ in range(warmup):
        step(); fwd()
    st_ms, st_native, fw_ms, fw_native = [], [], [], []
    for _ in range(steps):
        st_ms.append(timed(step, stream)); st_native.append(float(lib.dl_last_elapsed_ms(dyn._engine)))
        fw_ms.append(timed(fwd, stream)); fw_native.append(float(lib.dl_last_elapsed_ms(dyn._engine)))
    med = statistics.median
    out = dict(shape=name, B=B, N=N, L=spec.L, graph_type=spec.graph_type, steps=steps,
               step_ms=med(st_ms), step_native_ms=med(st_native), forward_ms=med(fw_ms), forward_native_ms=med(fw_native),
               molecules_per_s=B / (med(st_ms) * 1e-3),
               loss_kernels_overhead=med(st_native) / med(fw_native) - 1.0,
               step_over_forward=med(st_ms) / med(fw_ms) - 1.0,
               step_ms_spread=[min(st_ms), max(st_ms)], forward_ms_spread=[min(fw_ms), max(fw_ms)])
    out["reference_cpu"] = reference_cpu(spec, hp, ddpm, CPU_SAMPLE[name])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--shapes", default="cfg2_zinc,cfg2_zinc_L8,cfg3_geom,cfg4_pockets")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("loss_bench.py measures on a GPU; none is visible")
    name, power = card()
    rows = [run_shape(s, args.steps, args.warmup) for s in args.shapes.split(",")]
    print(json.dumps(dict(bench="diffusion_loss", card=name, power_limit=power, torch=torch.__version__, shapes=rows)))


if __name__ == "__main__":
    main()
