"""Shared test plumbing: golden-vector loading, seeded model construction (weights are reproduced from the seed
and verified by sha256 -- see oracle/make_golden.py), oracle configs."""
import contextlib
import hashlib
import json
import os

import numpy as np
import torch

from difflinker_b200 import synthetic
from oracle import difflinker_oracle as orc

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLDEN_THREADS = 8          # oracle/make_golden*.py generate the fixtures under torch.set_num_threads(8)


@contextlib.contextmanager
def golden_threads():
    """Replays a fixture on the CPU with the torch thread count it was generated with. torch's CPU results depend in the last
    bits on the intra-op thread count, and a chain of reverse steps amplifies those bits beyond the fixtures' tolerance (on a
    16-core host the oracle chains end 1 ulp of coordinates near 2e4 away from the reference's; at 8 threads, bit-exact)."""
    saved = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    try:
        yield
    finally:
        torch.set_num_threads(saved)


EXTRA_SPECS = {
    "small_fc": synthetic.WorkloadSpec("small_fc", B=3, N=12, n_min=7, l_min=2, l_max=4, F=8, L=2, T=20, seed=11),
    "small_geom": synthetic.WorkloadSpec("small_geom", B=5, N=23, n_min=11, l_min=1, l_max=9, F=9, L=3, T=20, seed=12,
                                         anchors_context=True),
}
for _gt in ("FC-10A-4A", "FC-4A", "4A"):
    EXTRA_SPECS[f"small_pocket_{_gt}"] = synthetic.WorkloadSpec(f"small_pocket_{_gt}", B=2, N=70, n_min=70, l_min=5,
                                                                l_max=5, F=9, L=2, T=20, seed=13, pocket=50,
                                                                graph_type=_gt)


def spec_by_name(name):
    return synthetic.SPECS.get(name) or EXTRA_SPECS[name]


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)
    meta = json.loads(str(z["meta"]))
    arrays = {k: torch.from_numpy(z[k]) for k in z.files if k != "meta"}
    return meta, arrays


def state_sha(sd) -> str:
    h = hashlib.sha256()
    for k, v in sd.items():
        h.update(k.encode())
        h.update(v.detach().cpu().float().contiguous().numpy().tobytes())
    return h.hexdigest()


def oracle_cfg(hp):
    return orc.OracleConfig(in_node_nf=hp['in_node_nf'], context_node_nf=hp['context_node_nf'], n_layers=hp['n_layers'],
                            inv_sublayers=hp['inv_sublayers'], norm_constant=hp['norm_constant'],
                            normalization_factor=hp['normalization_factor'], graph_type=hp['graph_type'])


def build_dynamics(spec, seed, edge_impl='auto', **over):
    """Product-side Dynamics with the fixture's weights (same seed, same construction order as the reference)."""
    from difflinker_b200 import Dynamics, DynamicsWithPockets
    hp = synthetic.model_hparams(spec)
    torch.manual_seed(seed)
    cls = DynamicsWithPockets if spec.pocket else Dynamics
    dyn = cls(in_node_nf=hp['in_node_nf'], n_dims=3, context_node_nf=hp['context_node_nf'], hidden_nf=128,
              n_layers=hp['n_layers'], norm_constant=hp['norm_constant'], inv_sublayers=hp['inv_sublayers'],
              normalization_factor=hp['normalization_factor'], graph_type=hp['graph_type'], edge_impl=edge_impl, **over)
    synthetic.init_reference_like_weights(dyn)
    return dyn, hp


def build_ddpm(spec, seed, edge_impl='auto', **over):
    from difflinker_b200 import DDPM
    hp = synthetic.model_hparams(spec)
    hp.update(over)
    torch.manual_seed(seed)
    m = DDPM(**hp, edge_impl=edge_impl)
    synthetic.init_reference_like_weights(m)
    return m, hp


def build_size_classifier(meta):
    """Host-side SizeClassifier with the fixture's weights (same seed and construction order as the reference) and the
    fixture's batch (collate_with_fragment_edges layout)."""
    from difflinker_b200 import linker_size
    spec = spec_by_name(meta["spec"])
    torch.manual_seed(meta["seed"])
    model = linker_size.SizeClassifier(in_node_nf=spec.F, hidden_nf=128, out_node_nf=meta["out_nf"], n_layers=3,
                                       normalization=meta["normalization"])
    synthetic.init_size_gnn_like_trained(model, meta["seed"])
    model.eval()
    data = linker_size.collate_with_fragment_edges(synthetic.make_items(spec, batch=meta["batch"]))
    return model, data


def seeded_noise(seed):
    g = torch.Generator().manual_seed(seed)
    return lambda shape: torch.randn(tuple(shape), generator=g)


def noise_tensor(seed, T, B, N, F):
    """The (T+2,B,N,3+F) tensor holding the reference's draw sequence: randn(B,N,3) then randn(B,N,F) per draw."""
    draw = seeded_noise(seed)
    out = torch.empty((T + 2, B, N, 3 + F))
    for r in range(T + 2):
        out[r, :, :, :3] = draw((B, N, 3))
        out[r, :, :, 3:] = draw((B, N, F))
    return out


def inpaint_noise_tensor(seed, T, B, N, F, node_mask, fragment_mask):
    """(2T+3,B,N,3+F): InpaintingEDM's draws in the reference's call order (edm.py:565,645,669,689,706), each already
    masked and, for the coordinates, projected to zero centre of mass -- the form dl_sample_chain(INPAINT) consumes."""
    from oracle import difflinker_oracle as orc
    draw = seeded_noise(seed)
    nm, fm = node_mask.float(), fragment_mask.float()
    masks = [nm] + [nm, fm] * T + [nm, nm]
    return torch.stack([orc.com_free_noise(draw, B, N, 3, F, m) for m in masks])


def context_of(batch, spec):
    if spec.pocket:
        fo = batch['fragment_only_mask']
        parts = [fo, batch['fragment_mask'] - fo]
    else:
        parts = [batch['fragment_mask']]
    if spec.anchors_context:
        parts = [batch['anchors']] + parts
    return torch.cat(parts, dim=-1)


def random_latent(batch, seed, pad_garbage=True):
    g = torch.Generator().manual_seed(seed)
    z = torch.cat([batch['positions'], batch['one_hot'] / 4], dim=2)
    z = z * batch['fragment_mask'] + torch.randn(z.shape, generator=g) * batch['linker_mask']
    if pad_garbage:
        z = z + 3.0 * torch.randn(z.shape, generator=g) * (1 - batch['atom_mask'].float())
    t = torch.rand((z.shape[0], 1), generator=g)
    return z, t


def build_c_example(out_dir):
    """gcc build of examples/c_sampler.c against the in-tree library and the CUDA runtime; returns the binary's path."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    lib_dir = os.path.join(root, "difflinker_b200")
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    exe = os.path.join(str(out_dir), "c_sampler")
    cmd = ["gcc", "-std=c99", "-O2", "-Wall", "-Wextra", os.path.join(root, "examples", "c_sampler.c"), "-I" + os.path.join(root, "include"),
           "-I" + os.path.join(cuda, "include"), "-L" + lib_dir, "-ldifflinker_b200", "-L" + os.path.join(cuda, "lib64"), "-lcudart",
           "-Wl,-rpath," + lib_dir, "-Wl,-rpath," + os.path.join(cuda, "lib64"), "-o", exe]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-3000:]
    assert "warning" not in res.stderr.replace("ISO C99 doesn", ""), res.stderr[-3000:]
    return exe

