"""GPU parity tests: the CUDA path (through the C-ABI, via the reference-facing modules) against the golden vectors
of the live reference and against the CPU oracle on the same seeded inputs.
Tolerance (BASELINE.json north_star): 1e-4 relative fp32 on coordinates/features, atom types identical."""
import math

import pytest
import torch

from difflinker_b200 import FoundNaNException, synthetic
from difflinker_b200.batching import collate, create_templates_for_linker_generation
import dl_helpers as helpers
from oracle import difflinker_oracle as orc

pytestmark = pytest.mark.gpu
REL_TOL = 1e-4

DYN_CASES = ["dyn_small_fc", "dyn_small_fc_tscalar", "dyn_cfg1", "dyn_small_geom_anchors",
             "dyn_small_pocket_FC-10A-4A", "dyn_small_pocket_FC-4A", "dyn_small_pocket_4A"]
IMPLS = ["simt", "auto"]


def dev():
    assert torch.cuda.is_available()
    torch.cuda.init()               # torch.cuda.default_generators is empty until torch's own lazy CUDA initialisation has run
    return torch.device("cuda", 0)


def rel_err(got, want):
    return (got.double() - want.double()).abs().max().item() / max(want.double().abs().max().item(), 1e-30)


def run_dyn(dyn, t, z, nm, lm, em, ctx, device):
    mv = lambda v: None if v is None else v.to(device)
    return dyn(mv(t), mv(z), mv(nm), mv(lm), mv(em), mv(ctx)).cpu()


@pytest.mark.parametrize("impl", IMPLS)
@pytest.mark.parametrize("name", DYN_CASES)
def test_dynamics_forward_matches_reference_golden(name, impl):
    meta, a = helpers.load_golden(name)
    spec = helpers.spec_by_name(meta["spec"])
    dyn, hp = helpers.build_dynamics(spec, meta["seed"], edge_impl=impl)
    assert helpers.state_sha(dyn.state_dict()) == meta["sha"]
    out = run_dyn(dyn, a["t"], a["xh"], a["node_mask"], a["linker_mask"], a["edge_mask"], a["context"], dev())
    assert out.shape == a["out"].shape
    assert rel_err(out[..., :3], a["out"][..., :3]) <= REL_TOL
    assert rel_err(out[..., 3:], a["out"][..., 3:]) <= REL_TOL
    assert torch.equal(out * (1 - a["node_mask"].float()), torch.zeros_like(out))   # masked rows exactly zero


@pytest.mark.parametrize("name", ["dyn_small_fc", "dyn_cfg1"])
def test_host_buffer_entry_point_equals_device_entry_point(name):
    meta, a = helpers.load_golden(name)
    dyn, hp = helpers.build_dynamics(helpers.spec_by_name(meta["spec"]), meta["seed"])
    on_dev = run_dyn(dyn, a["t"], a["xh"], a["node_mask"], a["linker_mask"], a["edge_mask"], a["context"], dev())
    on_host = dyn(a["t"], a["xh"], a["node_mask"], a["linker_mask"], a["edge_mask"], a["context"])   # CPU tensors
    assert not on_host.is_cuda and torch.equal(on_host, on_dev)


@pytest.mark.parametrize("impl", IMPLS)
@pytest.mark.parametrize("name", ["chain_cfg1", "chain_cfg1_nsteps20"])
def test_sample_chain_matches_reference_golden(name, impl):
    meta, a = helpers.load_golden(name)
    spec = helpers.spec_by_name(meta["spec"])
    ddpm, hp = helpers.build_ddpm(spec, meta["seed"], edge_impl=impl)
    ddpm.edm.T = meta["T"]
    d = dev()
    data = collate(synthetic.make_items(spec, batch=meta["batch"]))
    tpl = create_templates_for_linker_generation(data, data['linker_mask'].sum(1).view(-1).int())
    B, N = tpl['positions'].shape[:2]
    noise = helpers.noise_tensor(meta["noise_seed"], meta["T"], B, N, spec.F)
    from difflinker_b200 import utils
    x = utils.remove_partial_mean_with_mask(tpl['positions'], tpl['atom_mask'], tpl['fragment_mask'])
    mv = lambda v: v.to(d)
    chain = ddpm.edm.sample_chain(x=mv(x), h=mv(tpl['one_hot']), node_mask=mv(tpl['atom_mask']),
                                  fragment_mask=mv(tpl['fragment_mask']), linker_mask=mv(tpl['linker_mask']),
                                  edge_mask=mv(tpl['edge_mask']), context=mv(tpl['fragment_mask']),
                                  keep_frames=meta["keep_frames"], noise=mv(noise)).cpu()
    want = a["chain"]
    assert chain.shape == want.shape
    assert torch.equal(chain[0][..., 3:], want[0][..., 3:]), "atom types differ"
    lm = tpl['linker_mask']
    assert rel_err(chain[0][..., :3] * lm, want[0][..., :3] * lm) <= REL_TOL
    for f in range(1, meta["keep_frames"]):
        assert rel_err(chain[f], want[f]) <= REL_TOL, f
    # fragments pass through the sampler bit-identically (edm.py:137,206,229)
    fm = tpl['fragment_mask']
    assert torch.equal(chain[0][..., :3] * fm, x * fm)


class MOADDataset(list):
    """Stand-in with the reference class's NAME: lightning.py:441 switches the centre-of-mass mask on
    `isinstance(self.val_dataset, MOADDataset)`, which generate_with_pocket.py:249-250 sets before sampling."""


PUBLIC_CHAINS = ["chain_cfg1", "chain_small_pocket_FC-10A-4A", "chain_small_pocket_FC-4A", "chain_small_pocket_4A",
                 "chain_cfg2_zinc_T500", "chain_cfg2_zinc_L8_T500", "chain_cfg3_geom_T500"]


@pytest.mark.parametrize("name", PUBLIC_CHAINS)
def test_public_ddpm_sample_chain_matches_reference_golden(name):
    """The call generate.py:156 / generate_with_pocket.py:265 make -- `DDPM.sample_chain(data, keep_frames)` -- against chains
    the live reference produced through the SAME entry point (oracle/make_golden*.py), with the reference's noise draws
    injected through `EDM.draw_noise`. Covers the benchmarked shapes (configs 2 and 3 non-ragged, T=500, L=6 and the real
    ZINC depth L=8; 8-molecule slices) and pocket-conditioned sampling (MOAD prefix, val_dataset set, all three cut-off
    graph types: the graph is rebuilt from the current coordinates at every one of the T+1 calls)."""
    meta, a = helpers.load_golden(name)
    spec = helpers.spec_by_name(meta["spec"])
    ddpm, hp = helpers.build_ddpm(spec, meta["seed"], diffusion_steps=meta["table_timesteps"])
    assert helpers.state_sha(ddpm.edm.dynamics.state_dict()) == meta["sha"]
    ddpm.edm.T = meta["T"]
    items = synthetic.make_items(spec, batch=meta["batch"])
    if meta.get("moad_val_dataset"):
        ddpm.val_dataset = MOADDataset(items)
    d = dev()
    ddpm = ddpm.to(d)
    data = collate(items)
    sizes = data['linker_mask'].sum(1).view(-1).int()
    tpl = create_templates_for_linker_generation(data, sizes)
    B, N = tpl['positions'].shape[:2]
    noise = helpers.noise_tensor(meta["noise_seed"], meta["T"], B, N, spec.F)
    calls = []

    def injected(n_draws, n_samples, n_nodes, device, generator=None):
        calls.append((n_draws, n_samples, n_nodes))
        assert (n_draws, n_samples, n_nodes) == (meta["T"] + 2, B, N)
        return noise.to(device)
    ddpm.edm.draw_noise = injected
    data_dev = {k: (v.to(d) if torch.is_tensor(v) else v) for k, v in data.items()}
    chain, node_mask = ddpm.sample_chain(data_dev, keep_frames=meta["keep_frames"])
    assert len(calls) == 1
    chain, node_mask = chain.cpu(), node_mask.cpu()
    want = a["chain"]
    assert chain.shape == want.shape and torch.equal(node_mask, a["node_mask"])
    assert torch.equal(chain[0][..., 3:], want[0][..., 3:]), "atom types differ"
    lm = tpl['linker_mask']
    if "drift64" not in a:
        assert rel_err(chain[0][..., :3] * lm, want[0][..., :3] * lm) <= REL_TOL
        assert rel_err(chain[0][..., :3], want[0][..., :3]) <= REL_TOL
    else:
        # Per molecule: 1e-4 of the coordinate scale, or -- where the trajectory itself is ill-conditioned -- 30x the distance
        # between the REFERENCE's own fp32 and fp64 runs on the same noise (`drift64`, oracle/make_golden_r2.py drift). For the
        # L=6 and cfg3 fixtures drift64 is 1e-4 .. 6e-4 A on coordinates of 170 .. 330 A and the 1e-4 bound is the binding one
        # for every molecule. With random weights at L=8 (coord_mlp gain x100, 8 blocks) the reference's fp32 and fp64 results
        # are 6.7 A and 2.2 A apart for two of the eight molecules and 1e-3 .. 1e-2 A for three more; every re-ordering of the
        # fp32 arithmetic moves those by a comparable amount (the fp32 SIMT path lands 4.2 A from the fixture on molecule 1, the
        # tcgen05 path 6.3 A). At least half of the molecules must meet the plain 1e-4 bound outright (measured: 5 of 8 at L=8).
        scale = want[0][..., :3].abs().max().item()
        err = ((chain[0][..., :3] - want[0][..., :3]) * lm).abs().flatten(1).max(1).values
        tol = torch.maximum(torch.full_like(err, REL_TOL * scale), 30.0 * a["drift64"].float())
        assert (err <= tol).all(), (err.tolist(), tol.tolist())
        assert (err <= REL_TOL * scale).sum() >= (B + 1) // 2, (err.tolist(), REL_TOL * scale)
    for f in range(1, meta["keep_frames"]):
        assert rel_err(chain[f], want[f]) <= REL_TOL, f


@pytest.mark.parametrize("N,nb", [(32, 4), (64, 3), (256, 2)])
def test_forward_padded_n_sweep_l6_vs_oracle(N, nb):
    """BASELINE configs[4] (padded-N sweep) at its real depth L=6: N=32 and N=64 run the third-generation edge kernels
    (TMA-staged panels), N=256 the column-chunked second-generation ones."""
    spec = synthetic.SPECS[f"cfg5_sweep_N{N}"]
    dyn, hp = helpers.build_dynamics(spec, 0)
    assert hp['n_layers'] == 6
    batch = collate(synthetic.make_items(spec, batch=nb))
    z, t = helpers.random_latent(batch, 7)
    ctx = helpers.context_of(batch, spec)
    with torch.no_grad():
        want = orc.dynamics_forward(dyn.state_dict(), helpers.oracle_cfg(hp), t, z, batch['atom_mask'],
                                    batch['linker_mask'], batch['edge_mask'], ctx)
    got = run_dyn(dyn, t, z, batch['atom_mask'], batch['linker_mask'], batch['edge_mask'], ctx, dev())
    assert rel_err(got[..., :3], want[..., :3]) <= REL_TOL
    assert rel_err(got[..., 3:], want[..., 3:]) <= REL_TOL


@pytest.mark.parametrize("spec_name,nb", [("cfg2_zinc_ragged", 16), ("cfg3_geom_ragged", 8), ("small_pocket_FC-10A-4A", 2)])
def test_device_side_collate_and_templates_match_oracle(spec_name, nb):
    """datasets.collate / create_templates_for_linker_generation (datasets.py:332-375, 483-512) run as torch ops on the
    batch's device: every tensor of the result equals the oracle's per-molecule formulation bit for bit, with the
    reference's dtypes (int8 masks incl. the -1/-2 edge mask, or the batch-id vector for pockets)."""
    spec = helpers.spec_by_name(spec_name)
    items = synthetic.make_items(spec, batch=nb)
    want_c = orc.collate_molecules(items)
    g = torch.Generator().manual_seed(3)
    sizes = torch.randint(1, 12, (nb,), generator=g).int()
    want_t = orc.linker_templates(want_c, sizes)
    d = dev()
    items_dev = [{k: (v.to(d) if torch.is_tensor(v) else v) for k, v in it.items()} for it in items]
    got_c = collate(items_dev)
    got_t = create_templates_for_linker_generation(got_c, sizes.to(d))
    for want, got in ((want_c, got_c), (want_t, got_t)):
        for k, v in want.items():
            if torch.is_tensor(v):
                assert got[k].is_cuda and got[k].dtype == v.dtype and torch.equal(got[k].cpu(), v), k


@pytest.mark.parametrize("impl", IMPLS)
def test_inpainting_sample_chain_matches_reference_golden(impl):
    """InpaintingEDM (edm.py:549-727) through DDPM(inpainting=True): centring dynamics, all atoms move, fragments are
    re-noised from the data every step."""
    meta, a = helpers.load_golden("inpaint_chain_cfg1")
    spec = helpers.spec_by_name(meta["spec"])
    ddpm, hp = helpers.build_ddpm(spec, meta["seed"], edge_impl=impl, inpainting=True)
    from difflinker_b200 import InpaintingEDM, utils
    assert isinstance(ddpm.edm, InpaintingEDM)
    d = dev()
    data = collate(synthetic.make_items(spec, batch=meta["batch"]))
    B, N = data['positions'].shape[:2]
    noise = helpers.inpaint_noise_tensor(meta["noise_seed"], meta["T"], B, N, spec.F, data['atom_mask'], data['fragment_mask'])
    x = utils.remove_partial_mean_with_mask(data['positions'], data['atom_mask'], data['atom_mask'])
    mv = lambda v: v.to(d)
    chain = ddpm.edm.sample_chain(x=mv(x), h=mv(data['one_hot']), node_mask=mv(data['atom_mask']),
                                  fragment_mask=mv(data['fragment_mask']), linker_mask=mv(data['linker_mask']),
                                  edge_mask=mv(data['edge_mask']), context=mv(data['fragment_mask']),
                                  keep_frames=meta["keep_frames"], noise=mv(noise)).cpu()
    want = a["chain"]
    assert chain.shape == want.shape
    assert torch.equal(chain[0][..., 3:], want[0][..., 3:]), "atom types differ"
    for f in range(meta["keep_frames"]):
        assert rel_err(chain[f], want[f]) <= REL_TOL, f
    # the public entry point with its own noise: finite, one-hot atom types, zero centre of mass per molecule
    ddpm = ddpm.to(d)
    chain2, nm = ddpm.sample_chain(data, keep_frames=1)
    assert torch.isfinite(chain2).all()
    assert torch.equal(chain2[0][..., 3:].sum(-1).cpu(), data['atom_mask'].squeeze(-1).float())


@pytest.mark.parametrize("impl", IMPLS)
def test_centering_dynamics_forward_vs_oracle(impl):
    """Dynamics(centering=True) (egnn.py:404-410): the velocity is re-centred over all atoms."""
    spec = helpers.spec_by_name("cfg1_plumbing")
    dyn, hp = helpers.build_dynamics(spec, 3, edge_impl=impl, centering=True)
    batch = collate(synthetic.make_items(spec, batch=5))
    z, t = helpers.random_latent(batch, 11)
    ctx = helpers.context_of(batch, spec)
    ocfg = helpers.oracle_cfg(hp)
    ocfg.centering = True
    with torch.no_grad():
        want = orc.dynamics_forward(dyn.state_dict(), ocfg, t, z, batch['atom_mask'], None, batch['edge_mask'], ctx)
    got = run_dyn(dyn, t, z, batch['atom_mask'], None, batch['edge_mask'], ctx, dev())
    assert rel_err(got, want) <= REL_TOL


@pytest.mark.parametrize("impl", IMPLS)
@pytest.mark.parametrize("spec_name,nb", [("cfg2_zinc_ragged", 8), ("cfg3_geom_ragged", 4)])
def test_forward_at_config_shapes_vs_oracle(spec_name, nb, impl):
    spec = synthetic.SPECS[spec_name]
    dyn, hp = helpers.build_dynamics(spec, 0, edge_impl=impl)
    batch = collate(synthetic.make_items(spec, batch=nb))
    z, t = helpers.random_latent(batch, 5)
    ctx = helpers.context_of(batch, spec)
    with torch.no_grad():
        want = orc.dynamics_forward(dyn.state_dict(), helpers.oracle_cfg(hp), t, z, batch['atom_mask'],
                                    batch['linker_mask'], batch['edge_mask'], ctx)
    got = run_dyn(dyn, t, z, batch['atom_mask'], batch['linker_mask'], batch['edge_mask'], ctx, dev())
    assert rel_err(got[..., :3], want[..., :3]) <= REL_TOL
    assert rel_err(got[..., 3:], want[..., 3:]) <= REL_TOL


@pytest.mark.parametrize("impl", IMPLS)
@pytest.mark.parametrize("N,B,L", [(1, 2, 1), (2, 1, 1), (13, 3, 2), (150, 2, 1), (257, 1, 1)])
def test_odd_shapes_vs_oracle(N, B, L, impl):
    """N=1 (self loop only), N not a tile multiple, N > one 128-column chunk, N > 256."""
    spec = synthetic.WorkloadSpec(f"odd{N}", B=B, N=N, n_min=max(1, N // 2), l_min=0, l_max=max(0, min(5, N - 1)),
                                  F=8, L=L, T=4, seed=31)
    g = torch.Generator().manual_seed(N)
    items = []
    for b in range(B):
        n = N if b == 0 else max(1, N - 3 * b)
        lk = min(n - 1, 1 + b) if n > 1 else 0
        fm = torch.zeros(n); fm[:n - lk] = 1
        items.append(dict(uuid=b, name=str(b), positions=2 * torch.randn((n, 3), generator=g),
                          one_hot=torch.eye(8)[torch.randint(0, 8, (n,), generator=g)], anchors=torch.zeros(n),
                          fragment_mask=fm, linker_mask=1 - fm, num_atoms=n))
    batch = collate(items)
    dyn, hp = helpers.build_dynamics(spec, 1, edge_impl=impl)
    z, t = helpers.random_latent(batch, 9)
    with torch.no_grad():
        want = orc.dynamics_forward(dyn.state_dict(), helpers.oracle_cfg(hp), t, z, batch['atom_mask'],
                                    batch['linker_mask'], batch['edge_mask'], batch['fragment_mask'])
    got = run_dyn(dyn, t, z, batch['atom_mask'], batch['linker_mask'], batch['edge_mask'], batch['fragment_mask'], dev())
    assert (got - want).abs().max().item() <= REL_TOL * max(want.abs().max().item(), 1e-3)


def test_edge_mask_none_and_linker_mask_none():
    """edge_mask=None -> every pair weighs 1 (egnn.py:58-59 skipped); linker_mask=None -> every row moves
    (inpainting call sites, edm.py:505,632)."""
    spec = helpers.EXTRA_SPECS["small_fc"]
    dyn, hp = helpers.build_dynamics(spec, 4)
    batch = collate(synthetic.make_items(spec))
    z, t = helpers.random_latent(batch, 2, pad_garbage=False)
    for em, lm in [(None, batch['linker_mask']), (batch['edge_mask'], None), (None, None)]:
        with torch.no_grad():
            want = orc.dynamics_forward(dyn.state_dict(), helpers.oracle_cfg(hp), t, z, batch['atom_mask'], lm, em,
                                        batch['fragment_mask'])
        got = run_dyn(dyn, t, z, batch['atom_mask'], lm, em, batch['fragment_mask'], dev())
        assert rel_err(got, want) <= REL_TOL


def test_fully_masked_molecule_and_empty_linker():
    spec = helpers.EXTRA_SPECS["small_fc"]
    dyn, hp = helpers.build_dynamics(spec, 4)
    batch = collate(synthetic.make_items(spec))
    batch['atom_mask'][1] = 0                                    # molecule 1 has no valid atoms at all
    batch['edge_mask'] = batch['edge_mask'].view(spec.B, -1).clone()
    batch['edge_mask'][1] = 0
    batch['edge_mask'] = batch['edge_mask'].view(-1, 1)
    batch['linker_mask'][2] = 0                                  # molecule 2 has no linker atoms
    z, t = helpers.random_latent(batch, 3)
    with torch.no_grad():
        want = orc.dynamics_forward(dyn.state_dict(), helpers.oracle_cfg(hp), t, z, batch['atom_mask'],
                                    batch['linker_mask'], batch['edge_mask'], batch['fragment_mask'])
    got = run_dyn(dyn, t, z, batch['atom_mask'], batch['linker_mask'], batch['edge_mask'], batch['fragment_mask'], dev())
    assert rel_err(got, want) <= REL_TOL
    assert torch.equal(got[1], torch.zeros_like(got[1]))
    assert torch.equal(got[2][..., :3], torch.zeros_like(got[2][..., :3]))   # nothing moves without linker rows


def test_e3_equivariance():
    """Rotating + translating the input rotates vel and leaves h invariant (coord2diff uses differences only)."""
    spec = helpers.EXTRA_SPECS["small_fc"]
    dyn, hp = helpers.build_dynamics(spec, 6)
    batch = collate(synthetic.make_items(spec))
    z, t = helpers.random_latent(batch, 8, pad_garbage=False)
    g = torch.Generator().manual_seed(1)
    q, _ = torch.linalg.qr(torch.randn(3, 3, generator=g))
    if torch.det(q) < 0:
        q[:, 0] = -q[:, 0]
    z2 = z.clone()
    z2[..., :3] = (z[..., :3] @ q.T + torch.tensor([1.5, -2.0, 0.7])) * batch['atom_mask'].float()
    a = run_dyn(dyn, t, z, batch['atom_mask'], batch['linker_mask'], batch['edge_mask'], batch['fragment_mask'], dev())
    b = run_dyn(dyn, t, z2, batch['atom_mask'], batch['linker_mask'], batch['edge_mask'], batch['fragment_mask'], dev())
    assert (b[..., :3] - a[..., :3] @ q.T).abs().max().item() <= 2e-4 * max(a[..., :3].abs().max().item(), 1e-3)
    assert rel_err(b[..., 3:], a[..., 3:]) <= 2e-4


def test_nan_raises_found_nan_exception_with_indices():
    spec = helpers.EXTRA_SPECS["small_fc"]
    dyn, hp = helpers.build_dynamics(spec, 4)
    batch = collate(synthetic.make_items(spec))
    z, t = helpers.random_latent(batch, 3, pad_garbage=False)
    z[1, 0, 0] = float('nan')                                    # poisons coordinates and, through d_ij, features
    with pytest.raises(FoundNaNException) as ei:
        run_dyn(dyn, t, z, batch['atom_mask'], batch['linker_mask'], batch['edge_mask'], batch['fragment_mask'], dev())
    e = ei.value
    assert (e.x_h_nan_idx | e.only_x_nan_idx | e.only_h_nan_idx) == {1}
    # and the engine stays usable afterwards
    z[1, 0, 0] = 0.0
    out = run_dyn(dyn, t, z, batch['atom_mask'], batch['linker_mask'], batch['edge_mask'], batch['fragment_mask'], dev())
    assert torch.isfinite(out).all()


@pytest.mark.parametrize("impl", IMPLS)
def test_full_size_sampling_properties(impl):
    """BASELINE configs[1] size (B=256, N=40, L=6) with a shortened chain: size-independent invariants."""
    spec = synthetic.SPECS["cfg2_zinc_ragged"]
    ddpm, hp = helpers.build_ddpm(spec, 0, edge_impl=impl, diffusion_steps=12)
    d = dev()
    ddpm = ddpm.to(d)
    data = collate(synthetic.make_items(spec))
    data = {k: (v.to(d) if torch.is_tensor(v) else v) for k, v in data.items()}
    torch.manual_seed(123)
    chain, node_mask = ddpm.sample_chain(data, keep_frames=4)
    torch.manual_seed(123)
    chain2, _ = ddpm.sample_chain(data, keep_frames=4)
    assert chain.shape == (4, spec.B, spec.N, 3 + spec.F)                       # sample_trajectories.py:49-51
    assert torch.equal(chain, chain2), "same torch seed must give the same sample (deterministic kernels)"
    final = chain[0]
    nm = node_mask.float()
    assert torch.isfinite(chain).all()
    assert torch.equal(final * (1 - nm), torch.zeros_like(final))               # utils.py:99-101
    onehot = final[..., 3:]
    assert torch.equal(onehot.sum(-1), nm.squeeze(-1)) and set(onehot.unique().tolist()) <= {0.0, 1.0}
    fm = data['fragment_mask']
    from difflinker_b200 import utils
    x0 = utils.remove_partial_mean_with_mask(data['positions'], data['atom_mask'], fm)
    assert torch.equal(final[..., :3] * fm, x0 * fm)                            # fragments untouched
    assert torch.equal(final[..., 3:] * fm, data['one_hot'] * fm)
    lm = data['linker_mask']
    assert ((final[..., :3] * lm).abs().sum(dim=(1, 2)) > 0).all()              # every linker moved somewhere


def test_full_size_forward_vs_oracle_sampled_molecules():
    """Full B=256 launch on the GPU; the oracle checks a slice of molecules (they are independent)."""
    spec = synthetic.SPECS["cfg2_zinc_ragged"]
    dyn, hp = helpers.build_dynamics(spec, 0)
    batch = collate(synthetic.make_items(spec))
    z, t = helpers.random_latent(batch, 5)
    got = run_dyn(dyn, t, z, batch['atom_mask'], batch['linker_mask'], batch['edge_mask'], batch['fragment_mask'], dev())
    idx = torch.tensor([0, 1, 77, 128, 255])
    em = batch['edge_mask'].view(spec.B, -1)[idx].reshape(-1, 1)
    with torch.no_grad():
        want = orc.dynamics_forward(dyn.state_dict(), helpers.oracle_cfg(hp), t[idx], z[idx], batch['atom_mask'][idx],
                                    batch['linker_mask'][idx], em, batch['fragment_mask'][idx])
    assert rel_err(got[idx], want) <= REL_TOL


@pytest.mark.parametrize("b_mn_major", [0, 1, 2])
def test_umma_selftest_3xfp16(b_mn_major):
    """tcgen05 building block in isolation: one 128x256x128 hi/lo-split UMMA chain vs fp64 on the host, with the B operand
    in the K-major layout the kernels use (0), in the MN-major canonical layout (1), and with the A operand (the
    stationary W2) in tensor memory as k_edge_v3 keeps it (2)."""
    import ctypes as C
    from difflinker_b200 import _native
    dyn, hp = helpers.build_dynamics(helpers.EXTRA_SPECS["small_fc"], 0)
    eng = dyn.engine(0)
    lib = _native.load_library()
    ea, er = C.c_float(-1), C.c_float(-1)
    st = lib.dl_selftest_tc_layout(eng, b_mn_major, C.byref(ea), C.byref(er))
    assert st == 0, lib.dl_last_error()
    assert 0 <= er.value < 2e-6, (ea.value, er.value)
    if not b_mn_major:
        assert lib.dl_selftest_tc(eng, C.byref(ea), C.byref(er)) == 0 and 0 <= er.value < 2e-6


def test_simt_and_tcgen05_edge_paths_agree():
    spec = synthetic.SPECS["cfg2_zinc_ragged"]
    batch = collate(synthetic.make_items(spec, batch=16))
    z, t = helpers.random_latent(batch, 5)
    outs = {}
    for impl in ("simt", "tcgen05"):
        dyn, hp = helpers.build_dynamics(spec, 0, edge_impl=impl)
        outs[impl] = run_dyn(dyn, t, z, batch['atom_mask'], batch['linker_mask'], batch['edge_mask'],
                             batch['fragment_mask'], dev())
    assert rel_err(outs["tcgen05"], outs["simt"]) <= 2e-5


def test_pockets_full_size_slice_vs_oracle():
    """BASELINE configs[3] shape (N=300: 22 fragment + 270 pocket + 8 linker atoms, FC-10A-4A cut-off graph, L=6),
    a 3-molecule slice against the oracle's O((BN)^2) adjacency construction (egnn.py:565-596)."""
    spec = synthetic.SPECS["cfg4_pockets"]
    dyn, hp = helpers.build_dynamics(spec, 0)
    batch = collate(synthetic.make_items(spec, batch=3))
    z, t = helpers.random_latent(batch, 11)
    ctx = helpers.context_of(batch, spec)
    with torch.no_grad():
        want = orc.dynamics_forward(dyn.state_dict(), helpers.oracle_cfg(hp), t, z, batch['atom_mask'],
                                    batch['linker_mask'], batch['edge_mask'], ctx)
    got = run_dyn(dyn, t, z, batch['atom_mask'], batch['linker_mask'], batch['edge_mask'], ctx, dev())
    assert rel_err(got[..., :3], want[..., :3]) <= REL_TOL
    assert rel_err(got[..., 3:], want[..., 3:]) <= REL_TOL


@pytest.mark.parametrize("graph_type", ["4A", "FC-4A", "FC-10A-4A"])
def test_cutoff_graph_neighbour_lists_isolated_rows_and_chunked_rows(graph_type):
    """The tcgen05 path walks per-row neighbour lists (k_nbr): rows without any neighbour (pocket atoms moved far away),
    rows with more than one tile of neighbours (ligand rows, > 128 entries under FC-10A-4A) and everything between,
    against the oracle's adjacency construction (egnn.py:538-596) and against the dense SIMT path."""
    base = synthetic.SPECS["cfg4_pockets"]
    spec = synthetic.WorkloadSpec(base.name, B=3, N=base.N, n_min=base.n_min, l_min=base.l_min, l_max=base.l_max,
                                  F=base.F, L=2, T=10, seed=7, pocket=base.pocket, graph_type=graph_type)
    dyn, hp = helpers.build_dynamics(spec, 1)
    batch = collate(synthetic.make_items(spec, batch=3))
    z, t = helpers.random_latent(batch, 17, pad_garbage=False)
    # isolate a few pocket atoms of molecule 1: 200 A away and 50 A apart from each other
    pk = torch.nonzero(batch['pocket_mask'][1, :, 0] > 0).view(-1)[:5]
    for k, idx in enumerate(pk.tolist()):
        z[1, idx, :3] = torch.tensor([200.0 + 50.0 * k, -150.0, 90.0])
    ctx = helpers.context_of(batch, spec)
    with torch.no_grad():
        want = orc.dynamics_forward(dyn.state_dict(), helpers.oracle_cfg(hp), t, z, batch['atom_mask'],
                                    batch['linker_mask'], batch['edge_mask'], ctx)
    got = run_dyn(dyn, t, z, batch['atom_mask'], batch['linker_mask'], batch['edge_mask'], ctx, dev())
    assert rel_err(got[..., :3], want[..., :3]) <= REL_TOL
    assert rel_err(got[..., 3:], want[..., 3:]) <= REL_TOL
    dyn_simt, _ = helpers.build_dynamics(spec, 1, edge_impl='simt')
    got_simt = run_dyn(dyn_simt, t, z, batch['atom_mask'], batch['linker_mask'], batch['edge_mask'], ctx, dev())
    assert rel_err(got, got_simt) <= REL_TOL
    # what the neighbour-list kernel packed: exactly the reference's edges (+ one padding column per isolated live row),
    # in well-filled 128-edge tiles (first-fit decreasing over the rows of a molecule)
    import ctypes
    from difflinker_b200 import _native
    stats = (ctypes.c_int64 * 4)()
    _native.check(_native.load_library().dl_cut_graph_stats(dyn.engine(0), stats), "dl_cut_graph_stats")
    B, N = z.shape[:2]
    nmf = batch['atom_mask'].reshape(B * N, 1).float()
    flat = z.reshape(B * N, -1) * nmf
    cflat = ctx.reshape(B * N, -1)
    row, col = orc.pocket_edge_index(flat[:, :3], nmf, batch['edge_mask'].reshape(-1), batch['linker_mask'].reshape(B * N, 1),
                                     cflat[:, -2], cflat[:, -1], graph_type)
    deg = torch.bincount(row, minlength=B * N)
    isolated = int(((deg == 0) & (nmf.view(-1) > 0)).sum())
    assert isolated >= 5
    assert stats[2] == row.numel() + isolated
    assert stats[1] <= math.ceil(1.35 * stats[2] / 128) + B, (stats[1], stats[2])


@pytest.mark.parametrize("N", [128, 512])
def test_sweep_sizes_vs_oracle(N):
    """BASELINE configs[4] padded-N sweep end points (rows spanning 1 and 4 column chunks of the edge tile)."""
    spec = synthetic.SPECS[f"cfg5_sweep_N{N}"]
    spec2 = synthetic.WorkloadSpec(spec.name, B=2, N=N, n_min=N, l_min=8, l_max=8, F=8, L=2, T=10, seed=5)
    dyn, hp = helpers.build_dynamics(spec2, 0)
    batch = collate(synthetic.make_items(spec2))
    z, t = helpers.random_latent(batch, 13)
    with torch.no_grad():
        want = orc.dynamics_forward(dyn.state_dict(), helpers.oracle_cfg(hp), t, z, batch['atom_mask'],
                                    batch['linker_mask'], batch['edge_mask'], batch['fragment_mask'])
    got = run_dyn(dyn, t, z, batch['atom_mask'], batch['linker_mask'], batch['edge_mask'], batch['fragment_mask'], dev())
    assert rel_err(got[..., :3], want[..., :3]) <= REL_TOL
    assert rel_err(got[..., 3:], want[..., 3:]) <= REL_TOL


def test_chain_T500_cfg1_vs_oracle():
    """The headline chain length (T=500) on the small plumbing batch: 501 fused forwards against the oracle loop with
    the same injected noise -- error must not accumulate beyond the 1e-4 tolerance."""
    spec = synthetic.SPECS["cfg1_plumbing"]
    ddpm, hp = helpers.build_ddpm(spec, 0, diffusion_steps=500)
    data = collate(synthetic.make_items(spec))
    tpl = create_templates_for_linker_generation(data, data['linker_mask'].sum(1).view(-1).int())
    B, N = tpl['positions'].shape[:2]
    from difflinker_b200 import utils
    x = utils.remove_partial_mean_with_mask(tpl['positions'], tpl['atom_mask'], tpl['fragment_mask'])
    noise = helpers.noise_tensor(4242, 500, B, N, spec.F)
    d = dev()
    mv = lambda v: v.to(d)
    chain = ddpm.edm.sample_chain(x=mv(x), h=mv(tpl['one_hot']), node_mask=mv(tpl['atom_mask']),
                                  fragment_mask=mv(tpl['fragment_mask']), linker_mask=mv(tpl['linker_mask']),
                                  edge_mask=mv(tpl['edge_mask']), context=mv(tpl['fragment_mask']), keep_frames=1,
                                  noise=mv(noise)).cpu()
    gam = orc.gamma_table(hp['diffusion_noise_schedule'], 500, hp['diffusion_noise_precision'])
    with torch.no_grad():
        want = orc.edm_sample_chain(ddpm.edm.dynamics.state_dict(), helpers.oracle_cfg(hp), gam, 500, x, tpl['one_hot'],
                                    tpl['atom_mask'], tpl['fragment_mask'], tpl['linker_mask'], tpl['edge_mask'],
                                    tpl['fragment_mask'], keep_frames=1, norm_values=tuple(hp['normalize_factors']),
                                    noise_fn=helpers.seeded_noise(4242))
    assert torch.equal(chain[0][..., 3:], want[0][..., 3:]), "atom types differ"
    lm = tpl['linker_mask']
    assert rel_err(chain[0][..., :3] * lm, want[0][..., :3] * lm) <= REL_TOL


def test_restore_frame_vs_oracle():
    """generate.py:163-171 on the device, in place on chain[0] (row stride 3+F) and on a packed (B,N,3) tensor."""
    from difflinker_b200 import output
    spec = synthetic.SPECS["cfg2_zinc_ragged"]
    data = collate(synthetic.make_items(spec, batch=16))
    g = torch.Generator().manual_seed(5)
    chain0 = torch.randn(data['positions'].shape[:2] + (3 + spec.F,), generator=g)
    positions = data['positions'] + torch.tensor([11.0, -7.0, 3.5])
    for com_mask in (data['fragment_mask'], data['anchors']):
        if float(com_mask.sum(1).min()) == 0:
            continue
        want = orc.restore_frame(chain0[..., :3], positions, com_mask, data['atom_mask'])
        got = output.restore_frame(chain0.clone().to(dev()), positions, com_mask, data['atom_mask']).cpu()
        assert rel_err(got[..., :3], want) <= 1e-6
        assert torch.equal(got[..., 3:], chain0[..., 3:])
        got3 = output.restore_frame(chain0[..., :3].contiguous().to(dev()), positions, com_mask, data['atom_mask']).cpu()
        assert torch.equal(got3, got[..., :3])


def test_restore_frame_with_sampled_linker_sizes():
    """generate.py:165-171 with `sample_fn` set: chain[0] / node_mask have the TEMPLATE's padded length, positions and
    com_mask the input batch's (create_templates_for_linker_generation re-pads, datasets.py:483-512)."""
    from difflinker_b200 import output
    from difflinker_b200.batching import create_templates_for_linker_generation
    spec = synthetic.SPECS["cfg1_plumbing"]
    data = collate(synthetic.make_items(spec))
    sizes = torch.tensor([9, 2, 12, 5])[:data['positions'].shape[0]]
    tpl = create_templates_for_linker_generation(data, sizes)
    n_old, n_new = data['positions'].shape[1], tpl['positions'].shape[1]
    assert n_old != n_new
    g = torch.Generator().manual_seed(6)
    chain0 = torch.randn((tpl['positions'].shape[0], n_new, 3 + spec.F), generator=g)
    positions = data['positions'] + torch.tensor([4.0, -2.0, 9.5])
    com_mask = data['fragment_mask']
    mean = (positions * com_mask).sum(1, keepdim=True) / com_mask.sum(1, keepdim=True)
    want = chain0[..., :3] + mean * tpl['atom_mask']                       # generate.py:167-171 verbatim
    got = output.restore_frame(chain0.clone().to(dev()), positions, com_mask, tpl['atom_mask']).cpu()
    assert rel_err(got[..., :3], want) <= 1e-6 and torch.equal(got[..., 3:], chain0[..., 3:])


@pytest.mark.parametrize("name", ["size_gnn_zinc", "size_gnn_zinc_bn"])
def test_size_classifier_matches_reference_golden(name):
    """SizeClassifier.forward(return_loss=False) (linker_size_lightning.py:83-110): native logits vs the live reference's
    (eval-mode batch norm folded on the host in the _bn case); then the sample_fn of generate.py:90-99."""
    meta, a = helpers.load_golden(name)
    model, data = helpers.build_size_classifier(meta)
    d = dev()
    dd = {k: (v.to(d) if torch.is_tensor(v) else v) for k, v in data.items()}
    out, loss = model.forward(dd, return_loss=False)
    assert loss is None and out.shape == a["logits"].shape
    assert rel_err(out.cpu(), a["logits"]) <= 1e-5
    out2, loss2 = model.forward(dd, return_loss=True)
    assert torch.equal(out2, out) and torch.isfinite(loss2)
    sizes = model.sample_sizes(dd, generator=torch.Generator(device=d).manual_seed(0))
    assert sizes.dtype == torch.int8 and sizes.shape == (meta["batch"],)
    assert set(sizes.tolist()) <= set(model.linker_id2size)


def test_size_classifier_vs_oracle_ragged_geom_with_pocket_mask():
    """9 atom types, with_pocket=True (fragment_only_mask selects the atoms), padded rows and isolated fragment atoms."""
    from difflinker_b200 import linker_size
    spec = synthetic.SPECS["cfg4_pockets"]
    small = synthetic.WorkloadSpec(spec.name, B=3, N=70, n_min=70, l_min=5, l_max=5, F=9, L=2, T=10, seed=21, pocket=50,
                                   graph_type=spec.graph_type)
    torch.manual_seed(3)
    model = linker_size.SizeClassifier(in_node_nf=9, out_node_nf=33, n_layers=2, normalization=None,
                                       linker_size2id=linker_size.GEOM_TRAIN_LINKER_SIZE2ID,
                                       linker_id2size=linker_size.GEOM_TRAIN_LINKER_ID2SIZE)
    synthetic.init_size_gnn_like_trained(model, 3)
    model.eval()
    data = linker_size.collate_with_fragment_edges(synthetic.make_items(small, batch=3))
    data['positions'][1, 3] += 40.0                                       # an isolated fragment atom (only its self loop)
    with torch.no_grad():
        want = orc.size_classifier_forward(model.state_dict(), data, 9, 2, None, with_pocket=True)
    d = dev()
    got, _ = model.forward({k: (v.to(d) if torch.is_tensor(v) else v) for k, v in data.items()}, return_loss=False,
                           with_pocket=True)
    assert rel_err(got.cpu(), want) <= 1e-5


@pytest.mark.parametrize("name", ["bonds_zinc", "bonds_geom"])
def test_bond_orders_match_reference_golden(name):
    """build_xae_molecule (molecule_builder.py:44-74) batched: integer output, bit-exact against the live reference's E for
    every molecule of the fixture (incl. n > 25 where torch.cdist uses its matmul formulation), padding rows all zero."""
    from difflinker_b200 import molecule_builder as mb
    meta, a = helpers.load_golden(name)
    d = dev()
    T = 9 if meta["is_geom"] else 8
    one_hot = torch.nn.functional.one_hot(a["types"], T).float()
    E = mb.bond_orders(one_hot.to(d), a["positions"].to(d), a["node_mask"].to(d), meta["is_geom"]).cpu()
    assert E.dtype == torch.int8 and torch.equal(E, a["E"])
    # chain[0]-style strided input and the single-molecule reference signature
    xh = torch.cat([a["positions"], one_hot], dim=2)
    assert torch.equal(mb.bond_orders(one_hot.to(d), xh.to(d), a["node_mask"].to(d), meta["is_geom"]).cpu(), a["E"])
    n = int(a["node_mask"][1].sum())
    X, A, E1 = mb.build_xae_molecule(a["positions"][1, :n].to(d), a["types"][1, :n].to(d), meta["is_geom"])
    assert torch.equal(E1.cpu().to(torch.int8), a["E"][1, :n, :n]) and torch.equal(A.cpu(), a["E"][1, :n, :n] != 0)


def test_draw_noise_on_cuda_equals_the_reference_call_sequence():
    """The sampler's own noise on the GPU is the reference's torch.randn call sequence (same seed -> same CUDA stream)."""
    spec = synthetic.SPECS["cfg1_plumbing"]
    ddpm, hp = helpers.build_ddpm(spec, 0)
    d = dev()
    g = torch.Generator(device=d).manual_seed(77)
    got = ddpm.edm.draw_noise(5, 4, 30, d, generator=g)
    g2 = torch.Generator(device=d).manual_seed(77)
    for r in range(5):
        assert torch.equal(got[r, :, :, :3], torch.randn((4, 30, 3), device=d, generator=g2))
        assert torch.equal(got[r, :, :, 3:], torch.randn((4, 30, spec.F), device=d, generator=g2))


def test_device_side_noise_stream_equals_torch_cuda_randn_sequence():
    """dl_noise_fill / dl_sample_chain_rng regenerate, from (seed, offset) alone, the numbers torch's CUDA generator hands to
    the reference's call sequence randn(B,N,3), randn(B,N,F), ... (utils.py:189-192): bit-identical, for shapes below and
    above one grid of 256-thread blocks per call, and from a non-zero starting offset."""
    import ctypes as C
    from difflinker_b200 import _native
    lib = _native.load_library()
    d = dev()
    for spec_name, B, N, n_draws, warm in (("cfg1_plumbing", 4, 30, 5, 0), ("cfg2_zinc", 256, 40, 3, 3), ("cfg3_geom", 512, 300, 2, 1)):
        spec = synthetic.SPECS[spec_name]
        dyn, hp = helpers.build_dynamics(spec, 0)
        eng = dyn.engine(d.index or 0)
        torch.manual_seed(1234 + B)
        for _ in range(warm):
            torch.randn((7, 13), device=d)                       # the stream does not start at offset 0
        gen = torch.cuda.default_generators[d.index or 0]
        seed, offset = gen.initial_seed(), gen.get_offset()
        out = torch.empty((n_draws, B, N, 3 + spec.F), device=d)
        used = C.c_uint64(0)
        with torch.cuda.device(d):
            _native.check(lib.dl_noise_fill(eng, n_draws, B, N, seed, offset, out.data_ptr(), C.byref(used),
                                            torch.cuda.current_stream(d).cuda_stream), "dl_noise_fill")
        for r in range(n_draws):
            assert torch.equal(out[r, :, :, :3], torch.randn((B, N, 3), device=d)), (spec_name, r)
            assert torch.equal(out[r, :, :, 3:], torch.randn((B, N, spec.F), device=d)), (spec_name, r)
        assert gen.get_offset() == offset + used.value


def test_sampler_with_device_side_noise_equals_sampler_fed_the_torch_tensor():
    """EDM.sample_chain on CUDA draws inside its kernels (no noise tensor); the chain equals, bit for bit, the one the same
    engine produces from the tensor torch.randn would have drawn for the same seed, and the generator ends at the same offset."""
    spec = synthetic.SPECS["cfg1_plumbing"]
    ddpm, hp = helpers.build_ddpm(spec, 0)
    d = dev()
    ddpm = ddpm.to(d)
    data = {k: (v.to(d) if torch.is_tensor(v) else v) for k, v in collate(synthetic.make_items(spec)).items()}
    torch.manual_seed(99)
    chain_dev, _ = ddpm.sample_chain(data, keep_frames=3)
    end_dev = torch.cuda.default_generators[d.index or 0].get_offset()
    torch.manual_seed(99)
    ddpm.edm.noise_mode = 'reference_tensor'
    chain_ten, _ = ddpm.sample_chain(data, keep_frames=3)
    assert torch.cuda.default_generators[d.index or 0].get_offset() == end_dev
    assert torch.equal(chain_dev, chain_ten)


def test_plain_c_caller_samples_the_chain_the_python_entry_produces(tmp_path):
    """SURVEY 8(b): the boundary is a C-ABI. examples/c_sampler.c -- C99, no Python, no torch, no noise tensor -- creates the engine,
    loads the weights under the reference's state_dict names, and samples with `dl_sample_chain_rng` from a Philox (seed, offset)
    pair; its chain equals, bit for bit, what `EDM.sample_chain` returns in Python for a torch generator in that state (which in turn
    is the reference's torch.randn call sequence, see the tests above), and it reports the same generator advance."""
    import subprocess
    from difflinker_b200 import export_job
    from difflinker_b200.ddpm import sampler_inputs
    spec = synthetic.SPECS["cfg2_zinc_ragged"]
    ddpm, hp = helpers.build_ddpm(spec, 0)
    ddpm.edm.T = 25
    d = dev()
    ddpm = ddpm.to(d)
    data = {k: (v.to(d) if torch.is_tensor(v) else v) for k, v in collate(synthetic.make_items(spec, batch=6)).items()}
    kw = sampler_inputs(ddpm, data)
    seed = 20240607
    torch.manual_seed(seed)
    gen = torch.cuda.default_generators[d.index or 0]
    off0 = gen.get_offset()
    want = ddpm.edm.sample_chain(**kw, keep_frames=3).cpu()
    job, out = str(tmp_path / "job.bin"), str(tmp_path / "out.bin")
    meta = export_job.write_job(job, ddpm.edm, **kw, keep_frames=3, seed=seed, offset=off0, device_index=d.index or 0)
    exe = helpers.build_c_example(tmp_path)
    res = subprocess.run([exe, job, out], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, (res.stdout, res.stderr)
    status, consumed, chain, flags = export_job.read_result(out, meta["B"], meta["N"], meta["keep_frames"], meta["xd"])
    assert status == 0 and not flags.any()
    assert consumed == gen.get_offset() - off0
    assert torch.equal(chain, want)


@pytest.mark.parametrize("world", [2, 3])
def test_batch_slices_reproduce_the_single_gpu_chain(world):
    """Strong scaling (SURVEY 8(e)), emulated on one GPU: the ranks' slices of a batch, each sampled with
    `batch_slice=(lo, B)` from the same generator state, concatenate to exactly the chain of the unsplit batch (the
    slice consumes the slice's rows of the full-batch noise; molecules never interact)."""
    from difflinker_b200.ddpm import sampler_inputs
    from difflinker_b200.distributed import shard_range, slice_sampler_inputs
    spec = synthetic.SPECS["cfg2_zinc_ragged"]
    ddpm, hp = helpers.build_ddpm(spec, 0)
    ddpm.edm.T = 12
    d = dev()
    ddpm = ddpm.to(d)
    data = {k: (v.to(d) if torch.is_tensor(v) else v) for k, v in collate(synthetic.make_items(spec, batch=7)).items()}
    torch.manual_seed(5)
    full, _ = ddpm.sample_chain(data, keep_frames=2)
    kw = sampler_inputs(ddpm, data)
    parts = []
    for r in range(world):
        lo, hi = shard_range(7, r, world)
        torch.manual_seed(5)
        parts.append(ddpm.edm.sample_chain(**slice_sampler_inputs(kw, lo, hi), keep_frames=2, batch_slice=(lo, 7)))
    assert torch.equal(torch.cat(parts, dim=1), full)



def test_bench_dumps_the_last_timed_step_reproducibly(tmp_path):
    """`bench.py --dump-outputs DIR` writes the results of its last timed step; with the same arguments the inputs are the same
    seeded ones, so two runs write identical arrays. `--steps` sets the number of timed sampler calls."""
    import json, os, subprocess, sys
    import numpy as np
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = synthetic.SPECS["cfg1_plumbing"]
    runs = []
    for r in range(2):
        out = tmp_path / f"run{r}"
        res = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--workload", spec.name, "--T", "10", "--steps", "2",
                              "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(out)], capture_output=True, text=True,
                             timeout=600)
        assert res.returncode == 0, res.stderr[-3000:]
        line = json.loads([l for l in res.stdout.splitlines() if l.startswith("{")][-1])
        assert line["steps"] == 2 and len(line["loop_ms_device"]) == 2
        runs.append({n: np.load(out / f"{n}.npy") for n in ("chain", "e2e_chain", "e2e_node_mask")})
    a, b = runs
    assert a["chain"].shape == (1, spec.B, spec.N, 3 + spec.F) and a["chain"].dtype == np.float32
    assert a["e2e_chain"].shape == a["chain"].shape and a["e2e_node_mask"].shape == (spec.B, spec.N, 1)
    assert np.isfinite(a["chain"]).all()
    for n in a:
        assert np.array_equal(a[n], b[n]), n
