"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/*.npz from the LIVE, UNMODIFIED reference (/root/reference,
build container only) and, in the same run, pins oracle/difflinker_oracle.py and the product's host-side mirrors
(batching, noise schedule, step coefficients) against it.  Run:  python -m oracle.make_golden

Weights are not stored: fixtures record the torch seed and a sha256 of the resulting reference state_dict;
difflinker_b200.Dynamics constructs its parameters in the reference's order, so the same seed reproduces them
(tests verify the sha256 before trusting a fixture).
"""
import hashlib
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from difflinker_b200 import batching, synthetic  # noqa: E402
from difflinker_b200.edm import EDM as NativeEDM  # noqa: E402
from difflinker_b200.egnn import Dynamics as NativeDynamics  # noqa: E402
from oracle import difflinker_oracle as orc  # noqa: E402
from oracle.ref_loader import load_reference  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def state_sha(sd) -> str:
    h = hashlib.sha256()
    for k, v in sd.items():
        h.update(k.encode())
        h.update(v.detach().cpu().float().contiguous().numpy().tobytes())
    return h.hexdigest()


def seeded_noise(seed):
    g = torch.Generator().manual_seed(seed)
    return lambda shape: torch.randn(tuple(shape), generator=g)


def build_ref_dynamics(ns, spec, seed, pocket=False):
    hp = synthetic.model_hparams(spec)
    torch.manual_seed(seed)
    cls = ns.egnn.DynamicsWithPockets if pocket else ns.egnn.Dynamics
    dyn = cls(in_node_nf=hp['in_node_nf'], n_dims=3, context_node_nf=hp['context_node_nf'], hidden_nf=128,
              n_layers=hp['n_layers'], norm_constant=hp['norm_constant'], inv_sublayers=hp['inv_sublayers'],
              normalization_factor=hp['normalization_factor'], graph_type=hp['graph_type'])
    synthetic.init_reference_like_weights(dyn)
    return dyn.eval(), hp


def oracle_cfg(hp):
    return orc.OracleConfig(in_node_nf=hp['in_node_nf'], context_node_nf=hp['context_node_nf'], n_layers=hp['n_layers'],
                            inv_sublayers=hp['inv_sublayers'], norm_constant=hp['norm_constant'],
                            normalization_factor=hp['normalization_factor'], graph_type=hp['graph_type'])


def context_of(batch, spec):
    if spec.pocket:
        fo = batch['fragment_only_mask']
        parts = [fo, batch['fragment_mask'] - fo]
    else:
        parts = [batch['fragment_mask']]
    if spec.anchors_context:                                       # lightning.py:425-438
        parts = [batch['anchors']] + parts
    return torch.cat(parts, dim=-1)


def save(name, meta, **arrays):
    os.makedirs(OUT, exist_ok=True)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), meta=json.dumps(meta),
                        **{k: (v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in arrays.items()})
    print(f"  wrote {name}.npz  ({meta})")


def check_batching(ns, spec, nb):
    items = synthetic.make_items(spec, batch=nb)
    ref = ns.datasets.collate(items)
    mine = batching.collate(items)
    ora = orc.collate_molecules(items)
    for k, v in ref.items():
        if torch.is_tensor(v):
            assert v.dtype == mine[k].dtype and torch.equal(v, mine[k]), f"collate mismatch {k}"
            assert v.dtype == ora[k].dtype and torch.equal(v, ora[k]), f"oracle collate mismatch {k}"
    sizes = ref['linker_mask'].sum(1).view(-1).int() + 1
    rt = ns.datasets.create_templates_for_linker_generation(ref, sizes)
    mt = batching.create_templates_for_linker_generation(mine, sizes)
    ot = orc.linker_templates(ora, sizes)
    for k, v in rt.items():
        if torch.is_tensor(v):
            assert v.dtype == mt[k].dtype and torch.equal(v, mt[k]), f"template mismatch {k}"
            assert torch.equal(v, ot[k]), f"oracle template mismatch {k}"
    return ref


def golden_dynamics(ns, name, spec, nb, seed, pocket=False, t_scalar=False):
    dyn, hp = build_ref_dynamics(ns, spec, seed, pocket)
    batch = check_batching(ns, spec, nb)
    g = torch.Generator().manual_seed(seed + 7)
    B, N = batch['positions'].shape[:2]
    com = batch['fragment_only_mask'] if spec.pocket else batch['fragment_mask']
    x = ns.utils.remove_partial_mean_with_mask(batch['positions'], batch['atom_mask'], com)
    assert torch.allclose(x, orc.remove_partial_mean(batch['positions'], batch['atom_mask'], com))
    # a mid-trajectory latent: fragments clean, linker noised; garbage on padding rows to exercise the masking
    z = torch.cat([x, batch['one_hot'] / 4], dim=2)
    z = z * batch['fragment_mask'] + torch.randn(z.shape, generator=g) * batch['linker_mask']
    z = z + 3.0 * torch.randn(z.shape, generator=g) * (1 - batch['atom_mask'].float())
    t = torch.full((1,), 0.37) if t_scalar else torch.rand((B, 1), generator=g)
    ctx = context_of(batch, spec)
    with torch.no_grad():
        out = dyn(t, z, batch['atom_mask'], batch['linker_mask'], batch['edge_mask'], ctx)
        sd = dyn.state_dict()
        o2 = orc.dynamics_forward(sd, oracle_cfg(hp), t, z, batch['atom_mask'], batch['linker_mask'],
                                  batch['edge_mask'], ctx)
    err = (out - o2).abs().max().item()
    assert err < 2e-6, f"{name}: oracle vs reference {err}"
    torch.manual_seed(seed)
    mine = NativeDynamics(in_node_nf=hp['in_node_nf'], n_dims=3, context_node_nf=hp['context_node_nf'], hidden_nf=128,
                          n_layers=hp['n_layers'], norm_constant=hp['norm_constant'], inv_sublayers=hp['inv_sublayers'],
                          normalization_factor=hp['normalization_factor'], graph_type=hp['graph_type']) \
        if not pocket else None
    if mine is not None:
        synthetic.init_reference_like_weights(mine)
        assert state_sha(mine.state_dict()) == state_sha(sd), "native parameter construction order diverged"
    meta = dict(kind="dynamics", spec=spec.name, batch=nb, seed=seed, pocket=pocket, sha=state_sha(sd),
                oracle_max_abs_err=err, graph_type=hp['graph_type'])
    save(name, meta, t=t, xh=z, node_mask=batch['atom_mask'], linker_mask=batch['linker_mask'],
         edge_mask=batch['edge_mask'], context=ctx, out=out)


def golden_chain(ns, name, spec, nb, seed, keep_frames, n_steps=None, moad_val_dataset=False):
    hp = synthetic.model_hparams(spec)
    torch.manual_seed(seed)
    ddpm = ns.lightning.DDPM(**hp, data_path=None, batch_size=nb, lr=1e-4, torch_device='cpu', test_epochs=1,
                             n_stability_samples=1)
    synthetic.init_reference_like_weights(ddpm)
    ddpm.eval()
    if n_steps is not None:
        ddpm.edm.T = n_steps                                       # generate.py:103-104
    T = ddpm.edm.T
    if moad_val_dataset:                                           # generate_with_pocket.py:249-250
        ddpm.val_dataset = ns.datasets.MOADDataset(data=synthetic.make_items(spec, batch=nb))
    data = ns.datasets.collate(synthetic.make_items(spec, batch=nb))
    noise_seed = seed + 1000
    draw = seeded_noise(noise_seed)
    orig = ns.utils.sample_gaussian_with_mask
    ns.utils.sample_gaussian_with_mask = lambda size, device, node_mask: draw(size) * node_mask
    try:
        with torch.no_grad():
            chain, node_mask = ddpm.sample_chain(data, keep_frames=keep_frames)
    finally:
        ns.utils.sample_gaussian_with_mask = orig
    # oracle replay with the same draws
    tpl = orc.linker_templates(orc.collate_molecules(synthetic.make_items(spec, batch=nb)),
                               data['linker_mask'].sum(1).view(-1).int())
    ctx = context_of(tpl, spec)
    com = tpl['fragment_only_mask'] if spec.pocket else tpl['fragment_mask']
    x = orc.remove_partial_mean(tpl['positions'], tpl['atom_mask'], com)
    sd_dyn = {k[len("edm.dynamics."):]: v for k, v in ddpm.state_dict().items() if k.startswith("edm.dynamics.")}
    gam = orc.gamma_table(hp['diffusion_noise_schedule'], hp['diffusion_steps'], hp['diffusion_noise_precision'])
    assert torch.equal(gam, ddpm.edm.gamma.gamma.detach()), "oracle gamma table differs"
    with torch.no_grad():
        oc = orc.edm_sample_chain(sd_dyn, oracle_cfg(hp), gam, T, x, tpl['one_hot'], tpl['atom_mask'],
                                  tpl['fragment_mask'], tpl['linker_mask'], tpl['edge_mask'], ctx,
                                  keep_frames=keep_frames, norm_values=tuple(hp['normalize_factors']),
                                  noise_fn=seeded_noise(noise_seed))
    err = (oc - chain).abs().max().item()
    assert err < 5e-5, f"{name}: oracle chain vs reference {err}"
    assert torch.equal(oc[0][:, :, 3:], chain[0][:, :, 3:]), "atom types differ"
    # native host-side scalars vs the reference's own
    nat = NativeEDM(dynamics=None, in_node_nf=hp['in_node_nf'], n_dims=3, timesteps=hp['diffusion_steps'],
                    noise_schedule=hp['diffusion_noise_schedule'], noise_precision=hp['diffusion_noise_precision'],
                    loss_type='l2', norm_values=hp['normalize_factors'])
    assert torch.equal(nat.gamma.gamma, ddpm.edm.gamma.gamma)
    nat.T = T
    rows = nat.step_coefficients(keep_frames, nb)
    edm = ddpm.edm
    coef = np.zeros((T + 1, 4), dtype=np.float32)
    for r in range(T):
        s = T - 1 - r
        s_arr = torch.full((nb, 1), fill_value=s) / T
        t_arr = (torch.full((nb, 1), fill_value=s) + 1) / T
        gs, gt = edm.gamma(s_arr), edm.gamma(t_arr)
        zt = torch.zeros(nb, 1, 1)
        s2, sts, ats = edm.sigma_and_alpha_t_given_s(gt, gs, zt)
        sig_s, sig_t = edm.sigma(gs, zt), edm.sigma(gt, zt)
        coef[r] = [t_arr[0].item(), ats[0].item(), (s2 / ats / sig_t)[0].item(), (sts * sig_s / sig_t)[0].item()]
        got = [rows[r].t, rows[r].a, rows[r].b, rows[r].c]
        assert np.array_equal(coef[r], np.array(got, dtype=np.float32)), (r, coef[r], got)
    g0 = edm.gamma(torch.zeros(nb, 1))
    zt = torch.zeros(nb, 1, 1)
    coef[T] = [0.0, (1. / edm.alpha(g0, zt))[0].item(), edm.sigma(g0, zt)[0].item(), edm.SNR(-0.5 * g0)[0].item()]
    assert np.array_equal(coef[T], np.array([rows[T].t, rows[T].a, rows[T].b, rows[T].c], dtype=np.float32))
    meta = dict(kind="chain", spec=spec.name, batch=nb, seed=seed, noise_seed=noise_seed, keep_frames=keep_frames,
                T=T, table_timesteps=hp['diffusion_steps'], sha=state_sha(ddpm.edm.dynamics.state_dict()),
                oracle_max_abs_err=err, moad_val_dataset=bool(moad_val_dataset))
    save(name, meta, chain=chain, node_mask=node_mask, coef=coef)


def golden_inpaint_chain(ns, name, spec, nb, seed, keep_frames):
    """InpaintingEDM through the reference's DDPM.sample_chain (lightning.py:405-463 with inpainting=True)."""
    hp = synthetic.model_hparams(spec)
    hp['inpainting'] = True
    torch.manual_seed(seed)
    ddpm = ns.lightning.DDPM(**hp, data_path=None, batch_size=nb, lr=1e-4, torch_device='cpu', test_epochs=1,
                             n_stability_samples=1)
    synthetic.init_reference_like_weights(ddpm)
    ddpm.eval()
    T = ddpm.edm.T
    data = ns.datasets.collate(synthetic.make_items(spec, batch=nb))
    noise_seed = seed + 2000
    draw = seeded_noise(noise_seed)
    o1, o2 = ns.utils.sample_gaussian_with_mask, ns.utils.sample_center_gravity_zero_gaussian_with_mask
    ns.utils.sample_gaussian_with_mask = lambda size, device, node_mask: draw(size) * node_mask
    ns.utils.sample_center_gravity_zero_gaussian_with_mask = \
        lambda size, device, node_mask: ns.utils.remove_mean_with_mask(draw(size) * node_mask, node_mask)
    try:
        with torch.no_grad():
            chain, node_mask = ddpm.sample_chain(data, keep_frames=keep_frames)
    finally:
        ns.utils.sample_gaussian_with_mask, ns.utils.sample_center_gravity_zero_gaussian_with_mask = o1, o2
    d2 = orc.collate_molecules(synthetic.make_items(spec, batch=nb))
    x = orc.remove_partial_mean(d2['positions'], d2['atom_mask'], d2['atom_mask'])
    sd_dyn = {k[len("edm.dynamics."):]: v for k, v in ddpm.state_dict().items() if k.startswith("edm.dynamics.")}
    gam = orc.gamma_table(hp['diffusion_noise_schedule'], hp['diffusion_steps'], hp['diffusion_noise_precision'])
    ocfg = oracle_cfg(hp)
    ocfg.centering = True
    with torch.no_grad():
        oc = orc.inpainting_sample_chain(sd_dyn, ocfg, gam, T, x, d2['one_hot'], d2['atom_mask'], d2['fragment_mask'],
                                         d2['linker_mask'], d2['edge_mask'], d2['fragment_mask'], keep_frames=keep_frames,
                                         norm_values=tuple(hp['normalize_factors']), noise_fn=seeded_noise(noise_seed))
    err = (oc - chain).abs().max().item()
    assert err < 5e-5, f"{name}: oracle inpainting chain vs reference {err}"
    meta = dict(kind="inpaint_chain", spec=spec.name, batch=nb, seed=seed, noise_seed=noise_seed, keep_frames=keep_frames,
                T=T, sha=state_sha(ddpm.edm.dynamics.state_dict()), oracle_max_abs_err=err)
    save(name, meta, chain=chain, node_mask=node_mask)


def golden_size_classifier(ns):
    """SizeClassifier.forward(return_loss=False) of the live reference (linker_size_lightning.py:83-110) on batches built by
    the reference's collate_with_fragment_edges; pins oracle.size_classifier_forward and the host mirror's parameter
    layout / collate."""
    import importlib
    from difflinker_b200 import linker_size as mine
    lsl = importlib.import_module("src.linker_size_lightning")
    for name, spec, nb, normalization, seed in (("size_gnn_zinc", synthetic.SPECS["cfg1_plumbing"], 4, None, 5),
                                                ("size_gnn_zinc_bn", synthetic.SPECS["cfg2_zinc_ragged"], 6, "batch_norm", 6)):
        out_nf = len(ns.const.ZINC_TRAIN_LINKER_ID2SIZE)
        torch.manual_seed(seed)
        ref = lsl.SizeClassifier(None, None, None, in_node_nf=spec.F, hidden_nf=128, out_node_nf=out_nf, n_layers=3,
                                 batch_size=nb, lr=1e-3, torch_device='cpu', normalization=normalization)
        torch.manual_seed(seed)
        host = mine.SizeClassifier(in_node_nf=spec.F, hidden_nf=128, out_node_nf=out_nf, n_layers=3, normalization=normalization)
        assert list(ref.state_dict().keys()) == list(host.state_dict().keys()), name
        for k, v in ref.state_dict().items():
            assert torch.equal(v, host.state_dict()[k]), (name, k)
        synthetic.init_size_gnn_like_trained(ref, seed)
        ref.eval()
        items = synthetic.make_items(spec, batch=nb)
        data = ns.datasets.collate_with_fragment_edges(items)
        mydata = mine.collate_with_fragment_edges(items)
        assert torch.equal(data['edge_mask'], mydata['edge_mask']) and torch.equal(data['edges'][0], mydata['edges'][0]) \
            and torch.equal(data['edges'][1], mydata['edges'][1]), name
        with torch.no_grad():
            out, loss = ref.forward(data, return_loss=False)
            ora = orc.size_classifier_forward(ref.state_dict(), data, spec.F, 3, normalization)
        err = (out - ora).abs().max().item()
        assert err <= 1e-6 * max(1.0, out.abs().max().item()), f"{name}: oracle vs reference {err}"
        save(name, dict(kind="size_gnn", spec=spec.name, batch=nb, seed=seed, normalization=normalization, out_nf=out_nf,
                        sha=state_sha(ref.state_dict()), oracle_max_abs_err=err), logits=out)


def golden_bonds(ns):
    """molecule_builder.build_xae_molecule of the live reference on chain-like random molecules (bonded distances around
    1.1-1.6 A so that all of single / double / triple / none occur); pins oracle.xae_molecule and the host tables."""
    import importlib
    from difflinker_b200 import molecule_builder as mb
    ref = importlib.import_module("src.molecule_builder")
    g = torch.Generator().manual_seed(99)
    for name, is_geom, T in (("bonds_zinc", False, 8), ("bonds_geom", True, 9)):
        idx2atom = ns.const.GEOM_IDX2ATOM if is_geom else ns.const.IDX2ATOM
        mols = []
        for n in (5, 17, 30, 41):                    # > 25 atoms: torch.cdist switches to the matmul formulation
            step = torch.randn((n, 3), generator=g)
            step = step / step.norm(dim=1, keepdim=True) * (1.05 + 0.6 * torch.rand((n, 1), generator=g))
            pos = torch.cumsum(step, dim=0)
            types = torch.randint(0, T, (n,), generator=g)
            types[torch.rand((n,), generator=g) < 0.5] = 0                   # mostly carbon
            X, A, E = ref.build_xae_molecule(pos, types, is_geom=is_geom)
            oX, oA, oE = orc.xae_molecule(pos, types, idx2atom, mb.SINGLE, mb.DOUBLE, mb.TRIPLE, mb.MARGINS_EDM)
            assert torch.equal(E, oE) and torch.equal(A, oA), name
            mols.append((pos, types, E))
        N = max(m[0].shape[0] for m in mols)
        P = torch.zeros((len(mols), N, 3)); Ty = torch.zeros((len(mols), N), dtype=torch.long)
        M = torch.zeros((len(mols), N), dtype=torch.int8); Eb = torch.zeros((len(mols), N, N), dtype=torch.int8)
        for b, (pos, types, E) in enumerate(mols):
            n = pos.shape[0]
            P[b, :n] = pos; Ty[b, :n] = types; M[b, :n] = 1; Eb[b, :n, :n] = E.to(torch.int8)
        counts = [int((Eb == k).sum()) for k in range(4)]
        assert min(counts[1:]) > 0, counts
        save(name, dict(kind="bonds", is_geom=is_geom, counts=counts), positions=P, types=Ty, node_mask=M, E=Eb)


def golden_xyz(ns):
    """visualizer.save_xyz_file (visualizer.py:14-31) run for real into a temp dir; its files pin oracle.xyz_text."""
    import importlib
    import tempfile
    vis = importlib.import_module("src.visualizer")
    g = torch.Generator().manual_seed(77)
    for name, is_geom, F in (("xyz_zinc", False, 8), ("xyz_geom", True, 9)):
        B, N = 5, 13
        pos = torch.randn((B, N, 3), generator=g) * torch.tensor([1.0, 30.0, 1e-4])
        pos[0, 0] = torch.tensor([0.0, -0.0, 1.0])
        pos[0, 1] = torch.tensor([0.5e-9, 1.5e-9, 2.5e-9])             # rounding at the last printed digit
        pos[0, 2] = torch.tensor([123456.789, -98765.4321, 3.4e38])
        pos[0, 3] = torch.tensor([1e-10, -1e-10, 0.9999999995])
        pos[1, 0] = torch.tensor([float('nan'), float('inf'), float('-inf')])
        types = torch.randint(0, F, (B, N), generator=g)
        one_hot = torch.nn.functional.one_hot(types, F).float()
        n_valid = torch.tensor([13, 7, 1, 9, 4])
        node_mask = (torch.arange(N)[None, :] < n_valid[:, None]).to(torch.int8).unsqueeze(-1)
        node_mask[3, 2] = 0                                            # holes in the mask, not just padding
        names = [f"m{b}" for b in range(B)]
        with tempfile.TemporaryDirectory() as d:
            vis.save_xyz_file(d, one_hot, pos, node_mask, names=names, is_geom=is_geom, suffix='s')
            texts = [open(f"{d}/{n}_s.xyz").read() for n in names]
        idx2atom = ns.const.GEOM_IDX2ATOM if is_geom else ns.const.IDX2ATOM
        assert texts == orc.xyz_text(one_hot, pos, node_mask, idx2atom), name
        blob = "".join(texts).encode()
        offs = [0]
        for t in texts:
            offs.append(offs[-1] + len(t.encode()))
        save(name, dict(kind="xyz", is_geom=is_geom), positions=pos, one_hot=one_hot, node_mask=node_mask,
             text=torch.tensor(list(blob), dtype=torch.uint8), offsets=torch.tensor(offs))


def golden_reference_edm(ns, spec, seed=3):
    """The EDM of a freshly constructed reference DDPM (lightning.py:41-112): its state_dict keys in order, their shapes,
    a sha256 of the values and its T. `accelerate()` replaces exactly this module, so the test rebuilds it from these
    records; the native DDPM draws the same values for the same seed (asserted here)."""
    from difflinker_b200.ddpm import DDPM as NativeDDPM
    hp = synthetic.model_hparams(spec)
    torch.manual_seed(seed)
    ref = ns.lightning.DDPM(**hp, data_path=None, batch_size=2, lr=1e-4, torch_device='cpu', test_epochs=1,
                            n_stability_samples=1)
    sd = ref.edm.state_dict()
    torch.manual_seed(seed)
    mine = NativeDDPM(**hp).edm.state_dict()
    assert list(mine) == list(sd) and all(torch.equal(mine[k], v) for k, v in sd.items()), "native EDM construction diverged"
    save("ref_edm_small_fc", dict(kind="reference_edm", spec=spec.name, seed=seed, T=ref.edm.T, cls=type(ref.edm).__name__,
                                  keys=list(sd), shapes=[list(v.shape) for v in sd.values()], sha=state_sha(sd)))


def golden_schedules():
    ns = load_reference()
    arrs = {}
    for sched, T, prec in [("polynomial_2", 500, 1e-5), ("polynomial_2", 1000, 1e-5), ("polynomial_3", 100, 1e-4),
                           ("cosine", 200, 1e-4)]:
        ref = ns.noise.PredefinedNoiseSchedule(sched, timesteps=T, precision=prec).gamma.detach()
        assert torch.equal(ref, orc.gamma_table(sched, T, prec)), (sched, T)
        arrs[f"{sched}__{T}__{prec}"] = ref
    save("gamma_tables", dict(kind="gamma"), **arrs)


def main():
    torch.set_num_threads(8)
    ns = load_reference()
    S = synthetic.SPECS
    print("golden vectors from the live reference:")
    golden_schedules()
    small = synthetic.WorkloadSpec("small_fc", B=3, N=12, n_min=7, l_min=2, l_max=4, F=8, L=2, T=20, seed=11)
    golden_dynamics(ns, "dyn_small_fc", small, 3, seed=0)
    golden_dynamics(ns, "dyn_small_fc_tscalar", small, 3, seed=1, t_scalar=True)
    golden_reference_edm(ns, small)
    golden_dynamics(ns, "dyn_cfg1", S["cfg1_plumbing"], 4, seed=0)
    geom = synthetic.WorkloadSpec("small_geom", B=5, N=23, n_min=11, l_min=1, l_max=9, F=9, L=3, T=20, seed=12,
                                  anchors_context=True)
    golden_dynamics(ns, "dyn_small_geom_anchors", geom, 5, seed=2)
    for gt in ("FC-10A-4A", "FC-4A", "4A"):
        pk = synthetic.WorkloadSpec(f"small_pocket_{gt}", B=2, N=70, n_min=70, l_min=5, l_max=5, F=9, L=2, T=20,
                                    seed=13, pocket=50, graph_type=gt)
        golden_dynamics(ns, f"dyn_small_pocket_{gt}", pk, 2, seed=3, pocket=True)
    golden_chain(ns, "chain_cfg1", S["cfg1_plumbing"], 4, seed=0, keep_frames=5)
    golden_chain(ns, "chain_cfg1_nsteps20", S["cfg1_plumbing"], 4, seed=0, keep_frames=1, n_steps=20)
    golden_inpaint_chain(ns, "inpaint_chain_cfg1", S["cfg1_plumbing"], 4, seed=0, keep_frames=3)
    golden_xyz(ns)
    golden_bonds(ns)
    golden_size_classifier(ns)
    print("all oracle / host-mirror checks against the reference passed")


if __name__ == "__main__":
    main()
