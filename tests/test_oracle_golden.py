"""CPU: the oracle restatement against the golden vectors produced by the live reference
(oracle/make_golden.py), and the product's host-side mirrors against the oracle."""
import numpy as np
import pytest
import torch

from difflinker_b200 import batching, synthetic
from difflinker_b200.noise import PredefinedNoiseSchedule
from oracle import difflinker_oracle as orc
import dl_helpers as helpers

DYN_CASES = ["dyn_small_fc", "dyn_small_fc_tscalar", "dyn_cfg1", "dyn_small_geom_anchors",
             "dyn_small_pocket_FC-10A-4A", "dyn_small_pocket_FC-4A", "dyn_small_pocket_4A"]


@pytest.mark.parametrize("name", DYN_CASES)
def test_oracle_dynamics_matches_reference_golden(name):
    meta, a = helpers.load_golden(name)
    spec = helpers.spec_by_name(meta["spec"])
    dyn, hp = helpers.build_dynamics(spec, meta["seed"])
    assert helpers.state_sha(dyn.state_dict()) == meta["sha"], "seeded weights differ from the fixture's"
    with torch.no_grad():
        out = orc.dynamics_forward(dyn.state_dict(), helpers.oracle_cfg(hp), a["t"], a["xh"], a["node_mask"],
                                   a["linker_mask"], a["edge_mask"], a["context"])
    # same torch ops in the same order as the reference: bit-exact on the same torch build, tight otherwise
    assert (out - a["out"]).abs().max().item() <= 2e-6
    assert torch.equal(out * (1 - a["node_mask"].float()), torch.zeros_like(out))  # utils.py:99-101


@pytest.mark.parametrize("name", ["chain_cfg1", "chain_cfg1_nsteps20", "chain_small_pocket_FC-10A-4A",
                                  "chain_small_pocket_FC-4A", "chain_small_pocket_4A"])
def test_oracle_chain_matches_reference_golden(name):
    """(The T=500 chains at the benchmarked shapes -- chain_cfg2_zinc_T500 etc. -- were pinned against the oracle when they
    were generated, oracle/make_golden_r2.py; replaying them takes minutes of CPU, so here they only serve the GPU tests.)"""
    meta, a = helpers.load_golden(name)
    spec = helpers.spec_by_name(meta["spec"])
    ddpm, hp = helpers.build_ddpm(spec, meta["seed"], diffusion_steps=meta["table_timesteps"])
    assert helpers.state_sha(ddpm.edm.dynamics.state_dict()) == meta["sha"]
    data = orc.collate_molecules(synthetic.make_items(spec, batch=meta["batch"]))
    tpl = orc.linker_templates(data, data['linker_mask'].sum(1).view(-1).int())
    com = tpl['fragment_only_mask'] if spec.pocket else tpl['fragment_mask']   # lightning.py:441-444 (MOAD val_dataset)
    x = orc.remove_partial_mean(tpl['positions'], tpl['atom_mask'], com)
    gam = orc.gamma_table(hp['diffusion_noise_schedule'], hp['diffusion_steps'], hp['diffusion_noise_precision'])
    with torch.no_grad(), helpers.golden_threads():
        chain = orc.edm_sample_chain(ddpm.edm.dynamics.state_dict(), helpers.oracle_cfg(hp), gam, meta["T"], x,
                                     tpl['one_hot'], tpl['atom_mask'], tpl['fragment_mask'], tpl['linker_mask'],
                                     tpl['edge_mask'], helpers.context_of(tpl, spec), keep_frames=meta["keep_frames"],
                                     norm_values=tuple(hp['normalize_factors']),
                                     noise_fn=helpers.seeded_noise(meta["noise_seed"]))
    assert chain.shape == a["chain"].shape                              # (keep_frames,B,N,3+F)
    assert (chain - a["chain"]).abs().max().item() <= 5e-5
    assert torch.equal(chain[0][:, :, 3:], a["chain"][0][:, :, 3:])     # atom types identical


def test_oracle_inpainting_chain_matches_reference_golden():
    meta, a = helpers.load_golden("inpaint_chain_cfg1")
    spec = helpers.spec_by_name(meta["spec"])
    ddpm, hp = helpers.build_ddpm(spec, meta["seed"], inpainting=True)
    assert helpers.state_sha(ddpm.edm.dynamics.state_dict()) == meta["sha"]
    data = orc.collate_molecules(synthetic.make_items(spec, batch=meta["batch"]))
    x = orc.remove_partial_mean(data['positions'], data['atom_mask'], data['atom_mask'])   # lightning.py:417-419,438
    gam = orc.gamma_table(hp['diffusion_noise_schedule'], hp['diffusion_steps'], hp['diffusion_noise_precision'])
    ocfg = helpers.oracle_cfg(hp)
    ocfg.centering = True                                                                   # lightning.py:99
    with torch.no_grad(), helpers.golden_threads():
        chain = orc.inpainting_sample_chain(ddpm.edm.dynamics.state_dict(), ocfg, gam, meta["T"], x, data['one_hot'],
                                            data['atom_mask'], data['fragment_mask'], data['linker_mask'],
                                            data['edge_mask'], data['fragment_mask'], keep_frames=meta["keep_frames"],
                                            norm_values=tuple(hp['normalize_factors']),
                                            noise_fn=helpers.seeded_noise(meta["noise_seed"]))
    assert chain.shape == a["chain"].shape
    assert (chain - a["chain"]).abs().max().item() <= 5e-5
    assert torch.equal(chain[0][:, :, 3:], a["chain"][0][:, :, 3:])


@pytest.mark.parametrize("name", ["size_gnn_zinc", "size_gnn_zinc_bn"])
def test_oracle_size_classifier_matches_reference_golden(name):
    meta, a = helpers.load_golden(name)
    model, data = helpers.build_size_classifier(meta)
    assert helpers.state_sha(model.state_dict()) == meta["sha"]
    with torch.no_grad():
        out = orc.size_classifier_forward(model.state_dict(), data, model.in_node_nf, 3, meta["normalization"])
    assert out.shape == a["logits"].shape                               # (B, classes)
    assert (out - a["logits"]).abs().max().item() <= 2e-6 * max(1.0, a["logits"].abs().max().item())


@pytest.mark.parametrize("name", ["bonds_zinc", "bonds_geom"])
def test_oracle_bond_orders_match_reference_golden(name):
    from difflinker_b200 import molecule_builder as mb, output
    meta, a = helpers.load_golden(name)
    idx2atom = output.GEOM_IDX2ATOM if meta["is_geom"] else output.IDX2ATOM
    for b in range(a["positions"].shape[0]):
        n = int(a["node_mask"][b].sum())
        _, A, E = orc.xae_molecule(a["positions"][b, :n], a["types"][b, :n], idx2atom, mb.SINGLE, mb.DOUBLE, mb.TRIPLE,
                                   mb.MARGINS_EDM)
        assert torch.equal(E.to(torch.int8), a["E"][b, :n, :n]) and torch.equal(A, E.bool())
    # host threshold tables: [min type][max type], -1 where the reference's dictionaries have no entry
    t1, t2, t3 = mb.threshold_tables(meta["is_geom"])
    assert t1[0, 0] == 164 and t2[0, 0] == 139 and t3[0, 0] == 122          # C-C: 154+10, 134+5, 120+2
    assert t1[5, 7] == -1 and t1[6, 7] == -1                                 # Cl-I, Br-I: no typical bond length
    lower = torch.tril(torch.ones_like(t1), -1).bool()
    assert (t1[lower] == -1).all()                                           # only the index-ordered direction is ever read


def test_gamma_tables_match_reference_golden():
    _, a = helpers.load_golden("gamma_tables")
    for key, ref in a.items():
        sched, T, prec = key.split("__")
        assert torch.equal(orc.gamma_table(sched, int(T), float(prec)), ref), key
        assert torch.equal(PredefinedNoiseSchedule(sched, int(T), float(prec)).gamma.detach(), ref), key


@pytest.mark.parametrize("name", ["chain_cfg1", "chain_cfg1_nsteps20"])
def test_step_coefficients_match_reference_golden(name):
    meta, a = helpers.load_golden(name)
    spec = helpers.spec_by_name(meta["spec"])
    ddpm, hp = helpers.build_ddpm(spec, meta["seed"])
    ddpm.edm.T = meta["T"]                                              # --n_steps override, generate.py:103-104
    rows = ddpm.edm.step_coefficients(meta["keep_frames"], meta["batch"])
    got = np.array([[r.t, r.a, r.b, r.c] for r in rows], dtype=np.float32)
    assert np.array_equal(got, a["coef"].numpy())
    T, keep = meta["T"], meta["keep_frames"]
    # frame bookkeeping (edm.py:162): every frame > 0 has exactly one last writer, frame 0 belongs to the final step
    frames = [rows[r].frame for r in range(T)]
    for f in range(1, keep):
        writers = [T - 1 - r for r in range(T) if frames[r] == f]
        assert writers == [min(s for s in range(T) if (s * keep) // T == f)]
    assert all(f != 0 for f in frames) and rows[T].frame == -1


def test_inpainting_step_coefficients_and_noise_order_match_the_oracle():
    """InpaintingEDM host side: q(z_s|z_t,x) coefficients (edm.py:655-668, 716), chain-frame bookkeeping (edm.py:596-598: every
    step writes its frame after the COM projection, the last writer wins, chain[0] is overwritten at the end) and the order of
    the prepared noise slabs (edm.py:565,645,669,689,706)."""
    meta, a = helpers.load_golden("inpaint_chain_cfg1")
    spec = helpers.spec_by_name(meta["spec"])
    ddpm, hp = helpers.build_ddpm(spec, meta["seed"], inpainting=True)
    T, keep, B = meta["T"], meta["keep_frames"], meta["batch"]
    rows = ddpm.edm.step_coefficients(keep, B)
    gam = orc.gamma_table(hp['diffusion_noise_schedule'], hp['diffusion_steps'], hp['diffusion_noise_precision'])
    for r in range(T):
        s = T - 1 - r
        s_arr = torch.full((B, 1), fill_value=s)
        t_arr = (s_arr + 1) / T
        s_arr = s_arr / T
        g_s, g_t = orc.gamma_lookup(gam, s_arr, T), orc.gamma_lookup(gam, t_arr, T)
        sig2_ts, sig_ts, a_ts = orc._sigma_alpha_t_given_s(g_t, g_s)
        sig_s, sig_t, al_s = orc._sigma(g_s), orc._sigma(g_t), orc._alpha(g_s)
        assert rows[r].qa == float((a_ts * (sig_s ** 2) / (sig_t ** 2))[0])
        assert rows[r].qb == float((al_s * sig2_ts / (sig_t ** 2))[0])
        assert rows[r].a == float(a_ts[0]) and rows[r].c == float((sig_ts * sig_s / sig_t)[0])
    g0 = orc.gamma_lookup(gam, torch.zeros((B, 1)), T)
    assert rows[T].qa == float((orc._sigma(g0) / orc._alpha(g0))[0])
    frames = [rows[r].frame for r in range(T)]
    for f in range(1, keep):
        assert [T - 1 - r for r in range(T) if frames[r] == f] == [min(s for s in range(T) if (s * keep) // T == f)]
    assert all(f != 0 for f in frames)
    # prepared noise: same generator -> the slabs the GPU test injects
    from difflinker_b200.batching import collate
    data = collate(synthetic.make_items(spec, batch=B))
    N = data['positions'].shape[1]
    g = torch.Generator().manual_seed(meta["noise_seed"])
    got = ddpm.edm.draw_noise_inpaint(B, N, torch.device('cpu'), data['atom_mask'], data['fragment_mask'], generator=g)
    want = helpers.inpaint_noise_tensor(meta["noise_seed"], T, B, N, spec.F, data['atom_mask'], data['fragment_mask'])
    assert got.shape == (2 * T + 3, B, N, 3 + spec.F) and torch.equal(got, want)


@pytest.mark.parametrize("spec_name,nb", [("cfg1_plumbing", 4), ("cfg2_zinc_ragged", 6), ("cfg4_pockets", 2)])
def test_batching_matches_oracle_contract(spec_name, nb):
    spec = synthetic.SPECS[spec_name]
    items = synthetic.make_items(spec, batch=nb)
    mine, ora = batching.collate(items), orc.collate_molecules(items)
    for k, v in ora.items():
        if torch.is_tensor(v):
            assert v.dtype == mine[k].dtype and torch.equal(v, mine[k]), k
    assert mine['atom_mask'].dtype == torch.int8 and mine['edge_mask'].dtype == torch.int8
    if not spec.pocket:
        assert sorted(mine['edge_mask'].unique().tolist()) == [-2, -1, 0][-len(mine['edge_mask'].unique()):]
        em = mine['edge_mask'].view(nb, spec.N, spec.N)
        n0 = int(mine['atom_mask'][0].sum())
        assert int(em[0].diagonal()[:n0].min()) == -2 and int(em[0].diagonal()[:n0].max()) == -2  # live self loops
    sizes = mine['linker_mask'].sum(1).view(-1).int() + 2
    mt = batching.create_templates_for_linker_generation(mine, sizes)
    ot = orc.linker_templates(ora, sizes)
    for k, v in ot.items():
        if torch.is_tensor(v):
            assert torch.equal(v, mt[k]), k
    assert torch.equal(mt['linker_mask'].sum(1).view(-1).int(), sizes)


def test_empty_linker_and_single_atom_edge_cases():
    # a molecule whose requested linker size is 0 and a one-atom fragment still collate
    items = [dict(uuid=0, name='a', positions=torch.randn(1, 3), one_hot=torch.eye(8)[:1], anchors=torch.ones(1),
                  fragment_mask=torch.ones(1), linker_mask=torch.zeros(1), num_atoms=1),
             dict(uuid=1, name='b', positions=torch.randn(4, 3), one_hot=torch.eye(8)[:4], anchors=torch.zeros(4),
                  fragment_mask=torch.tensor([1., 1, 0, 0]), linker_mask=torch.tensor([0., 0, 1, 1]), num_atoms=4)]
    b = batching.collate(items)
    assert b['positions'].shape == (2, 4, 3) and b['edge_mask'].shape == (2 * 16, 1)
    t = batching.create_templates_for_linker_generation(b, [0, 3])
    assert t['positions'].shape == (2, 5, 3)
    assert t['atom_mask'][0].sum() == 1 and t['atom_mask'][1].sum() == 5
