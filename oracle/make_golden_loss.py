"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/loss_*.npz: the diffusion objective (EDM.forward, src/edm.py:41-124)
as the LIVE, UNMODIFIED reference computes it through DDPM.validation_step (src/lightning.py:228-247), and pins
oracle.loss_oracle.edm_loss_terms and the native per-molecule scalar table (EDM.loss_coefficients) against it.
Build container only (needs /root/reference). Run:  python -m oracle.make_golden_loss
make_golden.py's fixtures are not touched.

torch.randint (edm.py:49) and utils.sample_gaussian_with_mask (edm.py:67, utils.py:189-192) are patched to chosen
timesteps and seeded draws, as make_golden.golden_chain does for the sampler; the fixtures record both (the draws
unmasked), the seven outputs, the oracle's per-molecule terms, the reference's per-molecule scalars and the sha256 of the
state_dict (weights are rebuilt from the seed, see make_golden.py).
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from difflinker_b200 import synthetic  # noqa: E402
from difflinker_b200.edm import EDM as NativeEDM  # noqa: E402
from oracle import difflinker_oracle as orc  # noqa: E402
from oracle.loss_oracle import edm_loss_terms  # noqa: E402
from oracle.make_golden import context_of, oracle_cfg, save, seeded_noise, state_sha  # noqa: E402
from oracle.ref_loader import load_reference  # noqa: E402

OUTPUTS = ("delta_log_px", "kl_prior", "loss_term_t", "loss_term_0", "l2_loss", "noise_t", "noise_0")
COEF_ROWS = ("t", "alpha_t", "sigma_t", "alpha_1", "sigma2_1", "log_inv_sigma_1", "snr_weight", "log_sigma_x")


def reference_coefficients(edm, t_int, xh):
    """The per-molecule scalars of EDM.forward from the reference's own methods and shapes (edm.py:49-62, 98, 244-280)."""
    B = t_int.shape[0]
    t, s = t_int / edm.T, (t_int - 1) / edm.T
    gamma_t = edm.inflate_batch_array(edm.gamma(t), xh)
    gamma_s = edm.inflate_batch_array(edm.gamma(s), xh)
    gamma_1 = edm.gamma(torch.ones((B, 1)))
    sigma_1 = edm.sigma(gamma_1, xh)
    rows = [t, edm.alpha(gamma_t, xh), edm.sigma(gamma_t, xh), edm.alpha(gamma_1, xh), sigma_1 ** 2,
            torch.log(torch.ones_like(sigma_1) / sigma_1), edm.SNR(gamma_s - gamma_t) - 1,
            0.5 * edm.gamma(torch.zeros((B, 1))).view(B)]
    return torch.stack([r.reshape(B) for r in rows])


def golden_loss(ns, name, spec, nb, seed, t_int, table_timesteps=None, n_steps=None, moad_train_dataset=False):
    hp = synthetic.model_hparams(spec)
    if table_timesteps is not None:
        hp['diffusion_steps'] = table_timesteps
    torch.manual_seed(seed)
    ddpm = ns.lightning.DDPM(**hp, data_path=None, batch_size=nb, lr=1e-4, torch_device='cpu', test_epochs=1,
                             n_stability_samples=1)
    synthetic.init_reference_like_weights(ddpm)
    ddpm.eval()
    if n_steps is not None:
        ddpm.edm.T = n_steps
    T = ddpm.edm.T
    items = synthetic.make_items(spec, batch=nb)
    if moad_train_dataset:                                        # lightning.py:165 tests train_dataset
        ddpm.train_dataset = ns.datasets.MOADDataset(data=items)
    data = ns.datasets.collate(items)
    B, N = data['positions'].shape[:2]
    t_int = torch.as_tensor(t_int, dtype=torch.int64).reshape(B, 1)
    noise_seed = seed + 3000
    draw = seeded_noise(noise_seed)
    drawn = []

    def fake_randint(low, high, size, device=None, **kw):
        assert (low, high, tuple(size)) == (0, T + 1, (B, 1))
        return t_int.clone()

    def fake_gaussian(size, device, node_mask):
        drawn.append(draw(size))
        return drawn[-1] * node_mask

    o_randint, o_gauss = torch.randint, ns.utils.sample_gaussian_with_mask
    torch.randint, ns.utils.sample_gaussian_with_mask = fake_randint, fake_gaussian
    try:
        with torch.no_grad():
            metrics = ddpm.validation_step(data, 0)
    finally:
        torch.randint, ns.utils.sample_gaussian_with_mask = o_randint, o_gauss
    assert len(drawn) == 2
    eps = torch.cat(drawn, dim=2)                                 # unmasked: randn(B,N,3) then randn(B,N,F)

    # oracle replay with the same timesteps and draws
    ctx = context_of(data, spec)
    com = data['fragment_only_mask'] if spec.pocket and moad_train_dataset else data['fragment_mask']
    x = orc.remove_partial_mean(data['positions'], data['atom_mask'], com)
    sd_dyn = {k[len("edm.dynamics."):]: v for k, v in ddpm.state_dict().items() if k.startswith("edm.dynamics.")}
    gam = orc.gamma_table(hp['diffusion_noise_schedule'], hp['diffusion_steps'], hp['diffusion_noise_precision'])
    assert torch.equal(gam, ddpm.edm.gamma.gamma.detach()), "oracle gamma table differs"
    with torch.no_grad():
        per, outs = edm_loss_terms(sd_dyn, oracle_cfg(hp), gam, T, x, data['one_hot'], data['atom_mask'],
                                   data['fragment_mask'], data['linker_mask'], data['edge_mask'], ctx, t_int, eps,
                                   norm_values=tuple(hp['normalize_factors']))
    for k, o in zip(OUTPUTS, outs):
        r = metrics[k]
        if not torch.is_tensor(r):                                # the reference's `0.` when no molecule drew t = 0
            assert not torch.is_tensor(o) and o == r == 0., (name, k, o, r)
            continue
        if torch.isnan(r):
            assert torch.isnan(o), (name, k)
            continue
        assert float(o) == float(r), f"{name}: oracle {k} = {float(o)} vs reference {float(r)}"   # max |delta| = 0

    # the native per-molecule scalar table vs the reference's, bit for bit
    xh = torch.cat([x / hp['normalize_factors'][0], data['one_hot'] / hp['normalize_factors'][1]], dim=2)
    ref_coef = reference_coefficients(ddpm.edm, t_int.float(), xh)
    nat = NativeEDM(dynamics=None, in_node_nf=hp['in_node_nf'], n_dims=3, timesteps=hp['diffusion_steps'],
                    noise_schedule=hp['diffusion_noise_schedule'], noise_precision=hp['diffusion_noise_precision'],
                    loss_type=hp['diffusion_loss_type'], norm_values=hp['normalize_factors'])
    nat.T = T
    c = nat.loss_coefficients(t_int)
    mine = torch.stack([c[k].reshape(B) for k in COEF_ROWS])
    assert torch.equal(mine, ref_coef), f"{name}: native loss coefficients differ from the reference's"

    no_t0 = not torch.is_tensor(metrics['loss_term_0'])
    meta = dict(kind="loss", spec=spec.name, batch=nb, seed=seed, noise_seed=noise_seed, T=T,
                table_timesteps=hp['diffusion_steps'], sha=state_sha(ddpm.edm.dynamics.state_dict()),
                moad_train_dataset=bool(moad_train_dataset), no_t0=no_t0)
    outs_arr = {f"out_{k}": torch.tensor(float(metrics[k])) for k in OUTPUTS}
    save(name, meta, t_int=t_int, eps=eps, ref_coef=ref_coef, **outs_arr,
         **{f"per_{k}": v for k, v in per.items()})


def main():
    torch.set_num_threads(8)
    ns = load_reference()
    S = synthetic.SPECS
    print("diffusion-loss golden vectors from the live reference:")
    cfg1 = S["cfg1_plumbing"]
    golden_loss(ns, "loss_cfg1", cfg1, 4, seed=0, t_int=[0, 17, 0, 50])
    golden_loss(ns, "loss_cfg1_no_t0", cfg1, 4, seed=0, t_int=[5, 50, 1, 33])
    golden_loss(ns, "loss_cfg1_all_t0", cfg1, 4, seed=0, t_int=[0, 0, 0, 0])
    golden_loss(ns, "loss_cfg1_T20_table500", cfg1, 4, seed=0, t_int=[0, 1, 19, 20], table_timesteps=500, n_steps=20)
    g = torch.Generator().manual_seed(41)
    for name, spec in (("loss_cfg2_zinc_L6", S["cfg2_zinc"]), ("loss_cfg2_zinc_L8", S["cfg2_zinc_L8"])):
        t_int = torch.randint(0, spec.T + 1, (16,), generator=g)
        t_int[3], t_int[9] = 0, spec.T
        golden_loss(ns, name, spec, 16, seed=2, t_int=t_int)
    geom = synthetic.WorkloadSpec("small_geom", B=5, N=23, n_min=11, l_min=1, l_max=9, F=9, L=3, T=20, seed=12,
                                  anchors_context=True)
    golden_loss(ns, "loss_small_geom_anchors", geom, 5, seed=2, t_int=[3, 0, 20, 11, 1])
    for gt, t_int in (("4A", [0, 7]), ("FC-10A-4A", [13, 0])):
        pk = synthetic.WorkloadSpec(f"small_pocket_{gt}", B=2, N=70, n_min=70, l_min=5, l_max=5, F=9, L=2, T=20,
                                    seed=13, pocket=50, graph_type=gt)
        golden_loss(ns, f"loss_small_pocket_{gt}", pk, 2, seed=3, t_int=t_int, moad_train_dataset=True)
    print("oracle and native loss coefficients agree with the reference")


if __name__ == "__main__":
    main()
