"""CPU checks of the diffusion objective (EDM.forward, src/edm.py:41-124): the oracle against the reference's fixtures
(oracle/make_golden_loss.py), the native per-molecule scalar table against the reference's, and the refusals."""
import pytest
import torch

from difflinker_b200 import synthetic
from difflinker_b200.batching import collate
import dl_helpers as helpers
from oracle import difflinker_oracle as orc
from oracle.loss_oracle import edm_loss_terms

LOSS_CASES = ["loss_cfg1", "loss_cfg1_no_t0", "loss_cfg1_all_t0", "loss_cfg1_T20_table500", "loss_cfg2_zinc_L6",
              "loss_cfg2_zinc_L8", "loss_small_geom_anchors", "loss_small_pocket_4A", "loss_small_pocket_FC-10A-4A"]
OUTPUTS = ("delta_log_px", "kl_prior", "loss_term_t", "loss_term_0", "l2_loss", "noise_t", "noise_0")
PER_MOLECULE = ("t_int", "error_t", "l2", "loss_term_t", "loss_term_0", "kl_prior", "noise", "delta_log_px")
COEF_ROWS = ("t", "alpha_t", "sigma_t", "alpha_1", "sigma2_1", "log_inv_sigma_1", "snr_weight", "log_sigma_x")
BOUND = 5e-5            # the oracle chain replays' bound (test_oracle_golden.py)


def fixture_batch(meta):
    """The fixture's model (weights rebuilt from the seed and checked against the sha256) and collated batch."""
    spec = helpers.spec_by_name(meta["spec"])
    ddpm, hp = helpers.build_ddpm(spec, meta["seed"], diffusion_steps=meta["table_timesteps"])
    assert helpers.state_sha(ddpm.edm.dynamics.state_dict()) == meta["sha"]
    ddpm.edm.T = meta["T"]
    return spec, ddpm, hp, collate(synthetic.make_items(spec, batch=meta["batch"]))


@pytest.mark.parametrize("name", LOSS_CASES)
def test_oracle_loss_terms_match_reference_golden(name):
    meta, a = helpers.load_golden(name)
    spec, ddpm, hp, data = fixture_batch(meta)
    com = data['fragment_only_mask'] if meta["moad_train_dataset"] else data['fragment_mask']
    x = orc.remove_partial_mean(data['positions'], data['atom_mask'], com)
    sd = {k[len("edm.dynamics."):]: v for k, v in ddpm.state_dict().items() if k.startswith("edm.dynamics.")}
    gam = orc.gamma_table(hp['diffusion_noise_schedule'], hp['diffusion_steps'], hp['diffusion_noise_precision'])
    with helpers.golden_threads(), torch.no_grad():
        per, outs = edm_loss_terms(sd, helpers.oracle_cfg(hp), gam, meta["T"], x, data['one_hot'], data['atom_mask'],
                                   data['fragment_mask'], data['linker_mask'], data['edge_mask'],
                                   helpers.context_of(data, spec), a["t_int"], a["eps"],
                                   norm_values=tuple(hp['normalize_factors']))
    for k in PER_MOLECULE:
        want = a[f"per_{k}"]
        assert (per[k] - want).abs().max().item() <= BOUND * max(1.0, want.abs().max().item()), k
    for k, got in zip(OUTPUTS, outs):
        want = a[f"out_{k}"]
        if meta["no_t0"] and k in ("loss_term_0", "noise_0"):
            assert not torch.is_tensor(got) and got == 0.
        elif torch.isnan(want):
            assert torch.isnan(got), k
        else:
            assert abs(float(got) - float(want)) <= BOUND * max(1.0, abs(float(want))), k


@pytest.mark.parametrize("name", LOSS_CASES)
def test_loss_coefficients_equal_the_reference_bit_for_bit(name):
    """The per-molecule scalars (alpha_t, sigma_t, SNR(gamma_s - gamma_t) - 1, ...) the native EDM hands to the kernels are
    the reference's own, including t_int = 0 (s wraps to the end of the table) and T != table length."""
    meta, a = helpers.load_golden(name)
    _, ddpm, _, _ = fixture_batch(meta)
    c = ddpm.edm.loss_coefficients(a["t_int"])
    got = torch.stack([c[k].reshape(-1) for k in COEF_ROWS])
    assert torch.equal(got, a["ref_coef"])


def test_ddpm_forward_refuses_training():
    spec = synthetic.SPECS["cfg1_plumbing"]
    ddpm, _ = helpers.build_ddpm(spec, 0)
    with pytest.raises(NotImplementedError, match="no backward pass"):
        ddpm.forward(collate(synthetic.make_items(spec, batch=2)), training=True)


def test_inpainting_edm_forward_is_not_implemented():
    spec = synthetic.SPECS["cfg1_plumbing"]
    ddpm, _ = helpers.build_ddpm(spec, 0, inpainting=True)
    data = collate(synthetic.make_items(spec, batch=2))
    with pytest.raises(NotImplementedError):
        ddpm.edm.forward(data['positions'], data['one_hot'], data['atom_mask'], data['fragment_mask'],
                         data['linker_mask'], data['edge_mask'], data['fragment_mask'])
    with pytest.raises(NotImplementedError):
        ddpm.validation_step(data)
