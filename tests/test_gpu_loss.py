"""GPU tests of the diffusion objective (EDM.forward / DDPM.validation_step, src/edm.py:41-124, src/lightning.py:148-268)
through dl_diffusion_loss: against the reference's fixtures (oracle/make_golden_loss.py), the device-side noise stream
against torch's own draws, determinism, the NaN mapping and the accelerate() path."""
import math
import types

import pytest
import torch

import difflinker_b200
from difflinker_b200 import FoundNaNException, synthetic
from difflinker_b200.batching import collate
import dl_helpers as helpers

pytestmark = pytest.mark.gpu
REL_TOL = 1e-4
LOSS_CASES = ["loss_cfg1", "loss_cfg1_no_t0", "loss_cfg1_all_t0", "loss_cfg1_T20_table500", "loss_cfg2_zinc_L6",
              "loss_cfg2_zinc_L8", "loss_small_geom_anchors", "loss_small_pocket_4A", "loss_small_pocket_FC-10A-4A"]
OUTPUTS = ("delta_log_px", "kl_prior", "loss_term_t", "loss_term_0", "l2_loss", "noise_t", "noise_0")
PER_MOLECULE = ("error_t", "l2", "loss_term_t", "loss_term_0", "kl_prior", "noise", "delta_log_px")


class MOADDataset(list):
    """Stand-in with the reference class's NAME: lightning.py:165 switches the context and centre-of-mass mask on
    `isinstance(self.train_dataset, MOADDataset)`."""


def dev():
    assert torch.cuda.is_available()
    torch.cuda.init()
    return torch.device("cuda", 0)


def rel_err(got, want):
    return (got.double() - want.double()).abs().max().item() / max(want.double().abs().max().item(), 1e-30)


def to_dev(data, d):
    return {k: (v.to(d) if torch.is_tensor(v) else v) for k, v in data.items()}


def inject(edm, t_int, eps):
    """Test hooks: the timesteps and the unmasked draws the reference's randint / randn calls returned."""
    edm.draw_timesteps = lambda n, device: t_int.float().reshape(n, 1).to(device)
    edm.draw_noise = lambda n_draws, n_samples, n_nodes, device, generator=None: eps[None].to(device)


def spy_loss_terms(edm):
    """Keeps the per-molecule terms EDM.forward reduces."""
    seen = {}
    orig = edm.loss_terms

    def spy(*a, **k):
        seen.update(orig(*a, **k))
        return seen
    edm.loss_terms = spy
    return seen


def golden_model(meta, impl):
    spec = helpers.spec_by_name(meta["spec"])
    ddpm, hp = helpers.build_ddpm(spec, meta["seed"], edge_impl=impl, diffusion_steps=meta["table_timesteps"])
    assert helpers.state_sha(ddpm.edm.dynamics.state_dict()) == meta["sha"]
    ddpm.edm.T = meta["T"]
    items = synthetic.make_items(spec, batch=meta["batch"])
    if meta["moad_train_dataset"]:
        ddpm.train_dataset = MOADDataset(items)
    return ddpm, collate(items)


@pytest.mark.parametrize("impl", ["simt", "auto"])
@pytest.mark.parametrize("name", LOSS_CASES)
def test_validation_step_matches_reference_golden(name, impl):
    meta, a = helpers.load_golden(name)
    d = dev()
    ddpm, data = golden_model(meta, impl)
    ddpm = ddpm.to(d)
    inject(ddpm.edm, a["t_int"], a["eps"])
    per = spy_loss_terms(ddpm.edm)
    out = ddpm.validation_step(to_dev(data, d))
    assert torch.equal(per["t_int"].cpu(), a["per_t_int"])
    for k in PER_MOLECULE:
        assert rel_err(per[k].cpu(), a[f"per_{k}"]) <= REL_TOL, k
    for k in OUTPUTS:
        want = a[f"out_{k}"]
        if meta["no_t0"] and k in ("loss_term_0", "noise_0"):
            assert type(out[k]) is float and out[k] == 0.          # the reference's Python float (edm.py:118-120)
        elif torch.isnan(want):
            assert torch.isnan(out[k]).item(), k
        else:
            assert rel_err(out[k].cpu().reshape(1), want.reshape(1)) <= REL_TOL, k
    assert out['loss'] is out['l2_loss']                             # loss_type 'l2' (lightning.py:230-236)
    if not meta["no_t0"] and not torch.isnan(a["out_loss_term_t"]):
        vlb = out['kl_prior'] + out['loss_term_t'] + out['loss_term_0'] - out['delta_log_px']
        assert torch.equal(out['vlb_loss'], vlb)


def edm_inputs(spec, nb, d):
    data = collate(synthetic.make_items(spec, batch=nb))
    x = difflinker_b200.utils.remove_partial_mean_with_mask(data['positions'], data['atom_mask'], data['fragment_mask'])
    return dict(x=x.to(d), h=data['one_hot'].to(d), node_mask=data['atom_mask'].to(d),
                fragment_mask=data['fragment_mask'].to(d), linker_mask=data['linker_mask'].to(d),
                edge_mask=data['edge_mask'].to(d), context=helpers.context_of(data, spec).to(d))


@pytest.mark.parametrize("spec_name,nb", [("cfg1_plumbing", 4), ("cfg2_zinc", 256)])
def test_device_noise_stream_equals_torch_draws_bit_for_bit(spec_name, nb):
    """In-kernel noise = torch.randint + torch.randn(B,N,3) + torch.randn(B,N,F) on CUDA after the same seed, and the
    generator ends at the same offset."""
    d = dev()
    spec = synthetic.SPECS[spec_name]
    ddpm, _ = helpers.build_ddpm(spec, 2)
    edm = ddpm.to(d).edm
    kw = edm_inputs(spec, nb, d)
    gen = torch.cuda.default_generators[0]
    torch.manual_seed(1234)
    native = edm.forward(**kw)
    off_native = gen.get_offset()
    torch.manual_seed(1234)
    B, N = kw['x'].shape[:2]
    t_int = torch.randint(0, edm.T + 1, size=(B, 1), device=d)
    eps = torch.cat([torch.randn((B, N, 3), device=d), torch.randn((B, N, spec.F), device=d)], dim=2)
    off_torch = gen.get_offset()
    inject(edm, t_int, eps)
    fed = edm.forward(**kw)
    assert off_native == off_torch
    for k, u, v in zip(OUTPUTS, native, fed):
        if torch.is_tensor(u):
            assert torch.equal(u, v) or (torch.isnan(u).item() and torch.isnan(v).item()), k
        else:
            assert u == v, k


def test_same_seed_same_terms_and_forward_reduces_loss_terms():
    d = dev()
    spec = synthetic.SPECS["cfg1_plumbing"]
    ddpm, _ = helpers.build_ddpm(spec, 0)
    edm = ddpm.to(d).edm
    kw = edm_inputs(spec, 4, d)
    runs = []
    for _ in range(2):
        torch.manual_seed(7)
        runs.append(edm.loss_terms(**kw))
    assert all(torch.equal(runs[0][k], runs[1][k]) for k in runs[0])
    torch.manual_seed(7)
    out = edm.forward(**kw)
    lt = runs[0]
    z = (lt['t_int'] == 0).float()
    nz = 1 - z
    want = [lt['delta_log_px'].mean(), lt['kl_prior'].mean(), (lt['loss_term_t'] * nz).sum() / nz.sum(),
            (lt['loss_term_0'] * z).sum() / z.sum() if z.sum() > 0 else 0., lt['l2'].mean(),
            (lt['noise'] * nz).sum() / nz.sum(), (lt['noise'] * z).sum() / z.sum() if z.sum() > 0 else 0.]
    for k, u, v in zip(OUTPUTS, out, want):
        assert (torch.equal(u, v) if torch.is_tensor(v) else u == v), k


def test_nan_in_dynamics_raises_found_nan_exception():
    d = dev()
    spec = helpers.EXTRA_SPECS["small_fc"]
    ddpm, _ = helpers.build_ddpm(spec, 0)
    edm = ddpm.to(d).edm
    kw = edm_inputs(spec, 3, d)
    lm = kw['linker_mask'][1, :, 0].nonzero()[0, 0].item()
    kw['x'][1, lm, 0] = float('nan')                                 # a linker atom: poisons z_t, hence the dynamics
    with pytest.raises(FoundNaNException) as ei:
        edm.forward(**kw)
    e = ei.value
    assert (e.x_h_nan_idx | e.only_x_nan_idx | e.only_h_nan_idx) == {1}
    kw['x'][1, lm, 0] = 0.0
    torch.manual_seed(5)
    kl_prior = edm.forward(**kw)[1]                                  # and the engine stays usable afterwards
    assert math.isfinite(float(kl_prior))


def test_accelerated_module_edm_forward_equals_native_ddpm():
    """accelerate() swaps the EDM of a reference DDPM; its `edm.forward`, which the reference's own DDPM.forward /
    validation_step call (lightning.py:191-199), then returns exactly what the native DDPM's does."""
    d = dev()
    spec = synthetic.SPECS["cfg1_plumbing"]
    native, hp = helpers.build_ddpm(spec, 0)
    sd = native.edm.state_dict()
    ref = types.SimpleNamespace(hparams=hp, edm=types.SimpleNamespace(state_dict=lambda: sd, T=native.edm.T))
    difflinker_b200.accelerate(ref)
    kw = edm_inputs(spec, 4, d)
    outs = []
    for edm in (native.edm.to(d), ref.edm.to(d)):
        torch.manual_seed(11)
        outs.append(edm.forward(**kw))
    for k, u, v in zip(OUTPUTS, *outs):
        assert (torch.equal(u, v) if torch.is_tensor(u) else u == v), k


def test_inpainting_engine_is_refused_by_the_entry_point():
    import ctypes as C
    from difflinker_b200 import _native
    d = dev()
    spec = helpers.EXTRA_SPECS["small_fc"]
    dyn, _ = helpers.build_dynamics(spec, 0, centering=True)
    eng = dyn.engine(0)
    lib = _native.load_library()
    B, N, xd = 2, 8, 3 + spec.F
    f = lambda *s: torch.zeros(s, device=d)
    norm = (C.c_float * 3)(1.0, 4.0, 0.0)
    st = lib.dl_diffusion_loss(eng, B, N, f(B, N, xd).data_ptr(), torch.ones((B, N), dtype=torch.int8, device=d).data_ptr(),
                               f(B, N).data_ptr(), f(B, N).data_ptr(), None, f(B, N, 1).data_ptr(),
                               f(len(_native.LOSS_COEFS), B).data_ptr(), f(B, N, xd).data_ptr(), 0, 0, None, norm,
                               f(B, len(_native.LOSS_TERMS)).data_ptr(), None, torch.cuda.current_stream(d).cuda_stream)
    assert st == -4                                                  # DL_ERR_UNSUPPORTED
