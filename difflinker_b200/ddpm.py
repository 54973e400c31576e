"""Outer drop-in boundary: `DDPM.sample_chain(data, sample_fn=None, keep_frames=None) -> (chain, node_mask)`
(reference: src/lightning.py:405-463; constructor wiring src/lightning.py:39-113).

Two ways in:
  * `DDPM(**hparams)` -- a plain nn.Module with the reference's hyper-parameter names and state_dict layout
    (`edm.gamma.gamma`, `edm.dynamics.dynamics....`), for environments without pytorch_lightning;
  * `accelerate(ddpm)` -- swaps the `.edm` of an existing *reference* DDPM (e.g. one returned by
    `DDPM.load_from_checkpoint`) for the native one in place, so generate.py / sample.py run unchanged.
`DDPM.forward(data, training=False)`, `validation_step` and `test_step` (lightning.py:148-268) evaluate the diffusion
loss; training (backward, optimiser), datasets, metrics and visualisation are out of scope (SURVEY.md section 2).
"""
import torch
import torch.nn as nn

from . import utils
from .batching import create_templates_for_linker_generation
from .edm import EDM, InpaintingEDM
from .egnn import Dynamics, DynamicsWithPockets


def _build_edm(hp: dict, edge_impl='auto'):
    pocket = '.' in (hp.get('train_data_prefix') or '')
    graph_type = hp.get('graph_type')
    if graph_type is None:
        graph_type = '4A' if pocket else 'FC'                              # lightning.py:75-76
    activation = hp.get('activation', 'silu')
    if isinstance(activation, str):
        if activation != 'silu':
            raise Exception("activation fn not supported yet. Add it here.")  # lightning.py:23-27
        activation = nn.SiLU()
    dyn_cls = DynamicsWithPockets if pocket else Dynamics                  # lightning.py:81
    dynamics = dyn_cls(
        in_node_nf=hp['in_node_nf'], n_dims=hp['n_dims'], context_node_nf=hp['context_node_nf'],
        device=hp.get('torch_device', 'cpu'), hidden_nf=hp['hidden_nf'], activation=activation,
        n_layers=hp['n_layers'], attention=hp['attention'], tanh=hp['tanh'], norm_constant=hp['norm_constant'],
        inv_sublayers=hp['inv_sublayers'], sin_embedding=hp['sin_embedding'],
        normalization_factor=hp['normalization_factor'], aggregation_method=hp['aggregation_method'],
        model=hp['model'], normalization=hp.get('normalization'), centering=bool(hp.get('inpainting', False)),
        graph_type=graph_type, edge_impl=edge_impl)
    edm_cls = InpaintingEDM if hp.get('inpainting') else EDM                 # lightning.py:102
    return edm_cls(dynamics=dynamics, in_node_nf=hp['in_node_nf'], n_dims=hp['n_dims'],
               timesteps=hp['diffusion_steps'], noise_schedule=hp['diffusion_noise_schedule'],
               noise_precision=hp['diffusion_noise_precision'], loss_type=hp['diffusion_loss_type'],
               norm_values=hp['normalize_factors'])


def sampler_inputs(model, data, sample_fn=None):
    """What DDPM.sample_chain hands to EDM.sample_chain (lightning.py:405-452): the template batch, the context
    columns and the centred coordinates, as the keyword arguments of `edm.sample_chain`.
    `model` needs .inpainting, .anchors_context, .train_data_prefix, .center_of_mass, .val_dataset."""
    if sample_fn is None:
        linker_sizes = data['linker_mask'].sum(1).view(-1).int()
    else:
        linker_sizes = sample_fn(data)
    template = data if model.inpainting else create_templates_for_linker_generation(data, linker_sizes)
    x, h = template['positions'], template['one_hot']
    node_mask, edge_mask = template['atom_mask'], template['edge_mask']
    anchors, fragment_mask, linker_mask = template['anchors'], template['fragment_mask'], template['linker_mask']
    pocket = '.' in model.train_data_prefix
    if pocket:
        fragment_only = template['fragment_only_mask']
        pocket_only = fragment_mask - fragment_only
        parts = [anchors, fragment_only, pocket_only] if model.anchors_context else [fragment_only, pocket_only]
        context = torch.cat(parts, dim=-1)
    else:
        context = torch.cat([anchors, fragment_mask], dim=-1) if model.anchors_context else fragment_mask
    if model.inpainting:
        com_mask = node_mask
    elif type(getattr(model, 'val_dataset', None)).__name__ == 'MOADDataset' and model.center_of_mass == 'fragments':
        com_mask = template['fragment_only_mask']
    elif model.center_of_mass == 'fragments':
        com_mask = fragment_mask
    elif model.center_of_mass == 'anchors':
        com_mask = anchors
    else:
        raise NotImplementedError(model.center_of_mass)
    x = utils.remove_partial_mean_with_mask(x, node_mask, com_mask)
    return dict(x=x, h=h, node_mask=node_mask, edge_mask=edge_mask, fragment_mask=fragment_mask,
                linker_mask=linker_mask, context=context)


def sample_chain(model, data, sample_fn=None, keep_frames=None):
    """Body of DDPM.sample_chain (lightning.py:405-463), shared by `DDPM` below and by accelerated reference
    modules (`model` additionally needs .edm)."""
    kw = sampler_inputs(model, data, sample_fn)
    chain = model.edm.sample_chain(**kw, keep_frames=keep_frames)
    return chain, kw['node_mask']


def loss_forward(model, data):
    """Body of DDPM.forward(data, training=False) (lightning.py:148-199). `model` needs .anchors_context, .train_dataset,
    .inpainting, .center_of_mass and .edm. NB the pocket switch tests train_dataset here, where the sampler tests
    val_dataset (lightning.py:441)."""
    x = data['positions']
    h = data['one_hot']
    node_mask = data['atom_mask']
    edge_mask = data['edge_mask']
    anchors = data['anchors']
    fragment_mask = data['fragment_mask']
    linker_mask = data['linker_mask']
    if model.anchors_context:
        context = torch.cat([anchors, fragment_mask], dim=-1)
    else:
        context = fragment_mask
    moad = type(getattr(model, 'train_dataset', None)).__name__ == 'MOADDataset'
    if moad:
        fragment_only_mask = data['fragment_only_mask']
        pocket_only_mask = fragment_mask - fragment_only_mask
        if model.anchors_context:
            context = torch.cat([anchors, fragment_only_mask, pocket_only_mask], dim=-1)
        else:
            context = torch.cat([fragment_only_mask, pocket_only_mask], dim=-1)
    if model.inpainting:
        center_of_mass_mask = node_mask
    elif moad and model.center_of_mass == 'fragments':
        center_of_mass_mask = data['fragment_only_mask']
    elif model.center_of_mass == 'fragments':
        center_of_mass_mask = fragment_mask
    elif model.center_of_mass == 'anchors':
        center_of_mass_mask = anchors
    else:
        raise NotImplementedError(model.center_of_mass)
    x = utils.remove_partial_mean_with_mask(x, node_mask, center_of_mass_mask)
    # (the reference's assert_partial_mean_zero_with_mask is a host-synchronising check of the line above; not repeated)
    return model.edm.forward(x=x, h=h, node_mask=node_mask, fragment_mask=fragment_mask, linker_mask=linker_mask,
                             edge_mask=edge_mask, context=context)


def step_metrics(model, data):
    """The dict validation_step / test_step return (lightning.py:228-268)."""
    delta_log_px, kl_prior, loss_term_t, loss_term_0, l2_loss, noise_t, noise_0 = model.forward(data, training=False)
    vlb_loss = kl_prior + loss_term_t + loss_term_0 - delta_log_px
    if model.loss_type == 'l2':
        loss = l2_loss
    elif model.loss_type == 'vlb':
        loss = vlb_loss
    else:
        raise NotImplementedError(model.loss_type)
    return {
        'loss': loss,
        'delta_log_px': delta_log_px,
        'kl_prior': kl_prior,
        'loss_term_t': loss_term_t,
        'loss_term_0': loss_term_0,
        'l2_loss': l2_loss,
        'vlb_loss': vlb_loss,
        'noise_t': noise_t,
        'noise_0': noise_0
    }


class DDPM(nn.Module):
    """Hyper-parameter-compatible stand-in for the Lightning module: sampling, and the evaluation steps
    (validation_step / test_step)."""
    train_dataset = None
    val_dataset = None
    test_dataset = None
    FRAMES = 100

    def __init__(
        self,
        in_node_nf, n_dims, context_node_nf, hidden_nf, activation, tanh, n_layers, attention, norm_constant,
        inv_sublayers, sin_embedding, normalization_factor, aggregation_method,
        diffusion_steps, diffusion_noise_schedule, diffusion_noise_precision, diffusion_loss_type,
        normalize_factors, include_charges, model,
        data_path=None, train_data_prefix='', val_data_prefix='', batch_size=64, lr=2e-4, torch_device='cpu',
        test_epochs=None, n_stability_samples=None,
        normalization=None, log_iterations=None, samples_dir=None, data_augmentation=False,
        center_of_mass='fragments', inpainting=False, anchors_context=True, graph_type=None, edge_impl='auto',
    ):
        super().__init__()
        self.hparams = {k: v for k, v in locals().items() if k not in ('self', '__class__', 'edge_impl')}
        self.data_path, self.train_data_prefix, self.val_data_prefix = data_path, train_data_prefix, val_data_prefix
        self.batch_size, self.lr, self.torch_device = batch_size, lr, torch_device
        self.include_charges = include_charges
        self.samples_dir = samples_dir
        self.center_of_mass = center_of_mass
        self.inpainting = inpainting
        self.loss_type = diffusion_loss_type
        self.n_dims = n_dims
        self.num_classes = in_node_nf - include_charges
        self.anchors_context = anchors_context
        self.is_geom = ('geom' in train_data_prefix) or ('MOAD' in train_data_prefix)
        self.edm = _build_edm(self.hparams, edge_impl=edge_impl)

    def sample_chain(self, data, sample_fn=None, keep_frames=None):
        return sample_chain(self, data, sample_fn=sample_fn, keep_frames=keep_frames)

    def forward(self, data, training):
        """DDPM.forward (lightning.py:148-199): the diffusion objective of a collated batch through EDM.forward.
        Evaluation only (training=False, as validation_step / test_step call it)."""
        if training:
            raise NotImplementedError("DDPM.forward(training=True): no backward pass on the native path")
        return loss_forward(self, data)

    def validation_step(self, data, *args):
        """lightning.py:228-247 (without Lightning's logging)."""
        return step_metrics(self, data)

    def test_step(self, data, *args):
        """lightning.py:249-268."""
        return step_metrics(self, data)

    @classmethod
    def load_from_checkpoint(cls, checkpoint_path, map_location=None, strict=True, **overrides):
        """`DDPM.load_from_checkpoint(args.model, map_location=device)` (generate.py:101, sample.py:84) without
        pytorch_lightning: a Lightning checkpoint is a dict with `hyper_parameters` (what `save_hyperparameters()` stored,
        lightning.py:51) and `state_dict`. Keyword overrides replace saved hyper-parameters, as in Lightning."""
        return _load_lightning_checkpoint(cls, checkpoint_path, map_location, strict, overrides)


def _load_lightning_checkpoint(cls, checkpoint_path, map_location, strict, overrides):
    try:
        ckpt = torch.load(checkpoint_path, map_location='cpu', weights_only=False)
    except TypeError:                                        # older torch without the weights_only argument
        ckpt = torch.load(checkpoint_path, map_location='cpu')
    if 'state_dict' not in ckpt or 'hyper_parameters' not in ckpt:
        raise KeyError("not a Lightning checkpoint: expected the keys 'state_dict' and 'hyper_parameters'")
    hp = dict(ckpt['hyper_parameters'])
    hp.update(overrides)
    model = cls(**hp)
    model.load_state_dict(ckpt['state_dict'], strict=strict)
    if map_location is not None:
        model = model.to(map_location)
    return model


def accelerate(ddpm, edge_impl='auto'):
    """Replace `ddpm.edm` of a *reference* DDPM (src/lightning.py) by the native EDM, copying its weights
    (strict state_dict match) and its possibly overridden `.T` (generate.py:103-104). Returns `ddpm`."""
    hp = dict(ddpm.hparams) if hasattr(ddpm, 'hparams') and len(dict(ddpm.hparams)) else None
    if hp is None:
        raise ValueError("the module carries no hparams; construct difflinker_b200.DDPM(**hparams) instead")
    new_edm = _build_edm(hp, edge_impl=edge_impl)
    new_edm.load_state_dict(ddpm.edm.state_dict(), strict=True)
    new_edm.T = ddpm.edm.T
    ddpm.edm = new_edm
    return ddpm
