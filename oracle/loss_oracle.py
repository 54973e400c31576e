"""TEST INFRASTRUCTURE ONLY -- CPU oracle for the diffusion objective (EDM.forward, reference src/edm.py:41-124).

A restatement of the reference's training loss in its evaluation form, built on the sampling-path oracle
(oracle/difflinker_oracle.py: Dynamics.forward, the gamma table and the alpha / sigma helpers). Pinned to the live,
unmodified reference by oracle/make_golden_loss.py (max |delta| = 0 on every output of DDPM.validation_step) and re-checked
against tests/golden/loss_*.npz by tests/test_loss_host.py. The product (difflinker_b200/) never imports it.
"""
from __future__ import annotations

import math
from typing import Optional

import numpy as np
import torch

from oracle import difflinker_oracle as orc

Tensor = torch.Tensor


def edm_loss_terms(sd, cfg: orc.OracleConfig, gamma: Tensor, T: int, x, h, node_mask, fragment_mask, linker_mask, edge_mask,
                   context, t_int: Tensor, eps: Tensor, norm_values=(1.0, 4.0, 10.0), norm_biases=(None, 0.0, 0.0),
                   table_timesteps: Optional[int] = None):
    """EDM.forward (edm.py:41-124) with kl_prior (244-270), log_constant_of_p_x_given_z0 (272-280) and
    log_p_xh_given_z0_without_constants (282-318) inlined, for given timesteps `t_int` (B,1) and UNMASKED draws `eps`
    (B,N,3+F) -- what torch.randint (edm.py:49) and the two randn calls of edm.py:67 would return.
    Returns (per_molecule, outputs): per_molecule maps t_int, error_t, l2, loss_term_t, loss_term_0, kl_prior, noise,
    delta_log_px to (B,) tensors; outputs is the reference's 7-tuple (delta_log_px, kl_prior, loss_term_t, loss_term_0,
    l2_loss, noise_t, noise_0)."""
    if table_timesteps is None:
        table_timesteps = gamma.numel() - 1
    B = x.shape[0]
    nd, F_ = cfg.n_dims, cfg.in_node_nf
    x = x / norm_values[0]                                                # edm.py:347-350
    h = (h.float() - norm_biases[1]) / norm_values[1]
    xh = torch.cat([x, h], dim=2)
    n_linker = torch.sum(linker_mask.squeeze(2), dim=1)                   # edm.py:405-407
    dof = n_linker * nd                                                   # edm.py:402-403
    delta_log_px = -dof * np.log(norm_values[0])                          # edm.py:46, 398-399
    t_int = t_int.float()
    t = t_int / T                                                         # edm.py:49-53
    s = (t_int - 1) / T
    t_is_zero = (t_int == 0).squeeze().float()                            # edm.py:54-55
    t_is_not_zero = 1 - t_is_zero
    gamma_t = orc._bcast(orc.gamma_lookup(gamma, t, table_timesteps))             # edm.py:58-59 (index -1 wraps, as there)
    gamma_s = orc._bcast(orc.gamma_lookup(gamma, s, table_timesteps))
    alpha_t, sigma_t = orc._alpha(gamma_t), orc._sigma(gamma_t)                   # edm.py:62-63
    eps_t = torch.cat([eps[:, :, :nd] * linker_mask, eps[:, :, nd:] * linker_mask], dim=2)   # edm.py:67, 328-340
    z_t = alpha_t * xh + sigma_t * eps_t                                  # edm.py:71-72
    z_t = xh * fragment_mask + z_t * linker_mask
    eps_hat = orc.dynamics_forward(sd, cfg, t, z_t, node_mask, linker_mask, edge_mask, context) * linker_mask   # 75-85
    error_t = ((eps_t - eps_hat) ** 2).reshape(B, -1).sum(-1)            # edm.py:88
    l2 = error_t / ((nd + F_) * n_linker)                                 # edm.py:91-92
    # kl_prior (edm.py:244-270): q(z_1 | x) against N(0, 1); the h part sums every row, the x part uses d = 3 n_linker
    gamma_1 = orc.gamma_lookup(gamma, torch.ones((B, 1)), table_timesteps)
    alpha_1, sigma_1 = orc._bcast(orc._alpha(gamma_1)), orc._bcast(orc._sigma(gamma_1))
    mu = alpha_1 * xh
    mu_x, mu_h = mu[:, :, :nd], mu[:, :, nd:]
    one = torch.ones_like(sigma_1)
    kl_h = (torch.log(one / sigma_1) + 0.5 * (sigma_1 ** 2 + mu_h ** 2) / (one ** 2) - 0.5).reshape(B, -1).sum(-1)  # 420-432
    sig_x, one_x = sigma_1.view(-1), torch.ones_like(sigma_1.view(-1))
    mu_norm_2 = (mu_x ** 2).reshape(B, -1).sum(-1)                       # edm.py:434-448
    kl_x = dof * torch.log(one_x / sig_x) + 0.5 * (dof * sig_x ** 2 + mu_norm_2) / (one_x ** 2) - 0.5 * dof
    kl_prior = kl_x + kl_h
    snr_weight = (torch.exp(-(gamma_s - gamma_t)) - 1).squeeze(1).squeeze(1)   # edm.py:98
    loss_term_t = T * 0.5 * snr_weight * error_t                          # edm.py:99
    noise = torch.norm(eps_hat, dim=[1, 2])                               # edm.py:104
    # loss_term_0 (edm.py:107-116), evaluated for every molecule at its own gamma_t and masked by the caller
    log_sigma_x = 0.5 * orc.gamma_lookup(gamma, torch.zeros((B, 1)), table_timesteps).view(B)     # edm.py:272-280
    neg_log_constants = -(dof * (-log_sigma_x - 0.5 * np.log(2 * np.pi)))
    log_p_x = -0.5 * ((eps_t[:, :, :nd] - eps_hat[:, :, :nd]) ** 2).reshape(B, -1).sum(-1)   # edm.py:282-294
    sigma_0 = sigma_t * norm_values[1]
    h_un = h * norm_values[1] + norm_biases[1]                            # edm.py:297-301
    centered = z_t[:, :, nd:] * norm_values[1] + norm_biases[1] - 1
    cdf = lambda v: 0.5 * (1. + torch.erf(v / math.sqrt(2)))              # edm.py:420-422
    log_p_h_prop = torch.log(cdf((centered + 0.5) / sigma_0) - cdf((centered - 0.5) / sigma_0) + 1e-10)   # 303-309
    log_prob = log_p_h_prop - torch.logsumexp(log_p_h_prop, dim=2, keepdim=True)   # edm.py:311-313
    log_p_h = (log_prob * h_un * linker_mask).reshape(B, -1).sum(-1)     # edm.py:315-316
    loss_term_0 = -(log_p_x + log_p_h) + neg_log_constants
    per = dict(t_int=t_int.reshape(-1), error_t=error_t, l2=l2, loss_term_t=loss_term_t, loss_term_0=loss_term_0,
               kl_prior=kl_prior, noise=noise, delta_log_px=delta_log_px)
    # batch reductions (edm.py:46, 93, 96, 100-122)
    lt = (loss_term_t * t_is_not_zero).sum() / t_is_not_zero.sum()
    nt = (noise * t_is_not_zero).sum() / t_is_not_zero.sum()
    if t_is_zero.sum() > 0:
        l0 = (loss_term_0 * t_is_zero).sum() / t_is_zero.sum()
        n0 = (noise * t_is_zero).sum() / t_is_zero.sum()
    else:
        l0, n0 = 0., 0.
    return per, (delta_log_px.mean(), kl_prior.mean(), lt, l0, l2.mean(), nt, n0)
