"""Drop-in `EDM` sampler (reference: src/edm.py:14-463, sampling half) running the whole reverse-diffusion loop on
the device through `dl_sample_chain`: one CUDA-graph replay per step, no host synchronisation inside the loop.

What stays in Python (plumbing): normalisation of the inputs, the per-step scalar table -- computed with the very
torch ops the reference uses (edm.py:369-403) so the coefficients are bit-identical -- and the random draws, which
are made with the reference's `torch.randn` call order and shapes (edm.py:328-345) on the tensors' device, so a given
torch seed produces the same noise stream as the reference would on that device.
"""
import ctypes as C

import numpy as np
import torch
import torch.nn.functional as F

from . import _native
from .noise import PredefinedNoiseSchedule
from .utils import FoundNaNException, nan_exception_class


class EDM(torch.nn.Module):
    def __init__(
            self,
            dynamics,
            in_node_nf: int,
            n_dims: int,
            timesteps: int = 1000,
            noise_schedule='learned',
            noise_precision=1e-4,
            loss_type='vlb',
            norm_values=(1., 1., 1.),
            norm_biases=(None, 0., 0.),
    ):
        super().__init__()
        if noise_schedule == 'learned':
            # GammaNetwork (src/noise.py:131-169) is only valid with the vlb loss; every config trains with
            # l2 + polynomial_2 (train_difflinker.py:140-142). Out of scope for the sampling hot path.
            raise NotImplementedError("learned noise schedules are outside the difflinker_b200 hot path")
        self.gamma = PredefinedNoiseSchedule(noise_schedule, timesteps=timesteps, precision=noise_precision)
        self.dynamics = dynamics
        self.in_node_nf = in_node_nf
        self.n_dims = n_dims
        self.T = timesteps
        self.norm_values = norm_values
        self.norm_biases = norm_biases
        # 'reference_stream' (default): the reference's torch.randn call order, so seeds line up with the reference run on
        #   the same kind of device. On CUDA the numbers are regenerated INSIDE the kernels that consume them from the torch
        #   generator's (seed, offset) -- same values as the randn calls, no tensor, no launches (dl_sample_chain_rng).
        # 'reference_tensor': the same stream materialised with torch.randn (two launches per draw).
        # 'bulk': one randn call for the whole chain (a different stream).
        self.noise_mode = 'reference_stream'
        self.last_loop_ms = None               # device time of the last reverse loop (CUDA events)

    def forward(self, x, h, node_mask, fragment_mask, linker_mask, edge_mask, context=None):
        """The diffusion objective of a batch (edm.py:41-124), evaluation only: one q(z_t|x,h) draw per molecule, one
        Dynamics.forward and the loss terms, on the device. Returns the reference's tuple (delta_log_px, kl_prior,
        loss_term_t, loss_term_0, l2_loss, noise_t, noise_0); loss_term_0 and noise_0 are the float 0. when no molecule
        drew t = 0, and the t > 0 means are NaN when every molecule did, as in the reference. No gradients."""
        lt = self.loss_terms(x, h, node_mask, fragment_mask, linker_mask, edge_mask, context)
        delta_log_px = lt['delta_log_px'].mean()                                      # edm.py:46
        l2_loss = lt['l2'].mean()                                                     # edm.py:92-93
        kl_prior = lt['kl_prior'].mean()                                              # edm.py:96
        t_is_zero = (lt['t_int'] == 0).squeeze().float()                              # edm.py:54-55
        t_is_not_zero = 1 - t_is_zero
        loss_term_t = (lt['loss_term_t'] * t_is_not_zero).sum() / t_is_not_zero.sum()  # edm.py:100-101
        noise_t = (lt['noise'] * t_is_not_zero).sum() / t_is_not_zero.sum()           # edm.py:104-105
        if t_is_zero.sum() > 0:                                                       # edm.py:107-120
            loss_term_0 = (lt['loss_term_0'] * t_is_zero).sum() / t_is_zero.sum()
            noise_0 = (lt['noise'] * t_is_zero).sum() / t_is_zero.sum()
        else:
            loss_term_0 = 0.
            noise_0 = 0.
        return delta_log_px, kl_prior, loss_term_t, loss_term_0, l2_loss, noise_t, noise_0

    def draw_timesteps(self, n_samples, device):
        """edm.py:49: the reference's own randint call on the batch's device, so the generator advances as it would."""
        return torch.randint(0, self.T + 1, size=(n_samples, 1), device=device).float()

    def loss_coefficients(self, t_int):
        """Per-molecule scalars of EDM.forward for the timesteps `t_int` (B,1): a dict of (B,1) fp32 CPU tensors evaluated
        with the reference's ops and shapes (edm.py:49-62, 98, 244-254, 272-280), so they round as the reference's do --
        SNR(gamma_s - gamma_t) - 1 cancels badly near t = 0. For t_int = 0, s indexes the table at -1, which wraps to its
        last entry as in the reference; that term is masked out later."""
        gamma = self._cpu_schedule()
        t_int = t_int.detach().to(device='cpu', dtype=torch.float32).reshape(-1, 1)
        n = t_int.shape[0]
        t = t_int / self.T
        s = (t_int - 1) / self.T
        gamma_t, gamma_s = gamma(t), gamma(s)
        gamma_1 = gamma(torch.ones((n, 1)))
        sigma_1 = self.sigma(gamma_1)
        return dict(t=t, alpha_t=self.alpha(gamma_t), sigma_t=self.sigma(gamma_t), alpha_1=self.alpha(gamma_1),
                    sigma2_1=sigma_1 ** 2, log_inv_sigma_1=torch.log(torch.ones_like(sigma_1) / sigma_1),
                    snr_weight=self.SNR(gamma_s - gamma_t) - 1, log_sigma_x=0.5 * gamma(torch.zeros((n, 1))))

    @torch.no_grad()
    def loss_terms(self, x, h, node_mask, fragment_mask, linker_mask, edge_mask, context=None, eps=None):
        """Per-molecule terms of EDM.forward as (B,) tensors on x's device: t_int, error_t, l2, loss_term_t, loss_term_0,
        kl_prior, noise, delta_log_px (before the batch reductions of edm.py:92-120; e.g. to rank molecules by their
        loss). `eps` optionally injects the (B,N,3+F) unmasked draws."""
        lib = _native.load_library()
        n_samples, n_nodes = x.size(0), x.size(1)
        dev = x.device
        work = dev if dev.type == 'cuda' else torch.device('cuda', self.dynamics._device_index(x))
        d = self.n_dims + self.in_node_nf
        xn, hn = self.normalize(x, h)
        xh = torch.cat([xn, hn], dim=2).to(device=work, dtype=torch.float32).contiguous()
        t_int = self.draw_timesteps(n_samples, dev)                                  # edm.py:49, before the noise draw
        on_device = (eps is None and dev.type == 'cuda' and self.noise_mode == 'reference_stream'
                     and 'draw_noise' not in self.__dict__)
        if not on_device:
            if eps is None:
                eps = self.draw_noise(1, n_samples, n_nodes, dev)[0]
            eps = eps.to(device=work, dtype=torch.float32).contiguous()
            assert eps.shape == (n_samples, n_nodes, d), eps.shape
        c = self.loss_coefficients(t_int.cpu())
        coef = torch.cat([c[k].reshape(1, -1) for k in _native.LOSS_COEFS]).to(work).contiguous()
        eng = self.dynamics.engine(work.index)
        self.dynamics._check_graph_type()
        prep = lambda v, dt: None if v is None else v.detach().to(device=work, dtype=dt).contiguous()
        nm = prep(node_mask.reshape(n_samples, n_nodes), torch.int8)
        fm = prep(fragment_mask.reshape(n_samples, n_nodes), torch.float32)
        lm = prep(linker_mask.reshape(n_samples, n_nodes), torch.float32)
        em = None
        if self.dynamics.graph_type == 'FC' and edge_mask is not None:
            em = prep(edge_mask.reshape(-1), torch.int8)
            assert em.numel() == n_samples * n_nodes * n_nodes
        ctx = None if context is None else prep(
            context.reshape(n_samples, n_nodes, self.dynamics.context_node_nf), torch.float32)   # wrong width -> raises
        norm = (C.c_float * 3)(float(self.norm_values[0]), float(self.norm_values[1]), float(self.norm_biases[1]))
        terms = torch.empty((n_samples, len(_native.LOSS_TERMS)), device=work, dtype=torch.float32)
        flags = torch.zeros(n_samples, dtype=torch.int32, device=work)
        ptr = lambda v: None if v is None else v.data_ptr()
        with torch.cuda.device(work):
            stream = torch.cuda.current_stream(work).cuda_stream
            seed = offset = 0
            if on_device:
                gen = torch.cuda.default_generators[work.index]
                seed, offset = gen.initial_seed() & 0xFFFFFFFFFFFFFFFF, gen.get_offset()
            used = C.c_uint64(0)
            st = lib.dl_diffusion_loss(eng, n_samples, n_nodes, ptr(xh), ptr(nm), ptr(fm), ptr(lm), ptr(em), ptr(ctx),
                                       ptr(coef), ptr(eps), seed, offset, C.byref(used), norm, ptr(terms), ptr(flags), stream)
            _native.check(st, "dl_diffusion_loss")
            if on_device:
                gen.set_offset(offset + used.value)     # as if randn(B,N,3) and randn(B,N,F) had run (edm.py:67)
            if bool(flags.any().item()):             # the reference raises inside Dynamics.forward (egnn.py:441)
                raise nan_exception_class()(flags=flags.cpu().tolist())
        col = {k: terms[:, i] for i, k in enumerate(_native.LOSS_TERMS)}
        on = lambda v: v.reshape(-1).to(work)
        dof = col['n_linker'] * self.n_dims                                           # dimensionality, edm.py:402-403
        error_t = col['error_t']
        l2 = error_t / ((self.n_dims + self.in_node_nf) * col['n_linker'])             # edm.py:91-92
        loss_term_t = self.T * 0.5 * on(c['snr_weight']) * error_t                    # edm.py:98-99
        neg_log_constants = -(dof * (-on(c['log_sigma_x']) - 0.5 * np.log(2 * np.pi)))  # edm.py:272-280, 110
        loss_term_0 = -(col['log_p_x'] + col['log_p_h']) + neg_log_constants          # edm.py:114-115, 316
        out = dict(t_int=t_int.reshape(-1), error_t=error_t, l2=l2, loss_term_t=loss_term_t, loss_term_0=loss_term_0,
                   kl_prior=col['kl_prior'], noise=col['noise'],
                   delta_log_px=-dof * np.log(self.norm_values[0]))                    # edm.py:398-399
        return {k: v.to(dev) for k, v in out.items()}

    # ---- scalar helpers, same names/semantics as the reference -------------------------------------------------
    def sigma(self, gamma, target_tensor=None):
        return torch.sqrt(torch.sigmoid(gamma))

    def alpha(self, gamma, target_tensor=None):
        return torch.sqrt(torch.sigmoid(-gamma))

    @staticmethod
    def SNR(gamma):
        return torch.exp(-gamma)

    @staticmethod
    def sigma_and_alpha_t_given_s(gamma_t, gamma_s):
        sigma2_t_given_s = -torch.expm1(F.softplus(gamma_s) - F.softplus(gamma_t))
        alpha_t_given_s = torch.exp(0.5 * (F.logsigmoid(-gamma_t) - F.logsigmoid(-gamma_s)))
        return sigma2_t_given_s, torch.sqrt(sigma2_t_given_s), alpha_t_given_s

    def normalize(self, x, h):
        return x / self.norm_values[0], (h.float() - self.norm_biases[1]) / self.norm_values[1]

    def unnormalize(self, x, h):
        return x * self.norm_values[0], h * self.norm_values[1] + self.norm_biases[1]

    def _cpu_schedule(self):
        """The noise schedule with its gamma table on the host, for the scalar tables below."""
        gamma = PredefinedNoiseSchedule.__new__(PredefinedNoiseSchedule)
        torch.nn.Module.__init__(gamma)
        gamma.timesteps = self.gamma.timesteps
        gamma.gamma = torch.nn.Parameter(self.gamma.gamma.detach().cpu(), requires_grad=False)
        return gamma

    def step_coefficients(self, keep_frames, n_samples=1):
        """(T+1) rows of dl_step_coef: row r is reverse step s = T-1-r (edm.py:146-163, 178-208); row T is the
        final p(x,h|z_0) step (edm.py:210-235).  Evaluated on (n_samples,1) fp32 CPU tensors exactly as the
        reference does: torch's CPU transcendental kernels round differently for different tensor sizes, so this
        is what makes the scalars bit-identical to the reference's for the same batch size. Cached."""
        T = self.T
        key = (T, keep_frames, n_samples, self.gamma.gamma._version, self.gamma.gamma.data_ptr())
        if getattr(self, '_coef_cache', None) is not None and self._coef_cache[0] == key:
            return self._coef_cache[1]
        gamma = self._cpu_schedule()
        rows = (_native.DLStepCoef * (T + 1))()
        for r in range(T):
            s = T - 1 - r
            s_arr = torch.full((n_samples, 1), fill_value=s)
            t_arr = (s_arr + 1) / T                  # int64 / int -> fp32 true division, as edm.py:147-150
            s_arr = s_arr / T
            g_s, g_t = gamma(s_arr), gamma(t_arr)
            sigma2_ts, sigma_ts, alpha_ts = self.sigma_and_alpha_t_given_s(g_t, g_s)
            sigma_s, sigma_t = self.sigma(g_s), self.sigma(g_t)
            b = sigma2_ts / alpha_ts / sigma_t       # edm.py:199
            c = sigma_ts * sigma_s / sigma_t         # edm.py:202
            frame = (s * keep_frames) // T
            # only the last writer of a frame matters; frame 0 is finally overwritten by chain[0] (edm.py:174)
            last_writer = frame > 0 and (s == 0 or ((s - 1) * keep_frames) // T != frame)
            rows[r] = _native.DLStepCoef(float(t_arr[0]), float(alpha_ts[0]), float(b[0]), float(c[0]),
                                         frame if last_writer else -1, 0.0, 0.0, 0.0)
        g0 = gamma(torch.zeros(size=(n_samples, 1)))
        inv_alpha0 = 1. / self.alpha(g0)
        rows[T] = _native.DLStepCoef(0.0, float(inv_alpha0[0]), float(self.sigma(g0)[0]),
                                     float(self.SNR(-0.5 * g0)[0]), -1, 0.0, 0.0, 0.0)
        self._coef_cache = (key, rows)
        return rows

    def draw_noise(self, n_draws, n_samples, n_nodes, device, generator=None):
        """(n_draws, B, N, 3+F) standard normal. 'reference_stream': the reference's call order -- for every
        draw randn(B,N,3) then randn(B,N,F) (edm.py:328-340, utils.py:189-192) -- so seeds line up."""
        d = self.n_dims + self.in_node_nf
        if self.noise_mode == 'bulk':
            return torch.randn((n_draws, n_samples, n_nodes, d), device=device, generator=generator)
        # two launches per draw (straight into contiguous slabs: `out=` consumes the generator exactly like a fresh randn
        # of that shape) and one interleaving copy at the end, instead of four launches per draw
        zx = torch.empty((n_draws, n_samples, n_nodes, self.n_dims), device=device, dtype=torch.float32)
        zh = torch.empty((n_draws, n_samples, n_nodes, self.in_node_nf), device=device, dtype=torch.float32)
        for r in range(n_draws):
            torch.randn((n_samples, n_nodes, self.n_dims), generator=generator, out=zx[r])
            torch.randn((n_samples, n_nodes, self.in_node_nf), generator=generator, out=zh[r])
        return torch.cat([zx, zh], dim=3)

    @torch.no_grad()
    def sample_chain(self, x, h, node_mask, fragment_mask, linker_mask, edge_mask, context, keep_frames=None,
                     noise=None, batch_slice=None):
        """Same contract as the reference (edm.py:126-176): returns (keep_frames, B, N, 3+F); chain[0] holds the
        final coordinates and one-hot atom types. `noise` optionally injects the (T+2,B,N,3+F) draws (tests).
        `batch_slice=(b0, B_full)`: the inputs are rows [b0, b0+B) of a batch of B_full molecules (strong scaling,
        distributed.sample_chain_sharded); the device-side noise is then those rows of the full batch's draws."""
        lib = _native.load_library()
        n_samples, n_nodes = x.size(0), x.size(1)
        dev = x.device
        T = self.T
        if keep_frames is None:
            keep_frames = T
        else:
            assert keep_frames <= T
        d = self.n_dims + self.in_node_nf
        xn, hn = self.normalize(x, h)
        xh = torch.cat([xn, hn], dim=2).to(torch.float32).contiguous()
        # device-side stream unless a tensor is injected (tests), draw_noise is overridden on the instance, or another mode is set
        on_device = (noise is None and dev.type == 'cuda' and self.noise_mode == 'reference_stream'
                     and 'draw_noise' not in self.__dict__)
        if batch_slice is not None and not on_device:
            raise ValueError("batch_slice needs the device-side noise stream (CUDA tensors, noise_mode='reference_stream')")
        if not on_device:
            if noise is None:
                noise = self.draw_noise(T + 2, n_samples, n_nodes, dev)
            noise = noise.to(device=dev, dtype=torch.float32).contiguous()
            assert noise.shape == (T + 2, n_samples, n_nodes, d), noise.shape

        eng = self.dynamics.engine(self.dynamics._device_index(x))
        self.dynamics._check_graph_type()
        prep = lambda v, dt: None if v is None else v.detach().to(device=dev, dtype=dt).contiguous()
        nm = prep(node_mask.reshape(n_samples, n_nodes), torch.int8)
        fm = prep(fragment_mask.reshape(n_samples, n_nodes), torch.float32)
        lm = prep(linker_mask.reshape(n_samples, n_nodes), torch.float32)
        em = None
        if self.dynamics.graph_type == 'FC' and edge_mask is not None:
            em = prep(edge_mask.reshape(-1), torch.int8)
            assert em.numel() == n_samples * n_nodes * n_nodes
        ctx = None if context is None else prep(
            context.reshape(n_samples, n_nodes, self.dynamics.context_node_nf), torch.float32)   # wrong width -> raises
        coef = self.step_coefficients(keep_frames, n_samples)
        norm = (C.c_float * 3)(float(self.norm_values[0]), float(self.norm_values[1]), float(self.norm_biases[1]))
        chain = torch.empty((keep_frames, n_samples, n_nodes, d), device=dev, dtype=torch.float32)
        flags = torch.zeros(n_samples, dtype=torch.int32, device=dev)
        ptr = lambda v: None if v is None else v.data_ptr()
        if dev.type == 'cuda':
            with torch.cuda.device(dev):
                stream = torch.cuda.current_stream(dev).cuda_stream
                if on_device:
                    gen = torch.cuda.default_generators[dev.index if dev.index is not None else torch.cuda.current_device()]
                    seed, offset = gen.initial_seed() & 0xFFFFFFFFFFFFFFFF, gen.get_offset()
                    used = C.c_uint64(0)
                    if batch_slice is not None:
                        _native.check(lib.dl_set_noise_slice(eng, int(batch_slice[1]), int(batch_slice[0])), "dl_set_noise_slice")
                    st = lib.dl_sample_chain_rng(eng, _native.SAMPLER_LINKER, n_samples, n_nodes, T, keep_frames, ptr(xh),
                                                 ptr(nm), ptr(fm), ptr(lm), ptr(em), ptr(ctx), seed, offset, C.byref(used),
                                                 coef, norm, ptr(chain), ptr(flags), stream)
                    if batch_slice is not None:
                        lib.dl_set_noise_slice(eng, 0, 0)
                    _native.check(st, "dl_sample_chain_rng")
                    gen.set_offset(offset + used.value)          # as if the reference's (T+2) x 2 randn calls had run
                else:
                    st = lib.dl_sample_chain(eng, _native.SAMPLER_LINKER, n_samples, n_nodes, T, keep_frames, ptr(xh),
                                             ptr(nm), ptr(fm), ptr(lm), ptr(em), ptr(ctx), ptr(noise), coef, norm,
                                             ptr(chain), ptr(flags), stream)
                    _native.check(st, "dl_sample_chain")
                bad = bool(flags.any().item())   # one sync per chain instead of one per step (egnn.py:441)
        else:
            st = lib.dl_sample_chain_host(eng, _native.SAMPLER_LINKER, n_samples, n_nodes, T, keep_frames, ptr(xh),
                                          ptr(nm), ptr(fm), ptr(lm), ptr(em), ptr(ctx), ptr(noise), coef, norm,
                                          ptr(chain), ptr(flags))
            _native.check(st, "dl_sample_chain_host")
            bad = st == _native.DL_NAN_DETECTED
        self.last_loop_ms = float(lib.dl_last_elapsed_ms(eng))
        if bad:
            raise nan_exception_class()(flags=flags.cpu().tolist())
        return chain


class InpaintingEDM(EDM):
    """Full-molecule variant (reference: src/edm.py:466-730, sampling half): every atom is denoised by the network
    (`linker_mask=None`, dynamics built with centering=True), fragment atoms are then re-noised from the known
    fragments with q(z_s | z_t, x), and the centre of mass is projected out every step.
    NB the reference's positional order differs from EDM.sample_chain (edge_mask comes third): call by keyword."""

    def forward(self, *args, **kwargs):
        # no published config trains with inpainting; the objective of edm.py:466-547 is not ported
        raise NotImplementedError("InpaintingEDM.forward (src/edm.py:466-547) is not implemented on the native path")

    def loss_terms(self, *args, **kwargs):
        raise NotImplementedError("InpaintingEDM.forward (src/edm.py:466-547) is not implemented on the native path")

    @staticmethod
    def _com_free(x, mask):
        """utils.sample_center_gravity_zero_gaussian_with_mask (utils.py:158-168) applied to a raw draw."""
        xm = x * mask
        return xm - (xm.sum(dim=-2, keepdim=True) / mask.sum(dim=-2, keepdim=True)) * mask

    def draw_noise_inpaint(self, n_samples, n_nodes, device, node_mask, fragment_mask, generator=None):
        """(2T+3, B, N, 3+F): the reference's draws in call order, already masked and COM-projected:
        init (all atoms); per step: p(z_s|z_t) on all atoms then q(z_s|z_t,x) on fragment atoms; final p and q draws."""
        T, nd, nf = self.T, self.n_dims, self.in_node_nf
        masks = [node_mask] + [node_mask, fragment_mask] * T + [node_mask, node_mask]
        out = torch.empty((len(masks), n_samples, n_nodes, nd + nf), device=device, dtype=torch.float32)
        for r, m in enumerate(masks):
            m = m.to(device=device, dtype=torch.float32)
            out[r, :, :, :nd] = self._com_free(torch.randn((n_samples, n_nodes, nd), device=device, generator=generator), m)
            out[r, :, :, nd:] = torch.randn((n_samples, n_nodes, nf), device=device, generator=generator) * m
        return out

    def step_coefficients(self, keep_frames, n_samples=1):
        rows = super().step_coefficients(keep_frames, n_samples)
        if getattr(self, '_qcoef_key', None) == self._coef_cache[0]:
            return rows
        T = self.T
        gamma = self._cpu_schedule()
        for r in range(T):
            s = T - 1 - r
            s_arr = torch.full((n_samples, 1), fill_value=s)
            t_arr = (s_arr + 1) / T
            s_arr = s_arr / T
            g_s, g_t = gamma(s_arr), gamma(t_arr)
            sigma2_ts, _, alpha_ts = self.sigma_and_alpha_t_given_s(g_t, g_s)
            sigma_s, sigma_t, alpha_s = self.sigma(g_s), self.sigma(g_t), self.alpha(g_s)
            rows[r].qa = float((alpha_ts * (sigma_s ** 2) / (sigma_t ** 2))[0])      # edm.py:661-664
            rows[r].qb = float((alpha_s * sigma2_ts / (sigma_t ** 2))[0])
            # the chain frame is written after the COM projection by the per-molecule kernel; frame 0 is left to the final
            # step, which overwrites chain[0] with the sampled x, h (edm.py:716-725) -- hence `frame > 0`
            frame = (s * keep_frames) // T
            last_writer = (s == 0 or ((s - 1) * keep_frames) // T != frame) and frame > 0
            rows[r].frame = frame if last_writer else -1
        g0 = gamma(torch.zeros(size=(n_samples, 1)))
        rows[T].qa = float((self.sigma(g0) / self.alpha(g0))[0])                      # edm.py:716
        self._qcoef_key = self._coef_cache[0]
        return rows

    @torch.no_grad()
    def sample_chain(self, x, h, node_mask, edge_mask, fragment_mask, linker_mask, context, keep_frames=None,
                     noise=None):
        lib = _native.load_library()
        n_samples, n_nodes = x.size(0), x.size(1)
        dev = x.device
        T = self.T
        if keep_frames is None:
            keep_frames = T
        else:
            assert keep_frames <= T
        d = self.n_dims + self.in_node_nf
        xn, hn = self.normalize(x, h)
        xh = torch.cat([xn, hn], dim=2).to(torch.float32).contiguous()
        if noise is None:
            noise = self.draw_noise_inpaint(n_samples, n_nodes, dev, node_mask, fragment_mask)
        noise = noise.to(device=dev, dtype=torch.float32).contiguous()
        assert noise.shape == (2 * T + 3, n_samples, n_nodes, d), noise.shape
        eng = self.dynamics.engine(self.dynamics._device_index(x))
        self.dynamics._check_graph_type()
        prep = lambda v, dt: None if v is None else v.detach().to(device=dev, dtype=dt).contiguous()
        nm = prep(node_mask.reshape(n_samples, n_nodes), torch.int8)
        fm = prep(fragment_mask.reshape(n_samples, n_nodes), torch.float32)
        lm = prep(linker_mask.reshape(n_samples, n_nodes), torch.float32)
        em = None
        if self.dynamics.graph_type == 'FC' and edge_mask is not None:
            em = prep(edge_mask.reshape(-1), torch.int8)
        ctx = None if context is None else prep(
            context.reshape(n_samples, n_nodes, self.dynamics.context_node_nf), torch.float32)   # wrong width -> raises
        coef = self.step_coefficients(keep_frames, n_samples)
        norm = (C.c_float * 3)(float(self.norm_values[0]), float(self.norm_values[1]), float(self.norm_biases[1]))
        chain = torch.empty((keep_frames, n_samples, n_nodes, d), device=dev, dtype=torch.float32)
        flags = torch.zeros(n_samples, dtype=torch.int32, device=dev)
        ptr = lambda v: None if v is None else v.data_ptr()
        args = (eng, _native.SAMPLER_INPAINT, n_samples, n_nodes, T, keep_frames, ptr(xh), ptr(nm), ptr(fm), ptr(lm),
                ptr(em), ptr(ctx), ptr(noise), coef, norm, ptr(chain), ptr(flags))
        if dev.type == 'cuda':
            with torch.cuda.device(dev):
                st = lib.dl_sample_chain(*args, torch.cuda.current_stream(dev).cuda_stream)
                _native.check(st, "dl_sample_chain")
                bad = bool(flags.any().item())
        else:
            st = lib.dl_sample_chain_host(*args)
            _native.check(st, "dl_sample_chain_host")
            bad = st == _native.DL_NAN_DETECTED
        self.last_loop_ms = float(lib.dl_last_elapsed_ms(eng))
        if bad:
            raise nan_exception_class()(flags=flags.cpu().tolist())
        return chain
