"""``VDM`` / ``LightVDM``: variational diffusion model around the CUNet denoiser, B200-native.

Mirrors what the reference imports as ``mltools.models.vdm_model`` (constructor call:
trainVDM3D128_c_c_from_field_name_thick_lowbatch.py:128-132; sampler lines recovered from the traceback
in model_test.ipynb:678-682 = vdm_model.py:318-324, 370-378, 429-442, 531-557; ``return_ddnm`` /
``sample_zt_given_zs`` contract: src/utils.py:286-299).

The reverse ancestral loop is where the time goes (250-1000 denoiser calls per realisation).  Here
  * the schedule (gamma, alpha, sigma, c for every step) and every conditioning row the conv epilogues
    add are computed ONCE for all steps and selected on the device by a step counter,
  * one step = the CUNet trunk (vdm4cdm_b200.networks) + ONE fused update kernel (vdm_sampler_step:
    posterior mean, Philox noise in registers, and the packed bf16 network input of the next step),
  * that step is captured in a CUDA graph and replayed, so the host does nothing inside the loop,
  * realisations are independent units keyed by (seed, realisation id): shard them over ranks freely.
"""
from __future__ import annotations

import math
from typing import Optional, Sequence

import torch
import torch.nn as nn

from . import ops


class LearnedLinearSchedule(nn.Module):
    """gamma(t) = b + |w| t, initialised to [gamma_min, gamma_max]."""

    def __init__(self, gamma_min: float, gamma_max: float):
        super().__init__()
        self.b = nn.Parameter(torch.tensor(float(gamma_min)))
        self.w = nn.Parameter(torch.tensor(float(gamma_max - gamma_min)))

    def forward(self, t):
        return self.b + self.w.abs() * t

    def slope(self):
        return self.w.abs()


class FixedLinearSchedule(nn.Module):
    def __init__(self, gamma_min: float, gamma_max: float):
        super().__init__()
        self.register_buffer("b", torch.tensor(float(gamma_min)))
        self.register_buffer("w", torch.tensor(float(gamma_max - gamma_min)))

    def forward(self, t):
        return self.b + self.w * t

    def slope(self):
        return self.w


class _ZtFn(torch.autograd.Function):
    """z_t = alpha_t x + sigma_t eps in one kernel; backward = (d b, d w) of the schedule from dL/dz_t (two reductions +
    a one-block finalize), no gradient for the data or the noise."""

    @staticmethod
    def forward(ctx, x, noise, times, gamma_b, gamma_w, learned):
        ctx.save_for_backward(x, noise, times, gamma_b, gamma_w)
        ctx.learned = learned
        return ops.loss_zt(x, noise, times, gamma_b.detach(), gamma_w.detach(), learned)

    @staticmethod
    def backward(ctx, g_zt):
        x, noise, times, gamma_b, gamma_w = ctx.saved_tensors
        if not (ctx.needs_input_grad[3] or ctx.needs_input_grad[4]):
            return None, None, None, None, None, None
        g = ops.loss_zt_bwd(g_zt.contiguous(), x, noise, times, gamma_b.detach(), gamma_w.detach(), ctx.learned)
        return None, None, None, g[0].reshape(gamma_b.shape), g[1].reshape(gamma_w.shape), None


class _LossTermsFn(torch.autograd.Function):
    """(loss, [diffusion, latent, reconstruction]) from eps_hat in two kernels; backward = one elementwise kernel for
    d eps_hat and two scalar products for the schedule parameters."""

    @staticmethod
    def forward(ctx, pred, noise, x, noise0, gamma_b, gamma_w, learned, data_noise):
        out = ops.loss_terms(pred, noise, x, noise0, gamma_b.detach(), gamma_w.detach(), learned, data_noise)
        ctx.save_for_backward(pred, noise, out)
        ctx.shapes = (gamma_b.shape, gamma_w.shape)
        terms = out[1:4]
        ctx.mark_non_differentiable(terms)
        return out[0], terms

    @staticmethod
    def backward(ctx, g_loss, _g_terms):
        pred, noise, out = ctx.saved_tensors
        g = g_loss.reshape(1).float().contiguous()
        d_pred = ops.loss_dpred(pred, noise, out[4:5], g) if ctx.needs_input_grad[0] else None
        db = (g * out[5:6]).reshape(ctx.shapes[0]) if ctx.needs_input_grad[4] else None
        dw = (g * out[6:7]).reshape(ctx.shapes[1]) if ctx.needs_input_grad[5] else None
        return d_pred, None, None, None, db, dw, None, None


class VDM(nn.Module):
    def __init__(self, score_model, noise_schedule: str = "learned_linear", gamma_min: float = -13.3,
                 gamma_max: float = 13.3, antithetic_time_sampling: bool = True, data_noise: float = 1.0e-3,
                 w_cfg=None):
        super().__init__()
        self.score_model = score_model
        self.gamma_min = gamma_min
        self.gamma_max = gamma_max
        self.antithetic_time_sampling = antithetic_time_sampling
        self.data_noise = data_noise
        self.w_cfg = w_cfg
        if noise_schedule == "learned_linear":
            self.gamma = LearnedLinearSchedule(gamma_min, gamma_max)
        elif noise_schedule == "fixed_linear":
            self.gamma = FixedLinearSchedule(gamma_min, gamma_max)
        else:
            raise ValueError(f"Unknown noise schedule {noise_schedule}")
        self.use_cuda_graph = True

    # ---- schedule helpers -------------------------------------------------------------------------
    @staticmethod
    def sigma(gamma):
        return torch.sqrt(torch.sigmoid(gamma))

    @staticmethod
    def alpha(gamma):
        return torch.sqrt(torch.sigmoid(-gamma))

    def _gamma5(self, t, ref):
        if not torch.is_tensor(t):
            t = torch.full((1,), float(t), dtype=torch.float32, device=ref.device)   # no host->device copy (graph capture)
        g = self.gamma(t.to(device=ref.device, dtype=torch.float32))
        return g.reshape(-1, *([1] * (ref.dim() - 1)))

    def _t_net(self, gamma):
        return (gamma - self.gamma_min) / (self.gamma_max - self.gamma_min)

    def step_coefficients(self, t: torch.Tensor, s: torch.Tensor, final_rescale: bool = False) -> torch.Tensor:
        """fp32 [S, 4] rows (w_z, w_eps, noise_scale, out_scale) of z_s = out*(w_z z_t + w_eps eps + noise N):
        w_z = alpha_s/alpha_t, w_eps = -alpha_s/alpha_t c sigma_t, noise = sigma_s sqrt(c), c = -expm1(g_s - g_t)
        (vdm_model.py:370-378).  Evaluated in fp64 from the fp32 schedule parameters."""
        gt = self.gamma(t.float()).double()
        gs = self.gamma(s.float()).double()
        c = -torch.expm1(gs - gt)
        a_t, a_s = torch.sqrt(torch.sigmoid(-gt)), torch.sqrt(torch.sigmoid(-gs))
        s_t, s_s = torch.sqrt(torch.sigmoid(gt)), torch.sqrt(torch.sigmoid(gs))
        out = torch.ones_like(gt)
        if final_rescale:
            out[-1] = 1.0 / a_s[-1]          # x = z_0 / alpha_0 folded into the last update
        return torch.stack([a_s / a_t, -a_s / a_t * c * s_t, s_s * torch.sqrt(c), out], dim=1).float().contiguous()

    # ---- network call (vdm_model.py:318-327) -------------------------------------------------------
    def get_pred_noise(self, zt, gamma_t, **kwargs):
        t_net = self._t_net(gamma_t).reshape(-1)
        if self.w_cfg is None or self.training:
            return self.score_model(zt, t=t_net, **kwargs)
        assert "v_conditionings" in kwargs, "Need v_conditionings to mask out"
        cond = self.score_model(zt, t=t_net, **kwargs)
        masked = dict(kwargs)
        masked["v_conditionings"] = [torch.zeros_like(v) for v in kwargs["v_conditionings"]]
        uncond = self.score_model(zt, t=t_net, **masked)
        return (1.0 + self.w_cfg) * cond - self.w_cfg * uncond

    # ---- forward / reverse transitions ------------------------------------------------------------------
    def sample_zt_given_x(self, x, t, noise):
        gamma_t = self._gamma5(t, x)
        return self.alpha(gamma_t) * x + self.sigma(gamma_t) * noise, gamma_t

    @torch.no_grad()
    def sample_zs_given_zt(self, zt, t, s, return_ddnm=False, noise=None, seed=0, draw=1, realisation_id=None,
                           **kwargs):
        """One reverse step t -> s (vdm_model.py:370-378).  With ``return_ddnm`` returns
        (w_z, w_x_0t, x_0t, scale) such that z_s = w_z z + w_x_0t x_0t + scale eps (src/utils.py:296-299)."""
        dev = zt.device
        tt = torch.as_tensor(t, dtype=torch.float32, device=dev).reshape(1)
        ss = torch.as_tensor(s, dtype=torch.float32, device=dev).reshape(1)
        gamma_t = self._gamma5(tt, zt)
        pred_noise = self.get_pred_noise(zt=zt, gamma_t=gamma_t.expand(zt.shape[0], *gamma_t.shape[1:]), **kwargs)
        coef = self.step_coefficients(tt, ss)
        if return_ddnm:
            gt, gs = self.gamma(tt).double(), self.gamma(ss).double()
            c = -torch.expm1(gs - gt)
            a_t, a_s = torch.sqrt(torch.sigmoid(-gt)), torch.sqrt(torch.sigmoid(-gs))
            s_t, s_s = torch.sqrt(torch.sigmoid(gt)), torch.sqrt(torch.sigmoid(gs))
            x_0t = (zt - s_t.float() * pred_noise) / a_t.float()
            return (a_s * (1.0 - c) / a_t).float(), (a_s * c).float(), x_0t, (s_s * torch.sqrt(c)).float()
        return ops.sampler_step(zt.contiguous().float(), pred_noise.contiguous(), coef, seed=seed,
                                realisation_id=realisation_id, draw_base=draw, noise=noise)

    @torch.no_grad()
    def sample_zt_given_zs(self, zs, t, s, noise=None, seed=0, draw=1, realisation_id=None):
        """Forward re-noising s -> t: z_t = alpha_t/alpha_s z_s + sigma_t sqrt(c) eps (used by DDNM time travel)."""
        dev = zs.device
        tt = torch.as_tensor(t, dtype=torch.float32, device=dev).reshape(1)
        ss = torch.as_tensor(s, dtype=torch.float32, device=dev).reshape(1)
        gt, gs = self.gamma(tt).double(), self.gamma(ss).double()
        c = -torch.expm1(gs - gt)
        a_t, a_s = torch.sqrt(torch.sigmoid(-gt)), torch.sqrt(torch.sigmoid(-gs))
        s_t = torch.sqrt(torch.sigmoid(gt))
        coef = torch.stack([a_t / a_s, torch.zeros_like(c), s_t * torch.sqrt(c), torch.ones_like(c)], dim=1).float()
        zs = zs.contiguous().float()
        return ops.sampler_step(zs, zs, coef.contiguous(), seed=seed, realisation_id=realisation_id, draw_base=draw,
                                noise=noise)

    # ---- ancestral sampling loop (vdm_model.py:429-442) ---------------------------------------------------
    @torch.no_grad()
    def sample(self, batch_size, n_sampling_steps, device, z=None, return_all=False, verbose=False, seed=0,
               realisation_ids: Optional[Sequence[int]] = None, noise_fn=None, s_conditioning=None,
               v_conditionings=None):
        """x (B, 1, D, H, W) fp32 after ``n_sampling_steps`` reverse steps from z_1 ~ N(0, I).

        Noise is counter based: realisation r, draw d (0 = initial latent, i+1 = step i), element e ->
        Philox4x32-10(seed; e/4, d, r) + Box-Muller, so a realisation does not depend on the batch it
        was sampled in.  ``noise_fn(draw, shape)`` injects noise instead (parity tests)."""
        dev = torch.device(device)
        if self.w_cfg is not None and not self.training:
            return self._sample_generic(batch_size, n_sampling_steps, dev, z, return_all, seed, realisation_ids,
                                        noise_fn, s_conditioning=s_conditioning, v_conditionings=v_conditionings)
        sess = self.session(batch_size, n_sampling_steps, dev, z=z, seed=seed, realisation_ids=realisation_ids,
                            noise_fn=noise_fn, s_conditioning=s_conditioning, v_conditionings=v_conditionings,
                            fold_final_rescale=not return_all)
        zs = []
        it = range(n_sampling_steps)
        if verbose:
            from tqdm import trange
            it = trange(n_sampling_steps, desc="sampling")
        for _ in it:
            sess.step()
            if return_all:
                zs.append(sess.z.clone())
        if return_all:
            x = sess.z / self.alpha(self.gamma(sess.steps[-1]))
            return torch.stack(zs + [x], dim=0)
        return sess.z.clone()

    def session(self, batch_size, n_sampling_steps, device, **kw) -> "SamplerSession":
        """A (cached) ``SamplerSession`` for this batch size / step count, reset to a new chain."""
        key = (batch_size, n_sampling_steps, str(device), kw.get("s_conditioning") is not None,
               0 if kw.get("v_conditionings") is None else len(kw["v_conditionings"]),
               getattr(self.score_model, "precision", "bf16"))
        cache = self.__dict__.setdefault("_sessions", {})
        sess = cache.get(key)
        if sess is None:
            cache.clear()                      # one resident session: its buffers are O(GB) at 128^3
            sess = SamplerSession(self, batch_size, n_sampling_steps, device, **kw)
            cache[key] = sess
        else:
            sess.reset(**kw)
        return sess

    def _sample_generic(self, batch_size, n_sampling_steps, dev, z, return_all, seed, realisation_ids, noise_fn, **kw):
        """Step-by-step loop through ``sample_zs_given_zt`` (classifier-free guidance needs two network calls)."""
        shape = (batch_size, *self.score_model.shape)
        rid = None if realisation_ids is None else torch.as_tensor(list(realisation_ids), dtype=torch.int32, device=dev)
        if z is None:
            z = noise_fn(0, shape).to(dev).float() if noise_fn is not None else ops.philox_normal(shape, seed, 0, rid, dev)
        steps = torch.linspace(1.0, 0.0, n_sampling_steps + 1, device=dev)
        zs = []
        for i in range(n_sampling_steps):
            noise = noise_fn(i + 1, shape).to(dev).float().contiguous() if noise_fn is not None else None
            z = self.sample_zs_given_zt(zt=z, t=steps[i], s=steps[i + 1], noise=noise, seed=seed, draw=i + 1,
                                        realisation_id=rid, **kw)
            if return_all:
                zs.append(z)
        x = z / self.alpha(self.gamma(steps[-1]))
        return torch.stack(zs + [x], dim=0) if return_all else x

    # ---- training loss (continuous-time VDM, Kingma et al. 2021) -----------------------------------------
    def sample_times(self, batch_size, device, t0=None):
        if self.antithetic_time_sampling:
            if t0 is None:
                t0 = torch.rand((), device=device)
            return torch.remainder(t0 + torch.arange(batch_size, device=device) / batch_size, 1.0)
        return torch.rand(batch_size, device=device)

    def get_loss(self, x, noise=None, noise0=None, times=None, **kwargs):
        """Continuous-time VDM loss in bits per dimension, plus its three terms (batch means).

        Everything that touches a B x N^3 tensor runs in the kernels of csrc/vdm_loss.cu (z_t, the three per-sample sums,
        d eps_hat, the schedule gradients through z_t); torch autograd only carries gamma(t) into the time embedding."""
        bsz = x.shape[0]
        x = x.float().contiguous()
        if times is None:
            times = self.sample_times(bsz, x.device)
        if noise is None:
            noise = torch.randn_like(x)
        if noise0 is None:
            noise0 = torch.randn_like(x)
        times = times.to(device=x.device, dtype=torch.float32).contiguous()
        noise, noise0 = noise.float().contiguous(), noise0.float().contiguous()
        learned = isinstance(self.gamma, LearnedLinearSchedule)
        gb, gw = self.gamma.b, self.gamma.w
        zt = _ZtFn.apply(x, noise, times, gb, gw, learned)
        pred = self.get_pred_noise(zt, self._gamma5(times, x), **kwargs)
        loss, terms = _LossTermsFn.apply(pred.float().contiguous(), noise, x, noise0, gb, gw, learned, float(self.data_noise))
        return loss, {"diffusion_loss": terms[0], "latent_loss": terms[1], "reconstruction_loss": terms[2]}


class SamplerSession:
    """State of one ancestral chain for a batch of realisations: latent z (fp32), packed bf16 network
    input, per-step coefficient and conditioning tables, the device step counter, and the CUDA graph
    of one step.  ``step()`` advances every realisation by one reverse step; ``reset()`` starts a new
    chain in the same buffers, so the captured graph is reused across ``draw_samples`` calls."""

    def __init__(self, vdm: VDM, batch_size: int, n_sampling_steps: int, device, **kw):
        self.vdm, self.net, self.dev = vdm, vdm.score_model, torch.device(device)
        self.n_steps = n_sampling_steps
        self.shape = (batch_size, *self.net.shape)
        dev = self.dev
        self.z = torch.empty(self.shape, dtype=torch.float32, device=dev)
        self.eps = torch.empty(self.shape, dtype=torch.float32, device=dev)
        self.noise_buf = torch.empty(self.shape, dtype=torch.float32, device=dev)
        self.cond_buf = None
        # packed network input in the net's precision (bf16 [B, 2, D, H, W, 8] or, TF32, fp32 [B, 2, D, H, W, 4])
        self.tf32 = getattr(self.net, "precision", "bf16") == "tf32"
        self.c_pad = self.net.input_channels_pad()
        lanes = 4 if self.tf32 else 8
        self.packed = torch.empty((batch_size, self.c_pad // lanes) + tuple(self.net.shape[1:]) + (lanes,),
                                  dtype=torch.float32 if self.tf32 else torch.bfloat16, device=dev)
        self.step_idx = torch.zeros(1, dtype=torch.int32, device=dev)
        self.rid_buf = torch.zeros(batch_size, dtype=torch.int32, device=dev)
        self.steps = torch.linspace(1.0, 0.0, n_sampling_steps + 1, device=dev)
        self.coef = torch.empty((n_sampling_steps, 4), dtype=torch.float32, device=dev)
        self.rows = None
        self.graph = None
        self.graph_key = None
        self.kernels_per_step = 0
        self.reset(**kw)

    @torch.no_grad()
    def reset(self, z=None, seed: int = 0, realisation_ids: Optional[Sequence[int]] = None, noise_fn=None,
              s_conditioning=None, v_conditionings=None, fold_final_rescale: bool = True):
        vdm, net, dev = self.vdm, self.net, self.dev
        batch_size = self.shape[0]
        net.refresh_packed()
        self.seed = seed
        self.noise_fn = noise_fn
        if realisation_ids is not None:
            rid = torch.as_tensor(list(realisation_ids), dtype=torch.int32, device=dev)
            assert rid.numel() == batch_size
            self.rid_buf.copy_(rid)
        else:
            self.rid_buf.copy_(torch.arange(batch_size, dtype=torch.int32, device=dev))
        if z is not None:
            self.z.copy_(z.to(dev).float().reshape(self.shape))
        elif noise_fn is not None:
            self.z.copy_(noise_fn(0, self.shape).to(dev).float())
        else:
            self.z.copy_(ops.philox_normal(self.shape, seed, 0, self.rid_buf, device=dev))
        self.coef.copy_(vdm.step_coefficients(self.steps[:-1], self.steps[1:], final_rescale=fold_final_rescale))
        t_net = vdm._t_net(vdm.gamma(self.steps[:-1]).float())                         # (S,)
        vc = None if v_conditionings is None else [v.to(dev) for v in v_conditionings]
        rows = net.chan_add_rows(batch_size, t_net[:, None].expand(-1, batch_size), vc, dev)
        if self.rows is None:
            self.rows = rows
        else:
            for k, v in rows.items():
                self.rows[k].copy_(v)
        if s_conditioning is not None:
            c = s_conditioning.to(dev).float()
            if self.cond_buf is None:
                self.cond_buf = c.contiguous().clone()
            else:
                self.cond_buf.copy_(c)
        elif self.cond_buf is not None:
            raise ValueError("a session created with spatial conditioning must be reset with one")
        ops.pack_input(self.z, self.cond_buf, self.c_pad, out=self.packed)
        self.step_idx.zero_()
        self.done = 0
        # the graph bakes in pointers and the (seed, injected-noise or Philox) choice, nothing else
        key = (seed, noise_fn is not None)
        if key != self.graph_key:
            self.graph = None
            self.graph_key = key

    def _one_step(self):
        n0 = ops.launch_count()
        # NVTX ranges (no-ops without a profiler): `ncu --nvtx --nvtx-include "vdm.sampler_step/"` / Nsight Systems timelines
        with torch.cuda.nvtx.range("vdm.sampler_step"):
            with torch.cuda.nvtx.range("vdm.denoiser"):
                self.net.run_packed(self.packed, self.rows, step_ptr=self.step_idx, out=self.eps)
            self._update()
        self.kernels_per_step = ops.launch_count() - n0

    def _update(self):
        # (TF32: the fused update writes bf16 input planes only, so the fp32 input is re-packed by its own launch)
        ops.sampler_step(self.z, self.eps, self.coef, out=self.z, step_ptr=self.step_idx, seed=self.seed,
                         realisation_id=self.rid_buf, draw_base=1,
                         noise=self.noise_buf if self.noise_fn is not None else None, cond=self.cond_buf,
                         packed_out=None if self.tf32 else self.packed)
        if self.tf32:
            ops.pack_input(self.z, self.cond_buf, self.c_pad, out=self.packed)
        ops.increment(self.step_idx)

    @torch.no_grad()
    def step(self):
        assert self.done < self.n_steps, "chain already finished"
        if self.noise_fn is not None:
            self.noise_buf.copy_(self.noise_fn(self.done + 1, self.shape))
        if not self.vdm.use_cuda_graph or (self.graph is None and self.done == 0):
            self._one_step()                       # eager: also warms the buffer arena and weight caches
        elif self.graph is None:
            torch.cuda.synchronize(self.dev)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self._one_step()               # capture records the launches, it does not run them
            self.graph.replay()
        else:
            self.graph.replay()
        self.done += 1


class LightVDM(nn.Module):
    """Lightning-free ``LightVDM`` (ctor: trainVDM3D128_c_c_from_field_name_thick_lowbatch.py:128-132;
    ``draw_samples`` -> ``self.model.sample(..., device=self.device, ...)``: vdm_model.py:531-557)."""

    def __init__(self, score_model, draw_figure=None, gamma_min=-13.3, gamma_max=13.3,
                 noise_schedule="learned_linear", learning_rate=3.0e-4, **vdm_kwargs):
        super().__init__()
        self.model = VDM(score_model, noise_schedule=noise_schedule, gamma_min=gamma_min, gamma_max=gamma_max,
                         **vdm_kwargs)
        self.draw_figure = draw_figure
        self.learning_rate = learning_rate

    @property
    def device(self):
        return next(self.parameters()).device

    def get_loss(self, batch, **kw):
        return self.model.get_loss(batch["x"], s_conditioning=batch.get("conditioning"),
                                   v_conditionings=batch.get("conditioning_values"), **kw)

    def training_step(self, batch, batch_idx=0):
        return self.get_loss(batch)[0]

    def validation_step(self, batch, batch_idx=0):
        with torch.no_grad():
            return self.get_loss(batch)[0]

    def configure_optimizers(self):
        return torch.optim.AdamW(self.parameters(), lr=self.learning_rate)

    def draw_samples(self, batch_size, n_sampling_steps=250, verbose=False, return_all=False, **kwargs):
        return self.model.sample(batch_size=batch_size, n_sampling_steps=n_sampling_steps, device=self.device,
                                 verbose=verbose, return_all=return_all, **kwargs)
