"""GaussianDiffusion / SpacedDiffusion — sampling half of MuseDiffusion/models/diffusion.py, same names and
signatures, with the per-step arithmetic executed by the fused sm_100a kernels of the C-ABI library.

What is mirrored (reference file:line):
  get_named_beta_schedule / betas_for_alpha_bar(_left)   diffusion.py:22-118
  GaussianDiffusion.__init__ tables                       :136-185   (float64 numpy, cast to fp32 at upload as :914 does)
  q_sample                                                :229-255
  q_posterior_mean_variance / p_mean_variance / p_sample  :257-404
  p_sample_loop(_progressive)                             :406-540
  ddim_sample / ddim_sample_loop(_progressive)            :701-757, :797-901
  space_timesteps / SpacedDiffusion / _WrappedModel       :920-1032
Beyond the reference: dpm_solver_sample_loop, the DPM-Solver++(2M) sampler (md_dpm_solver_step) for tens of evaluations.
Training losses (:187-192, :542-699) are out of scope (SURVEY.md section 8) and raise NotImplementedError.

Noise.  The reference draws `torch.randn_like` every step (plus a host-synchronising rejection loop for top_p).
Here noise is generated inside the posterior kernel by a counter-based Philox stream keyed by
(torch.initial_seed(), call counter, global element index), so results do not depend on how a batch is sharded.
Set `diffusion.noise_source = fn(shape, kind) -> Tensor` (kind in {"randn", "truncated"}) to inject external noise
instead — the parity tests do this to feed the oracle's exact stream."""
import math

import numpy as np
import torch

from . import _lib, ops
from .rounding import rounding_weight_of


# ------------------------------------------------------------------------------------------------ schedules
def betas_for_alpha_bar(num_diffusion_timesteps, alpha_bar, max_beta=0.999):
    """diffusion.py:101-118."""
    T = num_diffusion_timesteps
    return np.array([min(1 - alpha_bar((i + 1) / T) / alpha_bar(i / T), max_beta) for i in range(T)])


def betas_for_alpha_bar_left(num_diffusion_timesteps, alpha_bar, max_beta=0.999):
    """diffusion.py:80-98: like betas_for_alpha_bar with an extra leading beta and one step fewer."""
    T = num_diffusion_timesteps
    head = [min(1 - alpha_bar(0), max_beta)]
    return np.array(head + [min(1 - alpha_bar((i + 1) / T) / alpha_bar(i / T), max_beta) for i in range(T - 1)])


def get_named_beta_schedule(schedule_name, num_diffusion_timesteps):
    """diffusion.py:22-77."""
    T = num_diffusion_timesteps
    scale = 1000 / T
    if schedule_name == "linear":
        return np.linspace(scale * 0.0001, scale * 0.02, T, dtype=np.float64)
    if schedule_name == "cosine":
        return betas_for_alpha_bar(T, lambda t: math.cos((t + 0.008) / 1.008 * math.pi / 2) ** 2)
    if schedule_name == "sqrt":
        return betas_for_alpha_bar(T, lambda t: 1 - np.sqrt(t + 0.0001))
    if schedule_name == "trunc_cos":
        return betas_for_alpha_bar_left(T, lambda t: np.cos((t + 0.1) / 1.1 * np.pi / 2) ** 2)
    if schedule_name == "trunc_lin":
        return np.linspace(scale * 0.0001 + 0.01, scale * 0.02 + 0.01, T, dtype=np.float64)
    if schedule_name == "pw_lin":
        lo, mid, hi = scale * 0.0001 + 0.01, scale * 0.0001, scale * 0.02
        return np.concatenate([np.linspace(lo, mid, 10, dtype=np.float64), np.linspace(mid, hi, T - 10, dtype=np.float64)])
    raise NotImplementedError(f"unknown beta schedule: {schedule_name}")


def space_timesteps(num_timesteps, section_counts):
    """diffusion.py:920-969."""
    if isinstance(section_counts, str):
        if section_counts.startswith("ddim"):
            want = int(section_counts[len("ddim"):])
            for stride in range(1, num_timesteps):
                if len(range(0, num_timesteps, stride)) == want:
                    return set(range(0, num_timesteps, stride))
            raise ValueError(f"cannot create exactly {num_timesteps} steps with an integer stride")
        section_counts = [int(x) for x in section_counts.split(",")]
    per, extra = divmod(num_timesteps, len(section_counts))
    start, steps = 0, []
    for i, count in enumerate(section_counts):
        size = per + (1 if i < extra else 0)
        if size < count:
            raise ValueError(f"cannot divide section of {size} steps into {count}")
        stride = 1 if count <= 1 else (size - 1) / (count - 1)
        pos = 0.0
        for _ in range(count):
            steps.append(start + round(pos))
            pos += stride
        start += size
    return set(steps)


def _extract_into_tensor(arr, timesteps, broadcast_shape):
    """diffusion.py:904-917 (API parity; the kernels read the same fp32 values from constant memory).  `arr` may also be
    the table already uploaded to the timesteps' device."""
    if not isinstance(arr, torch.Tensor):
        arr = torch.from_numpy(np.asarray(arr)).to(device=timesteps.device)
    res = arr[timesteps].float()
    while res.dim() < len(broadcast_shape):
        res = res[..., None]
    return res.expand(broadcast_shape)


# ------------------------------------------------------------------------------------------------ diffusion
_capture_state = {}          # device index -> [most recent graph, capture stream], kept for the life of the process


def _capture(dev, fn):
    """Record `fn`'s launches into a new CUDA graph.  Plain capture_begin / capture_end on a side stream instead of the
    `torch.cuda.graph` context: the context empties the caching allocator (device and pinned host) on entry, which at
    the bench size means returning and re-acquiring ~10 GB of step activations on EVERY sampling call (60-230 ms per
    call, measured with tools/e2e_overhead.py).  Every capture on a device allocates from the memory pool of the previous
    one (which is kept alive until the new graph exists, so the pool never dies): the step's temporaries are free blocks
    of that pool again by the time a capture ends, and the next call's capture takes the same blocks.  Only the newest
    graph of a device is ever replayed."""
    index = dev.index if dev.index is not None else torch.cuda.current_device()
    state = _capture_state.setdefault(index, [None, torch.cuda.Stream(device=dev)])
    previous, side = state
    graph = torch.cuda.CUDAGraph()
    main = torch.cuda.current_stream(dev)
    side.wait_stream(main)
    with torch.cuda.stream(side):
        graph.capture_begin(pool=previous.pool() if previous is not None else torch.cuda.graph_pool_handle())
        try:
            fn()
        finally:
            graph.capture_end()
    main.wait_stream(side)
    state[0] = graph
    return graph


def _noise_kind(mode, top_p):
    """(noise kind, top_p of the posterior kernel) of one reverse step: DDPM with top_p > 0 draws truncated noise;
    ddim_sample ignores top_p (diffusion.py:738)."""
    if mode == _lib.STEP_DDPM and top_p is not None and top_p > 0:
        return "truncated", top_p
    return "randn", 0.0


def _collect(steps, only_last):
    """the list p_sample_loop / ddim_sample_loop return: a copy of every sample (the loops reuse their buffers), or the
    last sample alone (an empty list for an empty chain)."""
    final = []
    for sample, _, _, _ in steps:
        if only_last:
            final = [sample]
        else:
            final.append(sample.clone())
    return final


def _log_snr(alphas_cumprod):
    """lambda_i = log alpha_i - log sigma_i of every index, alpha_i = sqrt(abar_i), sigma_i = sqrt(1 - abar_i) (float64)."""
    ab = np.asarray(alphas_cumprod, dtype=np.float64)
    return 0.5 * np.log(ab) - 0.5 * np.log1p(-ab)


def dpm_solver_indices(alphas_cumprod, t_start, steps):
    """The `steps` evaluation indices of dpm_solver_sample_loop: t_start = s_0 > s_1 > ... > s_{N-1} = 0 (N = 1: [t_start]).
    The targets are uniform in lambda: g_k is the fractional index whose lambda (interpolated in the table) is the k-th of N
    evenly spaced values from lambda[t_start] to lambda[0]; s_k = clip(round(g_k), N - 1 - k, s_{k-1} - 1) keeps the N
    indices distinct."""
    T = len(alphas_cumprod)
    t_start, steps = int(t_start), int(steps)
    if not 0 <= t_start < T:
        raise ValueError("t_start=%d outside the schedule's %d indices" % (t_start, T))
    if not 1 <= steps <= t_start + 1:
        raise ValueError("steps=%d: DPM-Solver++ needs 1 <= steps <= t_start + 1 = %d" % (steps, t_start + 1))
    lam = _log_snr(alphas_cumprod)[:t_start + 1]
    grid = np.arange(t_start + 1, dtype=np.float64)
    g = np.interp(np.linspace(lam[t_start], lam[0], steps), lam[::-1], grid[::-1])     # lambda decreases with the index
    s = [t_start]
    for k in range(1, steps):
        s.append(int(min(max(np.rint(g[k]), steps - 1 - k), s[-1] - 1)))
    return s


def dpm_solver_coefficients(alphas_cumprod, indices, order):
    """float64 [N, 4] rows (a, b, c0, c1) of md_dpm_solver_step for the evaluation indices (DPM-Solver++(2M), Lu et al. 2022,
    Algorithm 2).  Step k < N - 1 goes from c = s_k to n = s_{k+1}, h = lambda_n - lambda_c: a = sigma_n / sigma_c,
    b = -alpha_n expm1(-h); the first step (and every step at order 1) uses D = x0_k (c0 = 1, c1 = 0), later ones
    D = (1 + 1/(2r)) x0_k - 1/(2r) x0_{k-1} with r = h_{k-1} / h.  The last row (0, 1, 1, 0) returns x0_{N-1} itself."""
    if order not in (1, 2):
        raise ValueError("DPM-Solver++ order must be 1 or 2, got %r" % (order,))
    ab = np.asarray(alphas_cumprod, dtype=np.float64)
    lam = _log_snr(ab)
    alpha, sigma = np.sqrt(ab), np.sqrt(1.0 - ab)
    rows, h_prev = [], None
    for k in range(len(indices)):
        if k == len(indices) - 1:
            rows.append((0.0, 1.0, 1.0, 0.0))
            break
        c, n = indices[k], indices[k + 1]
        h = lam[n] - lam[c]
        a, b = sigma[n] / sigma[c], -alpha[n] * np.expm1(-h)
        if order == 1 or h_prev is None:
            rows.append((a, b, 1.0, 0.0))
        else:
            r = h_prev / h
            rows.append((a, b, 1.0 + 1.0 / (2.0 * r), -1.0 / (2.0 * r)))
        h_prev = h
    return np.array(rows, dtype=np.float64).reshape(-1, 4)


class GaussianDiffusion:
    """Sampling utilities with the reference's attribute and method names (diffusion.py:121-901)."""

    noise_source = None     # optional callable(shape, kind) -> CUDA float tensor; None = in-kernel Philox
    rounding_trace = None   # optional list: every fused rounding call appends (ids int32 [M], top-2 margin fp32 [M]) clones
    use_cuda_graph = True   # loops of >= GRAPH_MIN_STEPS steps replay captured CUDA graphs of the reverse step (fused path only)
    GRAPH_MIN_STEPS = 4
    seq_offset = 0          # global index of this rank's first sequence (keeps Philox noise shard-invariant)

    def __init__(self, *, betas, predict_xstart, rescale_timesteps=False, training_mode="s2s"):
        self.rescale_timesteps = rescale_timesteps
        self.predict_xstart = predict_xstart
        self.training_mode = training_mode
        betas = np.array(betas, dtype=np.float64)
        self.betas = betas
        assert betas.ndim == 1 and (betas > 0).all() and (betas <= 1).all()
        self.num_timesteps = int(betas.shape[0])
        alphas = 1.0 - betas
        self.alphas_cumprod = np.cumprod(alphas, axis=0)
        self.alphas_cumprod_prev = np.append(1.0, self.alphas_cumprod[:-1])
        self.alphas_cumprod_next = np.append(self.alphas_cumprod[1:], 0.0)
        self.sqrt_alphas_cumprod = np.sqrt(self.alphas_cumprod)
        self.sqrt_one_minus_alphas_cumprod = np.sqrt(1.0 - self.alphas_cumprod)
        self.log_one_minus_alphas_cumprod = np.log(1.0 - self.alphas_cumprod)
        self.sqrt_recip_alphas_cumprod = np.sqrt(1.0 / self.alphas_cumprod)
        self.sqrt_recipm1_alphas_cumprod = np.sqrt(1.0 / self.alphas_cumprod - 1)
        self.posterior_variance = betas * (1.0 - self.alphas_cumprod_prev) / (1.0 - self.alphas_cumprod)
        self.posterior_log_variance_clipped = np.log(np.append(self.posterior_variance[1], self.posterior_variance[1:]))
        self.posterior_mean_coef1 = betas * np.sqrt(self.alphas_cumprod_prev) / (1.0 - self.alphas_cumprod)
        self.posterior_mean_coef2 = (1.0 - self.alphas_cumprod_prev) * np.sqrt(alphas) / (1.0 - self.alphas_cumprod)
        # fixed-large model variance used by p_mean_variance (diffusion.py:313-317)
        self.model_variance = np.append(self.posterior_variance[1], self.betas[1:])
        self.model_log_variance = np.log(self.model_variance)
        self._noise_calls = 0
        self._sched_token = object()

    # -------------------------------------------------------------------------------------- plumbing
    def _upload_schedule(self):
        """fp32 coefficient tables -> __constant__ memory (once; re-uploaded only if another schedule displaced them)."""
        if ops.current_schedule_key() is not self._sched_token:
            ops.set_schedule({n: getattr(self, n) for n in ops.TABLE_ORDER}, key=self._sched_token)

    def _next_counter(self):
        self._noise_calls += 1
        return self._noise_calls

    @staticmethod
    def _seed():
        return int(torch.initial_seed()) & 0xFFFFFFFFFFFFFFFF

    def _external_noise(self, shape, kind, device):
        if self.noise_source is None:
            return None
        n = self.noise_source(tuple(shape), kind)
        if not isinstance(n, torch.Tensor):
            n = torch.from_numpy(np.ascontiguousarray(n))
        return n.to(device=device, dtype=torch.float32)

    def _scale_timesteps(self, t):
        """diffusion.py:207-210."""
        if self.rescale_timesteps:
            return t.float() * (1000.0 / self.num_timesteps)
        return t

    def training_losses(self, *a, **k):
        raise NotImplementedError("training is outside the scope of musediffusion_b200 (sampling hot path only)")

    # -------------------------------------------------------------------------------------- forward noising
    def q_sample(self, x_start, t, noise=None, mask=None):
        """diffusion.py:229-255.  x_start [B, ...]; t holds one index per sequence ([B] or [B, 1], as
        run/sample.py:196-197 passes it); mask (already broadcastable to x_start once unsqueezed) keeps x_start
        where it is 0."""
        self._upload_schedule()
        shape = x_start.shape
        B = shape[0]
        x3, m3 = x_start, mask
        if x_start.dim() == 4 and shape[-1] == 1:          # run/sample.py:197 passes [B, L, D, 1]
            x3 = x_start.squeeze(-1)
        elif x_start.dim() != 3:
            x3 = x_start.reshape(B, 1, -1)
            if mask is not None:
                m3 = torch.broadcast_to(mask.unsqueeze(-1), shape).reshape(B, 1, -1)
        if noise is None:
            noise = self._external_noise(shape, "randn", x_start.device)
        if noise is not None:
            noise = noise.reshape(x3.shape)
        out = ops.q_sample(x3, t.reshape(-1), noise=noise, seed=self._seed(), step_counter=self._next_counter(),
                           seq_offset=self.seq_offset, mask=m3)
        return out.view(shape)

    def _predict_xstart_from_eps(self, x_t, t, eps):
        """diffusion.py:194-199."""
        self._upload_schedule()
        return ops.xstart_from_eps(x_t, eps, t)

    # -------------------------------------------------------------------------------------- one reverse step
    def _model_timesteps(self, t):
        """value fed to the denoiser for schedule index t (overridden by SpacedDiffusion)."""
        return self._scale_timesteps(t)

    def _call_model(self, model, x, t, model_kwargs):
        """diffusion.py:309: `model(x, self._scale_timesteps(t), model_kwargs=model_kwargs)` — the kwarg is passed
        whole and the reference model drops it (network.py:131), which is preserved for arbitrary callables."""
        return model(x, self._model_timesteps(t), model_kwargs=model_kwargs if model_kwargs is not None else {})

    def _step(self, mode, model, x, t, clip_denoised, denoised_fn, model_kwargs, top_p, mask, x_start, eta,
              want_aux=True, model_output=None, out_bf16=None, noise=None):
        """Shared body of p_sample / ddim_sample / the generic loop: model call, rounding, fused posterior kernel.
        `noise`: the step's noise; None takes it from `noise_source`, or draws it in the kernel when that is None too."""
        self._upload_schedule()
        B = x.shape[0]
        assert t.numel() in (1, B)
        if model_output is None:
            model_output = self._call_model(model, x, t, model_kwargs)
        E, idx, pred = self._processed_x0(x, t, model_output, denoised_fn)
        kind, tp = _noise_kind(mode, top_p)
        if noise is None:
            noise = self._external_noise(x.shape, kind, x.device)
        pred_out = torch.empty_like(x, dtype=torch.float32) if want_aux else None
        mean_out = torch.empty_like(x, dtype=torch.float32) if want_aux else None
        sample = ops.posterior_step(
            x, t, mode, idx=idx, pred=pred, E=E, noise=noise, seed=self._seed(), step_counter=self._next_counter(),
            seq_offset=self.seq_offset, mask=mask, x_start=x_start, eta=eta, clip=clip_denoised, top_p=tp, out_bf16=out_bf16,
            pred_out=pred_out, mean_out=mean_out)
        return sample, pred_out, mean_out

    def _processed_x0(self, x, t, model_output, denoised_fn):
        """x0 of one step as the posterior / DPM kernels take it -> (E, idx, pred): the model output (through
        xstart_from_eps for an eps-predicting model), then rounded (ids into E, gathered by the kernel) when `denoised_fn`
        is our rounding callback, or passed through an arbitrary `denoised_fn`; the kernels clip after that."""
        B = x.shape[0]
        if not self.predict_xstart:
            model_output = ops.xstart_from_eps(x, model_output, t)
        E = rounding_weight_of(denoised_fn)
        idx = pred = None
        if E is not None:
            # fused distance contraction + row argmin on the tensor cores (rounding.py:21-28)
            trace = self.rounding_trace
            idx = ops.round_argmin_tc(model_output, ops.split_embedding(E), want_margin=trace is not None)
            if trace is not None:
                idx, margin = idx
                trace.append((idx.clone(), margin))
        elif denoised_fn is not None:
            pred = denoised_fn(model_output, t if t.numel() == B else t.expand(B))   # arbitrary user callable
        else:
            pred = model_output
        return E, idx, pred

    def q_posterior_mean_variance(self, x_start, x_t, t):
        """diffusion.py:257-278."""
        self._upload_schedule()
        mean = torch.empty_like(x_t, dtype=torch.float32)
        zeros = torch.zeros_like(mean)
        ops.posterior_step(x_t, t, _lib.STEP_DDPM, pred=x_start, noise=zeros, clip=False, mean_out=mean)
        return (mean, _extract_into_tensor(self.posterior_variance, t, x_t.shape),
                _extract_into_tensor(self.posterior_log_variance_clipped, t, x_t.shape))

    def _mean_variance(self, mean, pred, t, shape, tables=None):
        """p_mean_variance's dict (diffusion.py:343-347), with the fixed-large model variance of schedule index t.
        `tables`: (model_variance, model_log_variance) already on t's device (`_variance_tables`)."""
        var, log_var = tables if tables is not None else (self.model_variance, self.model_log_variance)
        return {"mean": mean, "variance": _extract_into_tensor(var, t.long(), shape),
                "log_variance": _extract_into_tensor(log_var, t.long(), shape), "pred_xstart": pred}

    def _variance_tables(self, device):
        """the two float64 model-variance tables on `device`, uploaded once per progressive loop instead of once per step"""
        return tuple(torch.from_numpy(a).to(device) for a in (self.model_variance, self.model_log_variance))

    def p_mean_variance(self, model, x, t, clip_denoised=True, denoised_fn=None, model_kwargs=None):
        """diffusion.py:280-347: dict(mean, variance, log_variance, pred_xstart)."""
        _, pred, mean = self._step(_lib.STEP_DDPM, model, x, t, clip_denoised, denoised_fn, model_kwargs, None, None, None,
                                   0.0, noise=torch.zeros_like(x, dtype=torch.float32))
        return self._mean_variance(mean, pred, t, x.shape)

    def p_sample(self, model, x, t, clip_denoised=True, denoised_fn=None, model_kwargs=None, top_p=None, mask=None,
                 x_start=None):
        """diffusion.py:349-404."""
        sample, pred, mean = self._step(_lib.STEP_DDPM, model, x, t, clip_denoised, denoised_fn, model_kwargs, top_p,
                                        mask, x_start, 0.0)
        return {"sample": sample, "pred_xstart": pred, "greedy_mean": mean, "out": self._mean_variance(mean, pred, t, x.shape)}

    def ddim_sample(self, model, x, t, clip_denoised=True, denoised_fn=None, model_kwargs=None, eta=0.0,
                    langevin_fn=None, mask=None, x_start=None):
        """diffusion.py:701-757.  `langevin_fn(sample, mean_pred, sigma, alpha_bar_prev[t[0]], t, x)` (:748-750) is applied
        to the un-masked sample; the mask select that follows it (:752-755) is md_q_sample's `mask == 0 ? x_start : sample`."""
        if not langevin_fn:
            sample, pred, _ = self._step(_lib.STEP_DDIM, model, x, t, clip_denoised, denoised_fn, model_kwargs, None, mask,
                                         x_start, eta)
            return {"sample": sample, "pred_xstart": pred}
        sample, pred, mean_pred = self._step(_lib.STEP_DDIM, model, x, t, clip_denoised, denoised_fn, model_kwargs, None, None,
                                             None, eta)
        tt = t.reshape(-1).long()
        ab, abp = self.alphas_cumprod, self.alphas_cumprod_prev
        sigma_tab = eta * np.sqrt((1 - abp) / (1 - ab)) * np.sqrt(1 - ab / abp)
        sigma = _extract_into_tensor(sigma_tab, tt if tt.numel() == x.shape[0] else tt.expand(x.shape[0]), x.shape)
        sample = langevin_fn(sample, mean_pred, sigma, self.alphas_cumprod_prev[int(tt[0])], t, x)
        if mask is not None:
            sample = ops.q_sample(sample.new_empty(0) if x_start is None else x_start.to(torch.float32).contiguous(), None,
                                  noise=sample.to(torch.float32).contiguous(), mask=mask)
        return {"sample": sample, "pred_xstart": pred}

    # -------------------------------------------------------------------------------------- loops
    def _fast_model(self, model):
        """our CUDA denoiser behind `model` (possibly wrapped), or None for arbitrary callables."""
        from .network import TransformerNetModel
        inner = model.model if isinstance(model, _WrappedModel) else model
        return inner if isinstance(inner, TransformerNetModel) else None

    def _loop_inputs(self, model, shape, noise, device, mask, x_start):
        """-> (device, x, mask, x_start) of a loop: the starting state (`noise`, else `noise_source`, else a Philox draw keyed by
        the next noise counter), and the mask and x_start converted once so that the per-step kernel calls allocate nothing."""
        if device is None:
            device = next(model.parameters()).device
        assert isinstance(shape, (tuple, list))
        if noise is not None:
            x = noise
        else:
            x = self._external_noise(shape, "randn", device)
            if x is None:
                x = ops.fill_normal(tuple(shape), device, seed=self._seed(), step_counter=self._next_counter(),
                                    elem_offset=self.seq_offset * int(np.prod(shape[1:])))
        if mask is not None:
            # the (usually int64, stride-0 expanded) mask as int32, still a stride-0 expand where it was one
            m = torch.broadcast_to(mask if mask.dim() == len(shape) else mask.unsqueeze(-1), tuple(shape))
            if m.stride(-1) == 0:
                mask = m[..., 0].to(torch.int32).contiguous().unsqueeze(-1).expand(tuple(shape))
            else:
                mask = m.to(torch.int32).contiguous()
        if x_start is not None:
            x_start = x_start.to(torch.float32).contiguous()
        return device, x.to(torch.float32).contiguous(), mask, x_start

    def _loop(self, mode, model, shape, noise, clip_denoised, denoised_fn, model_kwargs, device, progress, top_p,
              clamp_step, clamp_first, mask, x_start, eta, indices, want_aux):
        """Generator of (sample, pred_xstart, mean, t) per reverse step.  Our denoiser, in-kernel noise, a [B, L, D] state
        and `denoised_fn` either our rounding or None: the fused step bodies of `_fused_loop` (progressive loops, clamp
        gating and `rounding_trace` included), replayed as captured CUDA graphs for chains of >= GRAPH_MIN_STEPS steps
        unless `use_cuda_graph` is off or `ops.profile_step` is timing the launches.  What cannot be captured (arbitrary
        `model` / `denoised_fn` callables, `noise_source`, other state shapes) runs step by step through `_step`; with our
        denoiser there the posterior kernel also emits the bf16 operand of the next step's first GEMM, and the batch shares
        one time-embedding row (all sequences share t inside the loops, diffusion.py:516,887)."""
        device, x, mask, x_start = self._loop_inputs(model, shape, noise, device, mask, x_start)
        fast = self._fast_model(model)
        B = shape[0]
        if len(indices) == 0:
            return
        idx_list = list(indices)
        t_idx = torch.tensor(idx_list, dtype=torch.int32, device=device)
        t_model = self._model_timesteps(t_idx.long()).float()
        if progress:
            from tqdm.auto import tqdm
            indices = tqdm(idx_list)
        else:
            indices = idx_list

        def rounds_at(i):
            """clamp gating, diffusion.py:517-526 (the DDIM loop always rounds, :889-899); like the reference, the DDPM loop
            raises TypeError when clamp_step is left at its default None"""
            if mode != _lib.STEP_DDPM:
                return True
            return (i >= clamp_step) if clamp_first else not (i > clamp_step)

        E = rounding_weight_of(denoised_fn)
        if fast is not None and self.noise_source is None and (E is not None or denoised_fn is None) and x.dim() == 3:
            rounds = [rounds_at(i) and E is not None for i in idx_list]
            capture = self.use_cuda_graph and len(idx_list) >= self.GRAPH_MIN_STEPS and ops._PROFILE[0] is None
            yield from self._fused_loop(mode, fast, x, E, t_idx, t_model, indices, rounds, clip_denoised, top_p, mask, x_start,
                                        eta, want_aux, capture)
            return
        x_bf16 = None
        for k, i in enumerate(indices):
            fn = denoised_fn if rounds_at(i) else None
            if fast is not None:
                t_arg = t_idx[k:k + 1]
                model_output = fast.denoise(x, t_model[k:k + 1], x_bf16=x_bf16, uniform_t=True)
                Dp = fast.weight_pack().Dp          # padded operand width: its pad columns stay zero, the kernel never writes them
                x_bf16 = (torch.empty_like(x, dtype=torch.bfloat16) if Dp == x.shape[-1]
                          else torch.zeros(x.shape[:-1] + (Dp,), dtype=torch.bfloat16, device=x.device))
            else:
                t_arg, model_output = t_idx[k:k + 1].long().expand(B), None
            x, pred, mean = self._step(mode, model, x, t_arg, clip_denoised, fn, model_kwargs, top_p, mask, x_start, eta,
                                       want_aux=want_aux, model_output=model_output, out_bf16=x_bf16)
            yield x, pred, mean, t_arg

    def _fused_loop(self, mode, fast, x, E, t_idx, t_model, indices, rounds, clip_denoised, top_p, mask, x_start, eta,
                    want_aux, capture):
        """The chain as fixed reverse-step bodies whose per-step inputs live in device memory: `md_step_advance` moves a
        cursor over the index tables and publishes the schedule index, the denoiser's timestep value and the Philox
        counter of the step, which the posterior kernel reads.  x_t is updated in place (the posterior kernel is
        elementwise) and its bf16 copy, padded to the operand width Dp with zero columns, feeds the next step's first GEMM.
        `rounds[k]`: step k rounds to the embedding (`round_step`) or posts the model's x0 as is (`plain_step`, clamp
        gating, diffusion.py:517-526).  Clamp gating splits a chain into at most two contiguous runs of one body.
        `capture`: the first step of each run runs eagerly (one-time set-up: shared-memory attributes, weight pack, tensor
        maps, workspaces), the second is captured as a CUDA graph (SURVEY.md section 7 step 7) and every later step of the
        run replays it.  A run's graph is captured from the pool of the previous run's, which is never replayed again, so
        every buffer one body hands to the other is allocated here, before either capture.  Otherwise every step launches
        its body directly, so per-launch timings measure the kernels a replay runs.
        `want_aux` (progressive loops): the posterior kernel also writes pred_xstart and the mean, and every step yields
        clones of sample, pred_xstart and mean, which stay valid after later steps.  `rounding_trace`: the rounding kernel
        writes its top-2 margins and every rounding step appends clones of ids and margins."""
        dev = x.device
        self._upload_schedule()
        x = x.clone()                                   # updated in place: never the caller's tensor
        pk = fast.weight_pack()
        xb = ops.cast_bf16(x, width=pk.Dp)
        any_round, any_plain = any(rounds), not all(rounds)
        # x0-predicting model: the last Linear of a rounding step emits the [hi | lo] bf16 split that the rounding
        # contraction consumes, the fp32 model output never exists there; an eps-predicting model needs it in fp32 for
        # x0 = sr x_t - srm1 eps first, and a plain step hands it to the posterior kernel
        use_split = self.predict_xstart and pk.has_down
        mo = torch.empty_like(x) if any_plain or not use_split else None
        mo_split = torch.empty(x.shape[:-1] + (2 * pk.Dp,), dtype=torch.bfloat16, device=dev) if use_split and any_round else None
        cursor = torch.zeros(1, dtype=torch.int32, device=dev)
        t_cur = torch.zeros(1, dtype=torch.int32, device=dev)
        tm_cur = torch.zeros(1, dtype=torch.float32, device=dev)
        ctr_cur = torch.zeros(1, dtype=torch.int64, device=dev)
        ctr_base = self._noise_calls + 1                # the value _next_counter() hands to the first step of an eager loop
        seed = self._seed()
        M = x.shape[0] * x.shape[1]
        idx = torch.empty((M,), dtype=torch.int32, device=dev)
        trace = self.rounding_trace if any_round else None
        margin = torch.empty((M,), dtype=torch.float32, device=dev) if trace is not None else None
        pred_out = torch.empty_like(x) if want_aux else None
        mean_out = torch.empty_like(x) if want_aux else None
        if any_round:
            se = ops.split_embedding(E)
            # clip_denoised after rounding = gathering rows of clamp(E, -1, 1): built once per embedding matrix, not per
            # token and step
            E_step, clip_step = (se.E_clamped, 2) if clip_denoised else (E, 0)
        _, tp = _noise_kind(mode, top_p)
        post = dict(seed=seed, seq_offset=self.seq_offset, mask=mask, x_start=x_start, eta=eta, top_p=tp, out=x, out_bf16=xb,
                    pred_out=pred_out, mean_out=mean_out, step_counter_dev=ctr_cur)

        def model_x0():
            out = fast.denoise(x, tm_cur, x_bf16=xb, uniform_t=True, out=mo)
            return out if self.predict_xstart else ops.xstart_from_eps(x, out, t_cur)

        def round_step():
            ops.step_advance(cursor, t_idx, t_model, t_cur, tm_cur, ctr_cur, ctr_base)
            if use_split:
                fast.denoise(x, tm_cur, x_bf16=xb, uniform_t=True, split_out=mo_split)
                ops.round_argmin_tc(None, se, out=idx, presplit=mo_split, margin_out=margin)
            else:
                ops.round_argmin_tc(model_x0(), se, out=idx, margin_out=margin)
            ops.posterior_step(x, t_cur, mode, idx=idx, E=E_step, clip=clip_step, **post)

        def plain_step():
            ops.step_advance(cursor, t_idx, t_model, t_cur, tm_cur, ctr_cur, ctr_base)
            ops.posterior_step(x, t_cur, mode, pred=model_x0(), clip=clip_denoised, **post)

        graph, nodes = None, 0
        for k, i in enumerate(indices):
            body = round_step if rounds[k] else plain_step
            run_start = k == 0 or rounds[k] != rounds[k - 1]
            if run_start or not capture:
                graph = None
                body()
            else:
                if graph is None:
                    before = ops.launch_count()
                    graph = _capture(dev, body)
                    nodes = ops.launch_count() - before          # kernels recorded by the capture (nothing ran yet)
                    ops.add_launches(-nodes)
                graph.replay()
                ops.add_launches(nodes)
            self._noise_calls += 1
            if trace is not None and rounds[k]:
                trace.append((idx.clone(), margin.clone()))
            if want_aux:
                yield x.clone(), pred_out.clone(), mean_out.clone(), t_idx[k:k + 1]
            else:
                yield x, None, None, t_idx[k:k + 1]

    def p_sample_loop(self, model, shape, noise=None, clip_denoised=True, denoised_fn=None, model_kwargs=None,
                      device=None, progress=False, top_p=None, clamp_step=None, clamp_first=None, mask=None,
                      x_start=None, gap=1, eta=0.0, t_enc=None, only_last=False):
        """diffusion.py:406-473.  Returns a list of samples (one element when only_last)."""
        indices = list(range(self.num_timesteps))[::-1][slice(t_enc)]
        return _collect(self._loop(_lib.STEP_DDPM, model, shape, noise, clip_denoised, denoised_fn, model_kwargs, device,
                                   progress, top_p, clamp_step, clamp_first, mask, x_start, eta, indices, want_aux=False),
                        only_last)

    def p_sample_loop_progressive(self, model, shape, noise=None, clip_denoised=True, denoised_fn=None,
                                  model_kwargs=None, device=None, progress=False, top_p=None, clamp_step=None,
                                  clamp_first=None, mask=None, x_start=None, eta=0.0, t_enc=None):
        """diffusion.py:475-540: generator of p_sample dicts."""
        indices = list(range(self.num_timesteps))[::-1][slice(t_enc)]
        tables = None
        for sample, pred, mean, t in self._loop(_lib.STEP_DDPM, model, shape, noise, clip_denoised, denoised_fn,
                                                model_kwargs, device, progress, top_p, clamp_step, clamp_first, mask,
                                                x_start, eta, indices, want_aux=True):
            if tables is None:
                tables = self._variance_tables(t.device)
            yield {"sample": sample, "pred_xstart": pred, "greedy_mean": mean,
                   "out": self._mean_variance(mean, pred, t, sample.shape, tables)}

    def ddim_sample_loop(self, model, shape, noise=None, clip_denoised=True, denoised_fn=None, model_kwargs=None,
                         device=None, progress=False, top_p=None, clamp_step=None, clamp_first=None, mask=None,
                         x_start=None, gap=1, eta=0.0, t_enc=None, only_last=False):
        """diffusion.py:797-846 (top_p / clamp_step / clamp_first accepted and ignored, like the reference)."""
        indices = list(range(self.num_timesteps))[::-1][::gap][slice(t_enc)]
        return _collect(self._loop(_lib.STEP_DDIM, model, shape, noise, clip_denoised, denoised_fn, model_kwargs, device,
                                   progress, None, 0, True, mask, x_start, eta, indices, want_aux=False), only_last)

    def ddim_sample_loop_progressive(self, model, shape, noise=None, clip_denoised=True, denoised_fn=None,
                                     model_kwargs=None, device=None, progress=False, eta=0.0, langevin_fn=None,
                                     mask=None, x_start=None, gap=1, t_enc=None):
        """diffusion.py:848-901 (`langevin_fn` is accepted and, as in the reference, never handed to ddim_sample :866-877)."""
        indices = list(range(self.num_timesteps))[::-1][::gap][slice(t_enc)]
        for sample, pred, _, _ in self._loop(_lib.STEP_DDIM, model, shape, noise, clip_denoised, denoised_fn,
                                             model_kwargs, device, progress, None, 0, True, mask, x_start, eta, indices,
                                             want_aux=True):
            yield {"sample": sample, "pred_xstart": pred}

    # -------------------------------------------------------------------------------------- DPM-Solver++(2M)
    def dpm_solver_sample_loop(self, model, shape, noise=None, clip_denoised=True, denoised_fn=None, model_kwargs=None,
                               device=None, progress=False, mask=None, x_start=None, steps=20, t_start=None, order=2,
                               only_last=False):
        """DPM-Solver++(2M) (Lu et al., "DPM-Solver++", 2022, Algorithm 2; order=1 is its first-order form, DDIM at eta = 0):
        `steps` model evaluations at the indices of `dpm_solver_indices` from `t_start` (default: the last index) down
        to 0, starting from `noise` (the state at t_start; drawn like the other loops when None).  Each evaluation's x0 is
        processed as in ddim_sample_loop (rounded when `denoised_fn` rounds, then clipped) and the last one is returned as
        is.  The sampler draws no noise.  Not part of the reference, which samples with DDPM / DDIM only.  Returns the state
        after every evaluation, the last being x0 (one element when only_last)."""
        t_start = self.num_timesteps - 1 if t_start is None else int(t_start)
        indices = dpm_solver_indices(self.alphas_cumprod, t_start, steps)
        coef = dpm_solver_coefficients(self.alphas_cumprod, indices, order).astype(np.float32)
        return _collect(self._dpm_loop(model, shape, noise, clip_denoised, denoised_fn, model_kwargs, device, progress, mask,
                                       x_start, indices, coef), only_last)

    def _dpm_loop(self, model, shape, noise, clip_denoised, denoised_fn, model_kwargs, device, progress, mask, x_start, indices,
                  coef):
        """Generator of (state, None, None, t) per evaluation; path selection as in `_loop`: the fused body of
        `_dpm_fused_loop` (graph-replayed for >= GRAPH_MIN_STEPS evaluations) or, for what cannot be captured, one
        md_dpm_solver_step per evaluation with that evaluation's coefficient row."""
        device, x, mask, x_start = self._loop_inputs(model, shape, noise, device, mask, x_start)
        self._upload_schedule()
        fast = self._fast_model(model)
        B = shape[0]
        t_idx = torch.tensor(indices, dtype=torch.int32, device=device)
        t_model = self._model_timesteps(t_idx.long()).float()
        coef = torch.from_numpy(coef).to(device)
        ks = range(len(indices))
        if progress:
            from tqdm.auto import tqdm
            ks = tqdm(ks)
        E = rounding_weight_of(denoised_fn)
        if fast is not None and self.noise_source is None and (E is not None or denoised_fn is None) and x.dim() == 3:
            capture = self.use_cuda_graph and len(indices) >= self.GRAPH_MIN_STEPS and ops._PROFILE[0] is None
            yield from self._dpm_fused_loop(fast, x, E, t_idx, t_model, coef, ks, clip_denoised, mask, x_start, capture)
            return
        hist = torch.empty_like(x)              # x0 of the previous evaluation (first-order rows never read it)
        x_bf16 = None
        for k in ks:
            if fast is not None:
                t_arg = t_idx[k:k + 1]
                model_output = fast.denoise(x, t_model[k:k + 1], x_bf16=x_bf16, uniform_t=True)
                Dp = fast.weight_pack().Dp
                x_bf16 = (torch.empty_like(x, dtype=torch.bfloat16) if Dp == x.shape[-1]
                          else torch.zeros(x.shape[:-1] + (Dp,), dtype=torch.bfloat16, device=x.device))
            else:
                t_arg = t_idx[k:k + 1].long().expand(B)
                model_output = self._call_model(model, x, t_arg, model_kwargs)
            E, idx, pred = self._processed_x0(x, t_arg, model_output, denoised_fn)
            x = ops.dpm_solver_step(x, coef[k:k + 1], hist, idx=idx, pred=pred, E=E, mask=mask, x_start=x_start,
                                    clip=clip_denoised, out_bf16=x_bf16)
            yield x, None, None, t_arg

    def _dpm_fused_loop(self, fast, x, E, t_idx, t_model, coef, ks, clip_denoised, mask, x_start, capture):
        """`_fused_loop`'s structure with one body for every evaluation: md_step_advance -> denoiser (the last Linear emits
        the split the rounding consumes) -> md_round_argmin_tc -> md_dpm_solver_step, which takes its coefficient row at the
        cursor and updates x_t, its padded bf16 copy and the x0 history in place.  Everything the body touches is allocated
        here, before the capture; the first evaluation runs eagerly, the second is captured and every later one replays it."""
        dev = x.device
        x = x.clone()
        pk = fast.weight_pack()
        xb = ops.cast_bf16(x, width=pk.Dp)
        use_split = E is not None and self.predict_xstart and pk.has_down
        mo = None if use_split else torch.empty_like(x)
        mo_split = torch.empty(x.shape[:-1] + (2 * pk.Dp,), dtype=torch.bfloat16, device=dev) if use_split else None
        cursor = torch.zeros(1, dtype=torch.int32, device=dev)
        t_cur = torch.zeros(1, dtype=torch.int32, device=dev)
        tm_cur = torch.zeros(1, dtype=torch.float32, device=dev)
        ctr_cur = torch.zeros(1, dtype=torch.int64, device=dev)      # published by md_step_advance, unused: no noise
        hist = torch.empty_like(x)
        M = x.shape[0] * x.shape[1]
        trace = self.rounding_trace if E is not None else None
        idx = torch.empty((M,), dtype=torch.int32, device=dev) if E is not None else None
        margin = torch.empty((M,), dtype=torch.float32, device=dev) if trace is not None else None
        if E is not None:
            se = ops.split_embedding(E)
            E_step, clip_step = (se.E_clamped, 2) if clip_denoised else (E, 0)
        post = dict(cursor=cursor, mask=mask, x_start=x_start, out=x, out_bf16=xb)

        def model_x0():
            out = fast.denoise(x, tm_cur, x_bf16=xb, uniform_t=True, out=mo)
            return out if self.predict_xstart else ops.xstart_from_eps(x, out, t_cur)

        def body():
            ops.step_advance(cursor, t_idx, t_model, t_cur, tm_cur, ctr_cur, 0)
            if E is None:
                ops.dpm_solver_step(x, coef, hist, pred=model_x0(), clip=clip_denoised, **post)
                return
            if use_split:
                fast.denoise(x, tm_cur, x_bf16=xb, uniform_t=True, split_out=mo_split)
                ops.round_argmin_tc(None, se, out=idx, presplit=mo_split, margin_out=margin)
            else:
                ops.round_argmin_tc(model_x0(), se, out=idx, margin_out=margin)
            ops.dpm_solver_step(x, coef, hist, idx=idx, E=E_step, clip=clip_step, **post)

        graph, nodes = None, 0
        for k in ks:
            if k == 0 or not capture:
                body()
            else:
                if graph is None:
                    before = ops.launch_count()
                    graph = _capture(dev, body)
                    nodes = ops.launch_count() - before          # kernels recorded by the capture (nothing ran yet)
                    ops.add_launches(-nodes)
                graph.replay()
                ops.add_launches(nodes)
            if trace is not None:
                trace.append((idx.clone(), margin.clone()))
            yield x, None, None, t_idx[k:k + 1]


class SpacedDiffusion(GaussianDiffusion):
    """diffusion.py:972-1018: a diffusion process that keeps only `use_timesteps` of a base process."""

    def __init__(self, use_timesteps, **kwargs):
        self.use_timesteps = set(use_timesteps)
        self.timestep_map = []
        self.original_num_steps = len(kwargs["betas"])
        base = GaussianDiffusion(**kwargs)
        last, new_betas = 1.0, []
        for i, ac in enumerate(base.alphas_cumprod):
            if i in self.use_timesteps:
                new_betas.append(1 - ac / last)
                last = ac
                self.timestep_map.append(i)
        kwargs["betas"] = np.array(new_betas)
        super().__init__(**kwargs)

    def _wrap_model(self, model):
        if isinstance(model, _WrappedModel):
            return model
        return _WrappedModel(model, self.timestep_map, self.rescale_timesteps, self.original_num_steps)

    def _scale_timesteps(self, t):
        return t                                   # scaling is done by the wrapped model (diffusion.py:1015-1017)

    def _model_timesteps(self, t):
        """_WrappedModel.__call__ (diffusion.py:1027-1032) without the per-step H2D copy of the map."""
        m = getattr(self, "_map_dev", None)
        if m is None or m.device != t.device:
            m = torch.tensor(self.timestep_map, device=t.device, dtype=torch.long)
            self._map_dev = m
        new_ts = m[t.long()]
        if self.rescale_timesteps:
            new_ts = new_ts.float() * (1000.0 / self.original_num_steps)
        return new_ts

    def _call_model(self, model, x, t, model_kwargs):
        inner = model.model if isinstance(model, _WrappedModel) else model
        return inner(x, self._model_timesteps(t), model_kwargs=model_kwargs if model_kwargs is not None else {})

    def p_mean_variance(self, model, *args, **kwargs):
        return super().p_mean_variance(self._wrap_model(model), *args, **kwargs)


class _WrappedModel:
    """diffusion.py:1020-1032."""

    def __init__(self, model, timestep_map, rescale_timesteps, original_num_steps):
        self.model = model
        self.timestep_map = timestep_map
        self.rescale_timesteps = rescale_timesteps
        self.original_num_steps = original_num_steps

    def __call__(self, x, ts, **kwargs):
        map_tensor = torch.tensor(self.timestep_map, device=ts.device, dtype=ts.dtype)
        new_ts = map_tensor[ts]
        if self.rescale_timesteps:
            new_ts = new_ts.float() * (1000.0 / self.original_num_steps)
        return self.model(x, new_ts, **kwargs)


def unwrap_model(model, unwrap_parallel=True):
    """diffusion.py:1035-1041."""
    if isinstance(model, _WrappedModel):
        return unwrap_model(model.model)
    if isinstance(model, (torch.nn.parallel.DistributedDataParallel, torch.nn.parallel.DataParallel)) and unwrap_parallel:
        return unwrap_model(model.module)
    return model
