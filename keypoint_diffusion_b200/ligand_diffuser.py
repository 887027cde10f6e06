"""Drop-in KeypointDiffusion for the sampling hot path.

Same constructor, state_dict layout and sampling API as the reference's
models/ligand_diffuser.py:24-538; the 1000-step loop of sample_from_encoded_receptors runs as a
replayed CUDA graph inside libkpdiff_b200.so (ops.Sampler).  Training (`forward`, losses) is
out of scope (SURVEY.md section 8: sampling only) and raises NotImplementedError.
"""
import math
import numbers
import os
from math import ceil
from pathlib import Path
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn as nn

from . import hetero, ops
from .dynamics import LigRecDynamics, LigRecDynamicsGVP
from .n_nodes_dist import LigandSizeDistribution
from .receptor_encoder import ReceptorEncoder, ReceptorEncoderGVP
from .schedule import (SOLVERS, PredefinedNoiseSchedule, alpha, coefficient_rows, coefficient_table, frame_levels,
                       inpaint_rows, inpaint_table, multistep_rows, prediction_rows, prediction_table, sigma,
                       sigma_and_alpha_t_given_s, start_coefficients, step_grid)
from .utils import get_batch_idxs, split_bounds

DEFAULT_SUB_BATCHES = {"gvp": 4, "egnn": 2}      # measured on B200: profiles/r01_sweep_sub_batches_*.txt


class FixedReceptorEncoder(nn.Module):
    """reference models/receptor_encoder_fixed.py:9-66: keypoints := receptor atoms, kk := rr."""

    def __init__(self, n_vec_feats):
        super().__init__()
        self.n_vec_feats = n_vec_feats

    def forward(self, g, batch_idxs=None):
        rec = g.nodes["rec"].data
        nd = {"kp": {"x_0": rec["x_0"], "h_0": rec["h_0"]},
              "lig": dict(g.nodes["lig"].data),
              "rec": {k: v[:0] for k, v in rec.items()}}
        if self.n_vec_feats is not None:
            nd["kp"]["v_0"] = torch.zeros((rec["x_0"].shape[0], self.n_vec_feats, 3), device=g.device)
        zeros = torch.zeros_like(g.batch_num_nodes("rec"))
        rr = g.edges(form="uv", etype="rr")
        return hetero.HeteroBatch({"kp": g.batch_num_nodes("rec"), "lig": g.batch_num_nodes("lig"), "rec": zeros},
                                  nd, {("kp", "kk", "kp"): rr}, {("kp", "kk", "kp"): g.batch_num_edges("rr")})


class KeypointDiffusion(nn.Module):

    def __init__(self, atom_nf, rec_nf, processed_dataset_dir: Path, n_timesteps: int = 1000, keypoint_centered=False,
                 architecture: str = 'egnn', rec_encoder_type: str = 'learned', graph_config={}, dynamics_config={},
                 rec_encoder_config={}, rec_encoder_loss_config={}, precision=1e-4, lig_feat_norm_constant=1,
                 rl_dist_threshold=0, use_fake_atoms=False):
        super().__init__()
        self.n_lig_features = atom_nf
        self.n_kp_feat = rec_nf
        self.n_timesteps = n_timesteps
        self.lig_feat_norm_constant = lig_feat_norm_constant
        self.use_fake_atoms = use_fake_atoms
        self.rec_encoder_type = rec_encoder_type
        if architecture not in ['egnn', 'gvp']:
            raise ValueError(f'Unsupported architecture: {architecture}')
        self.architecture = architecture
        if use_fake_atoms:
            # dead and broken in the reference (SURVEY A8: torch.cumsum without dim, max_fake_atom_frac 0 everywhere)
            raise NotImplementedError("use_fake_atoms is not supported (no shipped config enables it)")
        self.lig_size_dist = LigandSizeDistribution(processed_dataset_dir=Path(processed_dataset_dir))
        self.gamma = PredefinedNoiseSchedule(noise_schedule='polynomial_2', timesteps=n_timesteps, precision=precision)
        dynamics_config = dict(dynamics_config)
        if 'no_cg' in rec_encoder_config:
            dynamics_config['no_cg'] = rec_encoder_config['no_cg']
        dynamics_class = LigRecDynamics if architecture == 'egnn' else LigRecDynamicsGVP
        self.dynamics = dynamics_class(atom_nf, rec_nf, **graph_config, **dynamics_config)
        if rec_encoder_type not in ['learned', 'fixed']:
            raise ValueError(f'Receptor encoder type must be either "learned" or "fixed". Got {rec_encoder_type=} instead.')
        if rec_encoder_type == 'learned':
            encoder_class = ReceptorEncoder if architecture == 'egnn' else ReceptorEncoderGVP
            self.rec_encoder = encoder_class(**graph_config, **rec_encoder_config)
        else:
            self.rec_encoder = FixedReceptorEncoder(rec_encoder_config['vector_size'] if architecture == 'gvp' else None)
        object.__setattr__(self, "_samplers", {})
        object.__setattr__(self, "_coef", {})
        object.__setattr__(self, "_coef2", {})
        object.__setattr__(self, "_pred", {})
        object.__setattr__(self, "_schedules", {})
        object.__setattr__(self, "last_launches_per_step", 0)
        object.__setattr__(self, "_streams", {})
        object.__setattr__(self, "cold_captures", 0)       # capacity buckets captured so far (a cold call each)

    # ------------------------------------------------------------------ training (out of scope)
    def forward(self, complex_graphs, interface_points=None):
        raise NotImplementedError("training is outside the sampling hot path this package implements")

    # ------------------------------------------------------------------ small helpers with reference names
    def normalize(self, g):
        g.nodes['lig'].data['h_0'] = g.nodes['lig'].data['h_0'] / self.lig_feat_norm_constant
        return g

    def unnormalize(self, g):
        g.nodes['lig'].data['h_0'] = g.nodes['lig'].data['h_0'] * self.lig_feat_norm_constant
        return g

    def sigma(self, gamma):
        return sigma(gamma)

    def alpha(self, gamma):
        return alpha(gamma)

    def sigma_and_alpha_t_given_s(self, gamma_t, gamma_s):
        return sigma_and_alpha_t_given_s(gamma_t, gamma_s)

    def _layout(self, g):
        return self.dynamics._layout(g)

    def remove_com(self, g, lig_batch_idx=None, kp_batch_idx=None, com: str = None):
        """reference :185-203 -- in place on g's lig / kp x_0, through kpd_remove_com."""
        if com is None:
            raise NotImplementedError('removing COM of receptor/ligand complex not implemented')
        if com not in ('ligand', 'receptor'):
            raise ValueError(f'invalid value for com: {com=}')
        batch, _ = self._layout(g)
        x_lig = g.nodes['lig'].data['x_0'].float().contiguous()
        x_kp = g.nodes['kp'].data['x_0'].float().contiguous()
        ops.remove_com(batch, x_lig, x_kp, com)
        g.nodes['lig'].data['x_0'] = x_lig
        g.nodes['kp'].data['x_0'] = x_kp
        return g

    def encode_receptors(self, g):
        return self.rec_encoder(g, get_batch_idxs(g))

    def coef_table(self, device) -> torch.Tensor:
        key = (str(device), self.gamma.gamma._version, self.gamma.gamma.data_ptr())
        if key not in self._coef:
            self._coef.clear()
            self._coef[key] = coefficient_table(self.gamma.gamma, self.n_timesteps).to(device)
        return self._coef[key]

    def inpaint_coef_table(self, device) -> torch.Tensor:
        """schedule.inpaint_table on `device`, cached like coef_table."""
        key = (str(device), self.gamma.gamma._version, self.gamma.gamma.data_ptr())
        if key not in self._coef2:
            self._coef2.clear()
            self._coef2[key] = inpaint_table(self.gamma.gamma, self.n_timesteps).to(device)
        return self._coef2[key]

    def prediction_coef_table(self, device) -> torch.Tensor:
        """schedule.prediction_table on `device`, cached like coef_table."""
        key = (str(device), self.gamma.gamma._version, self.gamma.gamma.data_ptr())
        if key not in self._pred:
            self._pred.clear()
            self._pred[key] = prediction_table(self.gamma.gamma, self.n_timesteps).to(device)
        return self._pred[key]

    MAX_CACHED_SCHEDULES = 8

    def schedule_tables(self, device, t_start: int, n: int, eta: Optional[float] = None, inpaint: bool = False,
                        solver: Optional[str] = None):
        """(coef [n,4], coef2 [n,4] or None, pred [n,2]) on `device`: the rows of the n-step grid over [0, t_start]
        (schedule.step_grid), ancestral (eta=None) or DDIM(eta) (schedule.coefficient_rows), with inpaint=True the
        fragment rows over the same grid (schedule.inpaint_rows), and the (alpha_t, sigma_t) rows a recorded trajectory
        reads (schedule.prediction_rows).  solver="dpmpp_2m" (eta must be None): coef holds the DDIM eta = 0 rows, and
        a fourth element, ms [n,4], the DPM-Solver++(2M) rows (schedule.multistep_rows).  n scalar rows cost
        milliseconds on the host; the last few schedules are cached (per device and gamma version), least recently
        used evicted first."""
        key = (str(device), self.gamma.gamma._version, self.gamma.gamma.data_ptr(), int(t_start), int(n),
               None if eta is None else float(eta), bool(inpaint), solver)
        hit = self._schedules.pop(key, None)
        if hit is None:
            grid, T, g = step_grid(t_start, n), self.n_timesteps, self.gamma.gamma
            hit = (coefficient_rows(g, T, grid, 0.0 if solver else eta).to(device),
                   inpaint_rows(g, T, grid).to(device) if inpaint else None, prediction_rows(g, T, grid).to(device))
            if solver:
                hit = hit + (multistep_rows(g, T, grid).to(device),)
            while len(self._schedules) >= self.MAX_CACHED_SCHEDULES:
                self._schedules.pop(next(iter(self._schedules)))
        self._schedules[key] = hit
        return hit

    # ------------------------------------------------------------------ one reverse step (reference :497-538)
    @torch.no_grad()
    def sample_p_zs_given_zt(self, s: torch.Tensor, t: torch.Tensor, g, batch_idxs=None, noise=None,
                             seed: Optional[int] = None):
        """Mutates lig x_0/h_0 and kp x_0 of g in place and returns g.  ``noise=(pos_noise, feat_noise)``
        injects the Gaussian draws (parity); otherwise Philox keyed by (seed, step, atom, channel).  With seed=None
        (default) a fresh seed is drawn from torch's global generator on every call, so a caller driving the
        reference-style per-step loop gets new noise per step, per batch and per run, and torch.manual_seed makes it
        reproducible -- like the reference's torch.randn draws (ligand_diffuser.py:520-527).  An explicit seed is
        deterministic: same (seed, step, atom, channel) -> same draw.

        Like the reference, any t > s is a step: t_int = round(t T) must exceed s_int = round(s T) (ValueError
        otherwise).  A strided step (t_int > s_int + 1) uses the row (s_int, t_int) of schedule.coefficient_rows; its
        Philox draws stay keyed by s_int."""
        T = self.n_timesteps
        s_int = int(torch.round(s.flatten()[0] * T).item())
        t_int = int(torch.round(t.flatten()[0] * T).item())
        if not s_int < t_int <= T:
            raise ValueError(f"a reverse step needs s < t <= 1, got s = {s_int}/{T}, t = {t_int}/{T}")
        if seed is None and noise is None:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        seed = 0 if seed is None else seed
        batch, _ = self._layout(g)
        eps_h, eps_x = self.dynamics(g, t, batch_idxs)
        step = torch.tensor([s_int], dtype=torch.int32, device=g.device)
        coef = self.coef_table(g.device)
        if t_int != s_int + 1:      # the kernel reads row s_int: the strided row goes there
            coef = torch.zeros(s_int + 1, 4, device=g.device)
            coef[s_int] = coefficient_rows(self.gamma.gamma, T, [s_int, t_int])[0].to(g.device)
        x_lig = g.nodes['lig'].data['x_0'].float().contiguous()
        h_lig = g.nodes['lig'].data['h_0'].float().contiguous()
        x_kp = g.nodes['kp'].data['x_0'].float().contiguous()
        nx, nh = (None, None) if noise is None else (noise[0].float().contiguous(), noise[1].float().contiguous())
        ops.ddpm_step(batch, x_lig, h_lig, x_kp, eps_x, eps_h, coef, step, nx, nh, seed)
        g.nodes['lig'].data['x_0'], g.nodes['lig'].data['h_0'], g.nodes['kp'].data['x_0'] = x_lig, h_lig, x_kp
        return g

    # ------------------------------------------------------------------ the loop (reference :342-469)
    MAX_CACHED_SAMPLERS = 24

    def _cache_get(self, key):
        """Captured samplers are cached on the CONTENT of what they were captured for (complex sizes, kk edge list,
        parameter versions, mode) -- never on object ids, which CPython and the caching allocator recycle -- and evicted
        least-recently-used, one at a time (a wipe would destroy captured graphs mid-workload)."""
        hit = self._samplers.pop(key, None)
        if hit is not None:
            self._samplers[key] = hit           # re-insert: most recently used last
            return hit
        while len(self._samplers) >= self.MAX_CACHED_SAMPLERS:
            self._samplers.pop(next(iter(self._samplers)))
        return None

    def _sampler(self, g, steps_per_graph, use_cuda_graph) -> ops.Sampler:
        batch, kk = self._layout(g)
        model = self.dynamics.device_model(g.device)
        key = ("one", self.dynamics.layout_key(), self.dynamics._st.model_key, steps_per_graph, use_cuda_graph,
               getattr(model, "precision", "fp32"))
        if self._cache_get(key) is None:
            self._samplers[key] = ops.Sampler(model, batch, self.dynamics.graph_params(), kk, self.coef_table(g.device),
                                              self.n_timesteps, self.n_lig_features, steps_per_graph=steps_per_graph,
                                              use_cuda_graph=use_cuda_graph,
                                              lig_feat_norm_constant=float(self.lig_feat_norm_constant))
        return self._samplers[key]

    def _sub_samplers(self, g, n_sub, steps_per_graph, use_cuda_graph):
        """The batch cut into n_sub contiguous groups of complexes, each with its own captured loop (ops.Sampler) and its
        own stream.  Complexes are independent (no cross-complex term anywhere in the loop), so the groups' kernels may
        run concurrently: a fused edge kernel of one group is only a few waves of long-running CTAs, and the CTAs of the
        other groups fill the SMs its tail leaves idle.  Noise is keyed by the GLOBAL atom index, so the split does not
        change what is drawn."""
        batch, kk = self._layout(g)
        model = self.dynamics.device_model(g.device)
        key = ("sub", self.dynamics.layout_key(), self.dynamics._st.model_key, n_sub, steps_per_graph, use_cuda_graph,
               getattr(model, "precision", "fp32"))
        if self._cache_get(key) is None:
            B = batch.B
            ks, kd = g.edges(form="uv", etype="kk")
            ks, kd = ks.cpu().long(), kd.cpu().long()
            kp_ptr = batch.kp_ptr.cpu().long()
            lig_ptr = batch.lig_ptr.cpu().long()
            bounds = split_bounds(B, n_sub)
            subs = []
            for a, b in zip(bounds[:-1], bounds[1:]):
                sb = ops.DeviceBatch(batch.lig_n[a:b], batch.kp_n[a:b], g.device)
                k0, k1, l0, l1 = int(kp_ptr[a]), int(kp_ptr[b]), int(lig_ptr[a]), int(lig_ptr[b])
                m = (kd >= k0) & (kd < k1)
                skk = ops.Csr.from_edges(ks[m] - k0, kd[m] - k0, sb.n_kp, g.device)
                smp = ops.Sampler(model, sb, self.dynamics.graph_params(), skk, self.coef_table(g.device), self.n_timesteps,
                                  self.n_lig_features, steps_per_graph=steps_per_graph, use_cuda_graph=use_cuda_graph,
                                  lig_feat_norm_constant=float(self.lig_feat_norm_constant), atom_offset=l0)
                subs.append((smp, (a, b), (k0, k1), (l0, l1), torch.cuda.Stream(device=g.device)))
            self._samplers[key] = subs
        return self._samplers[key]

    def default_sub_batches(self, n_complexes: int) -> int:
        """How many concurrently sampled groups a batch is cut into when the caller does not say (measured on B200,
        DESIGN.md section 4.4); KPD_SUB_BATCHES overrides."""
        env = os.environ.get("KPD_SUB_BATCHES")
        if env:
            return max(1, min(int(env), n_complexes))
        return max(1, min(DEFAULT_SUB_BATCHES[self.architecture], n_complexes // 16))

    def _capacity_sampler(self, instance: int, plan: "ops.CapacityPlan", device, steps_per_graph, use_cuda_graph,
                          resamplings: int = 0, record: bool = False, multistep: bool = False):
        """The captured loop of capacity bucket plan.key (created on first use, then shared by every batch that lands in
        the bucket -- whatever its per-complex sizes, pockets or kk graph).  Groups of one call that run concurrently
        and share a bucket take distinct instances 0, 1, ... of it.  resamplings >= 1: the inpainting loop with that
        many passes per step; record=True: the recording loop (visualize=True); multistep=True: the DPM-Solver++(2M)
        loop (solver="dpmpp_2m").  All are cached apart from the plain loop: their captured sequences differ."""
        model = self.dynamics.device_model(device)
        key = ("cap", instance, plan.key, self.dynamics._st.model_key, steps_per_graph, use_cuda_graph,
               getattr(model, "precision", "fp32"), self.n_timesteps)
        if resamplings:
            key = key + ("inpaint", int(resamplings))
        if record:
            key = key + ("record",)
        if multistep:
            key = key + ("multistep",)
        hit = self._cache_get(key)
        if hit is None:
            kp_width = self.n_kp_feat
            v_width = self.dynamics.vector_size if self.architecture == "gvp" else 0
            hit = ops.CapacitySampler(model, plan, self.dynamics.graph_params(), self.coef_table(device), self.n_timesteps,
                                      self.n_lig_features, kp_width, v_width, steps_per_graph=steps_per_graph,
                                      use_cuda_graph=use_cuda_graph,
                                      lig_feat_norm_constant=float(self.lig_feat_norm_constant), resamplings=resamplings,
                                      inpaint_coef=self.inpaint_coef_table(device) if resamplings else None,
                                      record=record, multistep=multistep)
            self._samplers[key] = hit
            object.__setattr__(self, "cold_captures", self.cold_captures + 1)
        return hit

    @torch.no_grad()
    def sample_from_encoded_receptors(self, g, visualize=False, init_lig_pos: torch.Tensor = None, noise=None,
                                      seed: Optional[int] = None, steps_per_graph: int = 50, use_cuda_graph: bool = True,
                                      return_device_tensors: bool = False, sub_batches: Optional[int] = None,
                                      decode: bool = False, capacity: bool = True, fixed_mask: torch.Tensor = None,
                                      fixed_pos: torch.Tensor = None, fixed_feat: torch.Tensor = None,
                                      resamplings: int = 1, start_pos: torch.Tensor = None,
                                      start_feat: torch.Tensor = None, start_step: Optional[int] = None,
                                      timesteps: Optional[int] = None, eta: Optional[float] = None,
                                      frame_every: Optional[int] = None, solver: Optional[str] = None):
        """Returns (lig_pos, lig_feat): one CPU tensor per complex, as the reference does (:342-469).  ``g`` may live
        on the CPU (pinned or not): its keypoint tensors are uploaded here, straight into the sampler's buffers -- the
        host->device boundary of the path (reference test.py:152-161).

        The batch is sampled by capacity-bucketed captured loops (ops.plan_capacity / ops.CapacitySampler): a new
        tuple of ligand sizes, another pocket or another kk graph re-uses the CUDA graphs captured for its bucket
        instead of re-capturing, so the reference's real entry points -- random sizes per call, :490-495 -- stay warm.
        ``capacity=False`` selects samplers captured for the exact layout (kept for A/B tests).  ``decode=True`` also
        returns the atom types (argmax over the feature channels, computed on the device: test.py:199-203).

        Fragment-conditioned sampling (inpainting; an extension beyond the reference, DESIGN.md section 6.1): with
        ``fixed_mask`` (bool [n_lig], g's ligand order) the atoms it marks are pinned to ``fixed_pos`` ([n_lig,3], in the
        frame the ligands are returned in) and ``fixed_feat`` ([n_lig,F], returned feature space); rows of unmarked atoms
        are ignored.  Every reverse step runs ``resamplings`` denoiser passes (RePaint resampling, jump length 1), so a
        call costs about ``resamplings`` plain calls.  Complexes without a marked atom are sampled exactly as without
        a mask at resamplings=1.  Only the capacity path supports it: ``capacity=False`` raises ValueError.

        Ligand optimisation by partial noising (SDEdit-style; an extension beyond the reference, DESIGN.md section 6.2):
        with ``start_pos`` ([n_lig,3], g's ligand order, in the frame the ligands are returned in), ``start_feat``
        ([n_lig,F], returned feature space) and ``start_step`` = t0 in [0, T], every ligand starts from its start ligand
        noised to level t0, and the loop runs the t0 reverse steps t0-1 .. 0 (about t0/T of a plain call): a small t0
        gives close variants, a large one ligands that only loosely follow the start.  The frame is the start ligands'
        own: ``init_lig_pos`` is not used and must not be given.  Composes with a fragment (which then stays pinned) and
        with sub-batches; capacity path only.

        Fewer-step sampling (DESIGN.md section 6.3): ``timesteps`` = n in [1, t_start] (t_start = T, or t0 of a start
        ligand) runs n reverse steps on the grid tau_k = (k t_start) // n instead of every step, for about n / t_start
        of the cost; ``eta`` in [0, 1] makes them DDIM(eta) steps instead of ancestral ones (eta = 0: deterministic
        steps, though a fragment's known part is still noised at every step).  timesteps = t_start with eta=None is the
        default run bit for bit; eta alone keeps every step.  Composes with fragments, start ligands and sub-batches,
        captures nothing new; capacity path only, and not with start_step = 0.

        Trajectories (DESIGN.md section 6.4): ``visualize=True`` records the run inside the captured loop, every
        ``frame_every``-th executed step (None: every step, as the reference records), and returns one more element,
        last: one dict per complex with m = ceil(n / frame_every) for the n steps run,
        ``'t'`` long [m+1] (diffusion level of each frame; 0 for the last), ``'positions'`` [m+1, n_atoms, 3] and
        ``'features'`` [m+1, n_atoms, F] (frame j < m: the state before executed step j*frame_every; frame m: the
        returned ligand), ``'pred_positions'`` [m, n_atoms, 3] and ``'pred_features'`` [m, n_atoms, F] (the denoiser's
        clean-ligand estimate (z - sigma_t eps) / alpha_t at frame j).  Every frame is in the frame and feature space the
        ligands are returned in.  Recording does not change the ligands; capacity path only.

        Second-order multistep sampling (DESIGN.md section 6.5): ``solver="dpmpp_2m"`` runs DPM-Solver++(2M) steps on the
        grid of ``timesteps`` (all t_start rows without it): each step is the DDIM eta = 0 step plus a correction from
        the previous step's clean-ligand estimate, more accurate than DDIM at the same step count (10-25 steps is where
        it pays; pass steps_per_graph <= timesteps so that those steps replay a captured graph).  Composes with start
        ligands, sub-batches and visualize=True (the prediction frames are the estimates the solver uses).  ValueError
        with eta, a fragment, capacity=False or start_step = 0.  solver=None (default) is the run without it."""
        n_lig_total = int(g.num_nodes('lig'))
        inpaint = self._check_fragment_args(n_lig_total, fixed_mask, fixed_pos, fixed_feat, resamplings)
        start = self._check_start_args(n_lig_total, start_pos, start_feat, start_step)
        if inpaint and not capacity:
            raise ValueError("fragment-conditioned sampling runs on the capacity path only (capacity=True)")
        if start and not capacity:
            raise ValueError("sampling from a start ligand runs on the capacity path only (capacity=True)")
        if start and init_lig_pos is not None:
            raise ValueError("init_lig_pos is not used with a start ligand (the start ligands' means set the frame)")
        t_start = int(start_step) if start else self.n_timesteps
        n_sched = self._check_schedule_args(timesteps, eta, t_start, capacity, solver, inpaint)
        every = self._check_visualize_args(visualize, frame_every, capacity)
        dev = torch.device("cuda", torch.cuda.current_device()) if g.device.type != "cuda" else g.device
        batch_size = g.batch_size
        if start:
            init_pos = torch.zeros(batch_size, 3)                   # not read by a run from a start ligand
            a_t0, s_t0 = start_coefficients(self.gamma.gamma, int(start_step))
        elif init_lig_pos is not None:
            assert init_lig_pos.shape == (batch_size, 3)
            init_pos = init_lig_pos
        else:
            if g.num_nodes('rec') == 0:
                raise ValueError("init_lig_pos is required when the graph has no 'rec' nodes (fixed encoder; "
                                 "the reference would take a mean over zero nodes here, SURVEY N7)")
            init_pos = hetero.readout_nodes(g, feat='x_0', op='mean', ntype='rec')
        if seed is None:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())      # follows torch.manual_seed like the reference
        sched = None if n_sched is None else self.schedule_tables(dev, t_start, n_sched, eta, inpaint, solver)
        pred = None
        if visualize:
            pred = self.prediction_coef_table(dev) if sched is None else sched[2]
            n_run = t_start if n_sched is None else n_sched
            levels = frame_levels(list(range(self.n_timesteps + 1)) if n_sched is None else step_grid(t_start, n_sched),
                                  n_run, every)
        n_sub = self.default_sub_batches(batch_size) if sub_batches is None else max(1, min(int(sub_batches), batch_size))
        if noise is not None:
            n_sub = 1          # injected noise (parity runs) is laid out for the undivided batch
        if not capacity:
            return self._sample_exact_layout(g, dev, init_pos, noise, seed, steps_per_graph, use_cuda_graph,
                                             return_device_tensors, n_sub)
        kp = g.nodes['kp'].data
        lig_n = g.batch_num_nodes('lig').tolist()
        kp_n = g.batch_num_nodes('kp').tolist()
        ks, kd = g.edges(form="uv", etype="kk")
        kk_n = g.batch_num_edges('kk').tolist()
        grouped = sum(kk_n) == int(ks.numel())          # kk edges grouped by complex (dgl.batch / hetero.batch order)
        lig_ptr = [0]
        kp_ptr = [0]
        kk_ptr = [0]
        for b in range(batch_size):
            lig_ptr.append(lig_ptr[-1] + lig_n[b]); kp_ptr.append(kp_ptr[-1] + kp_n[b]); kk_ptr.append(kk_ptr[-1] + kk_n[b])
        bounds = split_bounds(batch_size, n_sub)
        gp = self.dynamics.graph_params()
        cur = torch.cuda.current_stream(dev)
        ready = torch.cuda.Event()
        ready.record(cur)
        parts, used, launches, taken = [], [], 0, {}
        kv = kp.get('v_0')
        for slot, (a, b) in enumerate(zip(bounds[:-1], bounds[1:])):
            k0, k1, l0 = kp_ptr[a], kp_ptr[b], lig_ptr[a]
            if grouped:
                gs, gd = ks[kk_ptr[a]:kk_ptr[b]] - k0, kd[kk_ptr[a]:kk_ptr[b]] - k0
            else:
                m = (kd >= k0) & (kd < k1)
                gs, gd = ks[m] - k0, kd[m] - k0
            plan = ops.plan_capacity(lig_n[a:b], kp_n[a:b], int(gs.numel()), gp)
            inst = taken.get(plan.key, 0)
            taken[plan.key] = inst + 1
            smp = self._capacity_sampler(inst, plan, dev, steps_per_graph, use_cuda_graph,
                                         resamplings=int(resamplings) if inpaint else 0, record=visualize,
                                         multistep=solver is not None)
            frag = None
            if inpaint:
                l1 = lig_ptr[b]
                frag = (fixed_mask[l0:l1], fixed_pos[l0:l1], fixed_feat[l0:l1])
            st_rows = None
            if start:
                l1 = lig_ptr[b]
                st_rows = (start_pos[l0:l1], start_feat[l0:l1], t_start if n_sched is None else n_sched, a_t0, s_t0)
            if n_sub > 1 and (slot, str(dev)) not in self._streams:
                self._streams[(slot, str(dev))] = torch.cuda.Stream(device=dev)
            st = self._streams[(slot, str(dev))] if n_sub > 1 else cur
            if n_sub > 1:
                st.wait_event(ready)
            with torch.cuda.stream(st):
                out = smp.run(plan, kp['x_0'][k0:k1], kp['h_0'][k0:k1], kv[k0:k1] if kv is not None else None, gs, gd,
                              init_pos[a:b], seed=seed, atom_offset=l0, noise=noise, decode=decode, fragment=frag,
                              start=st_rows, schedule=None if sched is None else sched[:2],
                              record_every=every if visualize else None, pred_coef=pred,
                              multistep=None if solver is None else sched[3])
            if n_sub > 1:
                for t in out:
                    for v in (t.values() if isinstance(t, dict) else (t,)):
                        v.record_stream(cur)
                used.append(st)
            parts.append(out)
            launches += smp.sampler.launches_per_step
        for st in used:
            cur.wait_stream(st)
        cat = (lambda i: parts[0][i]) if len(parts) == 1 else (lambda i: torch.cat([p[i] for p in parts]))
        x_lig, h_lig, x_kp = cat(0), cat(1), cat(2)
        atom_type = cat(3) if decode else None
        object.__setattr__(self, "last_launches_per_step", launches)
        if g.device.type == "cuda":
            g.nodes['lig'].data['x_0'], g.nodes['lig'].data['h_0'], g.nodes['kp'].data['x_0'] = x_lig, h_lig, x_kp
        frames = []
        if visualize:       # sub-batches hold consecutive complexes: their frames join along the atom axis
            fr = {k: torch.cat([p[-1][k] for p in parts], dim=1) for k in parts[0][-1]}
            fr = {k: v if return_device_tensors else v.cpu() for k, v in fr.items()}
            t = levels.to(dev) if return_device_tensors else levels
            split = {k: torch.split(v, lig_n, dim=1) for k, v in fr.items()}
            frames = [dict(t=t, **{k: split[k][i] for k in split}) for i in range(batch_size)]
        if return_device_tensors:
            res = (x_lig, h_lig, atom_type) if decode else (x_lig, h_lig)
            return res + (frames,) if visualize else res
        pos_cpu, feat_cpu = x_lig.cpu(), h_lig.cpu()                # device -> host boundary (reference :464)
        res = (list(torch.split(pos_cpu, lig_n)), list(torch.split(feat_cpu, lig_n)))
        if decode:
            res = res + (list(torch.split(atom_type.cpu(), lig_n)),)
        return res + (frames,) if visualize else res

    def _check_schedule_args(self, timesteps, eta, t_start: int, capacity, solver=None, fragment=False) -> Optional[int]:
        """ValueError for a bad fewer-step or solver request (host-side checks, before any device work); the step count
        of the schedule to run, or None for the default tables."""
        if timesteps is not None:
            if isinstance(timesteps, bool) or not isinstance(timesteps, numbers.Integral):
                raise ValueError(f"timesteps must be an int, got {timesteps!r}")
            if t_start == 0:
                raise ValueError("timesteps must be None with start_step = 0 (no reverse step runs)")
            if not 1 <= int(timesteps) <= t_start:
                raise ValueError(f"timesteps must be in [1, {t_start}], got {timesteps}")
        if eta is not None and (isinstance(eta, bool) or not isinstance(eta, numbers.Real) or not math.isfinite(eta)
                                or not 0 <= eta <= 1):
            raise ValueError(f"eta must be a finite number in [0, 1], got {eta!r}")
        if (timesteps is not None or eta is not None) and not capacity:
            raise ValueError("fewer-step sampling runs on the capacity path only (capacity=True)")
        if solver is not None:
            if not isinstance(solver, str) or solver not in SOLVERS:
                raise ValueError(f"solver must be None or one of {SOLVERS}, got {solver!r}")
            if eta is not None:
                raise ValueError(f"solver={solver!r} takes no eta (its steps are built on the eta = 0 rows)")
            if fragment:
                raise ValueError(f"solver={solver!r} does not combine with a fragment (re-noising breaks its history)")
            if not capacity:
                raise ValueError(f"solver={solver!r} runs on the capacity path only (capacity=True)")
            if t_start == 0:
                raise ValueError(f"solver={solver!r} needs start_step > 0 (no reverse step runs at start_step = 0)")
        if (timesteps is None and eta is None and solver is None) or t_start == 0:
            return None
        return t_start if timesteps is None else int(timesteps)

    @staticmethod
    def _check_visualize_args(visualize, frame_every, capacity) -> int:
        """ValueError for a bad trajectory request (host-side checks, before any device work); the frame stride."""
        if frame_every is not None:
            if not visualize:
                raise ValueError("frame_every needs visualize=True")
            if isinstance(frame_every, bool) or not isinstance(frame_every, numbers.Integral) or frame_every < 1:
                raise ValueError(f"frame_every must be an integer >= 1, got {frame_every!r}")
        if visualize and not capacity:
            raise ValueError("visualize=True runs on the capacity path only (capacity=True)")
        return 1 if frame_every is None else int(frame_every)

    def _check_fragment_args(self, n_lig: int, fixed_mask, fixed_pos, fixed_feat, resamplings) -> bool:
        """ValueError for an inconsistent fragment request (host-side checks, before any device work); True when the
        call is fragment-conditioned."""
        if int(resamplings) < 1:
            raise ValueError(f"resamplings must be >= 1, got {resamplings}")
        if fixed_mask is None:
            if fixed_pos is not None or fixed_feat is not None:
                raise ValueError("fixed_pos / fixed_feat need fixed_mask")
            if int(resamplings) > 1:
                raise ValueError("resamplings > 1 needs fixed atoms (fixed_mask)")
            return False
        if fixed_pos is None or fixed_feat is None:
            raise ValueError("fixed_mask needs fixed_pos and fixed_feat")
        F = self.n_lig_features
        if tuple(fixed_mask.shape) != (n_lig,):
            raise ValueError(f"fixed_mask must have shape [{n_lig}], got {tuple(fixed_mask.shape)}")
        if fixed_pos.dim() != 2 or fixed_pos.shape[1] != 3 or fixed_pos.shape[0] != n_lig:
            raise ValueError(f"fixed_pos must have shape [{n_lig}, 3], got {tuple(fixed_pos.shape)}")
        if fixed_feat.dim() != 2 or fixed_feat.shape[1] != F or fixed_feat.shape[0] != n_lig:
            raise ValueError(f"fixed_feat must have shape [{n_lig}, {F}], got {tuple(fixed_feat.shape)}")
        if int(resamplings) > 1 and not bool(fixed_mask.any()):
            raise ValueError("resamplings > 1 needs at least one fixed atom")
        return True

    def _check_start_step(self, start_step):
        if start_step is None:
            return
        if isinstance(start_step, bool) or int(start_step) != start_step or not 0 <= int(start_step) <= self.n_timesteps:
            raise ValueError(f"start_step must be an integer in [0, {self.n_timesteps}], got {start_step}")

    def _check_start_args(self, n_lig: int, start_pos, start_feat, start_step) -> bool:
        """ValueError for an inconsistent start-ligand request (host-side checks, before any device work); True when the
        call runs from a start ligand."""
        self._check_start_step(start_step)
        given = start_pos is not None or start_feat is not None
        if not given:
            if start_step is not None:
                raise ValueError("start_step needs a start ligand (start_pos and start_feat)")
            return False
        if start_pos is None or start_feat is None:
            raise ValueError("a start ligand needs both start_pos and start_feat")
        if start_step is None:
            raise ValueError("a start ligand needs start_step")
        F = self.n_lig_features
        if start_pos.dim() != 2 or tuple(start_pos.shape) != (n_lig, 3):
            raise ValueError(f"start_pos must have shape [{n_lig}, 3], got {tuple(start_pos.shape)}")
        if start_feat.dim() != 2 or tuple(start_feat.shape) != (n_lig, F):
            raise ValueError(f"start_feat must have shape [{n_lig}, {F}], got {tuple(start_feat.shape)}")
        return True

    def _check_start_ligands(self, start_ligands, start_step, n_lig_atoms, init_lig_pos, use_ref_lig_com,
                             sampler_kw) -> bool:
        """Host-side validation of _sample's per-receptor start ligands; True when the call runs from them."""
        self._check_start_step(start_step)
        if start_ligands is None:
            if start_step is not None:
                raise ValueError("start_step needs start ligands")
            return False
        if start_step is None:
            raise ValueError("start ligands need start_step")
        if init_lig_pos is not None or use_ref_lig_com:
            raise ValueError("init_lig_pos / use_ref_lig_com are not used with start ligands (their means set the frame)")
        if not sampler_kw.get("capacity", True):
            raise ValueError("sampling from a start ligand runs on the capacity path only (capacity=True)")
        if len(start_ligands) != len(n_lig_atoms):
            raise ValueError(f"start_ligands: one entry per receptor, got {len(start_ligands)} for "
                             f"{len(n_lig_atoms)} receptors")
        F = self.n_lig_features
        for r, lig in enumerate(start_ligands):
            if lig is None:
                raise ValueError(f"receptor {r} has no start ligand")
            pos, feat = lig
            if pos.dim() != 2 or pos.shape[1] != 3:
                raise ValueError(f"start ligand of receptor {r}: positions must be [m, 3], got {tuple(pos.shape)}")
            if feat.dim() != 2 or feat.shape[1] != F or feat.shape[0] != pos.shape[0]:
                raise ValueError(f"start ligand of receptor {r}: features must be [{pos.shape[0]}, {F}], got "
                                 f"{tuple(feat.shape)}")
            m = int(pos.shape[0])
            other = [int(n) for n in n_lig_atoms[r] if int(n) != m]
            if other:
                raise ValueError(f"receptor {r}: requested ligand size {other[0]} differs from its {m}-atom start ligand")
        return True

    def _check_fragments(self, fragments, n_lig_atoms, resamplings) -> bool:
        """Host-side validation of _sample's per-receptor fragments; True when at least one atom is fixed."""
        if int(resamplings) < 1:
            raise ValueError(f"resamplings must be >= 1, got {resamplings}")
        any_fixed = False
        if fragments is not None:
            if len(fragments) != len(n_lig_atoms):
                raise ValueError(f"fragments: one entry (or None) per receptor, got {len(fragments)} for "
                                 f"{len(n_lig_atoms)} receptors")
            F = self.n_lig_features
            for r, frag in enumerate(fragments):
                if frag is None:
                    continue
                pos, feat = frag
                if pos.dim() != 2 or pos.shape[1] != 3:
                    raise ValueError(f"fragment of receptor {r}: positions must be [m, 3], got {tuple(pos.shape)}")
                if feat.dim() != 2 or feat.shape[1] != F or feat.shape[0] != pos.shape[0]:
                    raise ValueError(f"fragment of receptor {r}: features must be [{pos.shape[0]}, {F}], got "
                                     f"{tuple(feat.shape)}")
                m = int(pos.shape[0])
                small = [int(n) for n in n_lig_atoms[r] if int(n) < m]
                if small:
                    raise ValueError(f"receptor {r}: requested ligand size {small[0]} is below its {m}-atom fragment")
                any_fixed = any_fixed or (m > 0 and len(n_lig_atoms[r]) > 0)
        if int(resamplings) > 1 and not any_fixed:
            raise ValueError("resamplings > 1 needs at least one fragment atom")
        return any_fixed

    def _sample_exact_layout(self, g, dev, init_pos, noise, seed, steps_per_graph, use_cuda_graph, return_device_tensors,
                             n_sub):
        """Samplers captured for the exact per-complex layout of g (one per distinct tuple of sizes)."""
        if g.device.type != "cuda":
            g = g.to(dev)
        init_pos = init_pos.to(dev, torch.float32, non_blocking=True)
        kp = g.nodes['kp'].data
        if n_sub == 1:
            sampler = self._sampler(g, steps_per_graph, use_cuda_graph)
            x_lig, h_lig, x_kp = sampler.run(kp['x_0'], kp['h_0'], kp.get('v_0'), init_pos, noise=noise, seed=seed)
            object.__setattr__(self, "last_launches_per_step", sampler.launches_per_step)
        else:
            subs = self._sub_samplers(g, n_sub, steps_per_graph, use_cuda_graph)
            cur = torch.cuda.current_stream(dev)
            kx, kh, kv = kp['x_0'].float().contiguous(), kp['h_0'].float().contiguous(), kp.get('v_0')
            kv = kv.float().contiguous() if kv is not None else None
            init_pos = init_pos.float().contiguous()
            ready = torch.cuda.Event()
            ready.record(cur)
            parts = []
            for smp, (a, b), (k0, k1), _, st in subs:
                st.wait_event(ready)
                with torch.cuda.stream(st):
                    out = smp.run(kx[k0:k1], kh[k0:k1], kv[k0:k1] if kv is not None else None, init_pos[a:b], seed=seed)
                for t in out:
                    t.record_stream(cur)
                parts.append(out)
            for *_, st in subs:
                cur.wait_stream(st)
            x_lig = torch.cat([p[0] for p in parts])
            h_lig = torch.cat([p[1] for p in parts])
            x_kp = torch.cat([p[2] for p in parts])
            object.__setattr__(self, "last_launches_per_step", sum(smp.launches_per_step for smp, *_ in subs))
        g.nodes['lig'].data['x_0'], g.nodes['lig'].data['h_0'], g.nodes['kp'].data['x_0'] = x_lig, h_lig, x_kp
        if return_device_tensors:
            return x_lig, h_lig
        sizes = g.batch_num_nodes('lig').tolist()
        pos_cpu, feat_cpu = x_lig.cpu(), h_lig.cpu()
        return list(torch.split(pos_cpu, sizes)), list(torch.split(feat_cpu, sizes))

    # ------------------------------------------------------------------ batch drivers (reference :270-340, :472-495)
    @torch.no_grad()
    def _encode_all(self, ref_graphs: List, rec_enc_batch_size: int, encoded: bool):
        """All receptors encoded and batched into ONE graph on the model's device, plus the per-receptor mean of the
        'rec' positions (what sample_from_encoded_receptors falls back to for init_lig_pos, reference :359-360)."""
        dev = self.gamma.gamma.device
        if encoded:
            enc = hetero.batch(ref_graphs)
            enc = enc if enc.device == dev else enc.to(dev)
        else:
            # rec_enc_batch_size receptors per encoder pass (reference :277-287), on the device the weights live on
            chunks = []
            for b in range(ceil(len(ref_graphs) / rec_enc_batch_size)):
                chunk = hetero.batch(ref_graphs[b * rec_enc_batch_size:(b + 1) * rec_enc_batch_size])
                chunks.append(self.encode_receptors(chunk if chunk.device == dev else chunk.to(dev)))
            enc = chunks[0] if len(chunks) == 1 else hetero.batch(chunks)
        rec_mean = hetero.readout_nodes(enc, feat='x_0', op='mean', ntype='rec') if enc.num_nodes('rec') > 0 else None
        return enc, rec_mean

    @torch.no_grad()
    def _sample(self, ref_graphs: List, n_lig_atoms: List[List[int]], rec_enc_batch_size: int = 32,
                diff_batch_size: int = 32, visualize=False, use_ref_lig_com: bool = False, encoded: bool = False,
                init_lig_pos: Optional[List[torch.Tensor]] = None, noise: Optional[List[torch.Tensor]] = None,
                complexes: Optional[List[int]] = None, fragments: Optional[List] = None, resamplings: int = 1,
                start_ligands: Optional[List] = None, start_step: Optional[int] = None, **sampler_kw):
        """ref_graphs: one single-complex graph per receptor (reference :270-340).  ``encoded=True`` skips the receptor
        encoder (graphs already hold kp nodes + kk edges).  init_lig_pos: optional [3] tensor per receptor.
        noise: optional injected Gaussian draws, one [n+1, n_lig*(3+F)] tensor per diffusion batch (parity runs), n the
        reverse steps a call runs: T, t0 of start ligands, or ``timesteps``.
        complexes: optional subset (indices into the flattened receptor-major list of requested ligands) to sample --
        what sample_sharded deals to this rank; the returned lists then hold only those.
        fragments: optional, one ``(pos [m,3], feat [m,F])`` or None per receptor: every ligand requested for that
        receptor starts with those m atoms, pinned (fragment growing; positions in the receptor's frame, features in the
        returned feature space), with ``resamplings`` denoiser passes per reverse step (see
        sample_from_encoded_receptors).  A diffusion batch without any fragment atom is sampled by the plain loop.
        start_ligands / start_step: optional, one ``(pos [m,3], feat [m,F])`` per receptor and t0 in [0, T]: every
        ligand requested for that receptor (each of size m) is a variant of its start ligand, noised to level t0 and
        denoised from there (ligand optimisation, see sample_from_encoded_receptors); with fragments too, the fragment
        is the start ligand's first atoms and stays pinned.
        timesteps / eta / solver (passed on to sample_from_encoded_receptors, like every other keyword): fewer-step and
        multistep sampling, checked here before any receptor is encoded.
        visualize / frame_every: trajectories (see sample_from_encoded_receptors); every receptor's dict then also
        holds ``'frames'``, one trajectory dict per ligand.  Not with ``complexes`` (sample_sharded).

        The diffusion batches are assembled on the device (hetero.expand_complexes): no per-complex graph copies."""
        has_fragment = self._check_fragments(fragments, n_lig_atoms, resamplings)
        has_start = self._check_start_ligands(start_ligands, start_step, n_lig_atoms, init_lig_pos, use_ref_lig_com,
                                              sampler_kw)
        self._check_schedule_args(sampler_kw.get("timesteps"), sampler_kw.get("eta"),
                                  int(start_step) if has_start else self.n_timesteps, sampler_kw.get("capacity", True),
                                  sampler_kw.get("solver"), has_fragment)
        self._check_visualize_args(visualize, sampler_kw.get("frame_every"), sampler_kw.get("capacity", True))
        if visualize and complexes is not None:
            raise ValueError("visualize=True is not supported by sample_sharded")
        n_receptors = len(ref_graphs)
        enc, rec_mean = self._encode_all(ref_graphs, rec_enc_batch_size, encoded)
        dev = enc.device
        pocket_of = [r for r in range(n_receptors) for _ in n_lig_atoms[r]]
        sizes = [int(n) for r in range(n_receptors) for n in n_lig_atoms[r]]
        todo = list(range(len(sizes))) if complexes is None else list(complexes)
        if init_lig_pos is not None:
            centers = torch.stack([c.reshape(3) for c in init_lig_pos]).to(dev, torch.float32)
        elif use_ref_lig_com:
            # copy_graph zero-fills the ligand before the mean is taken, so this is the origin (SURVEY N10)
            centers = torch.zeros(n_receptors, 3, device=dev)
        else:
            centers = rec_mean
        pocket_t = torch.tensor(pocket_of, dtype=torch.long, device=dev)
        size_t = torch.tensor(sizes, dtype=torch.long, device=dev)
        lig_pos, lig_feat, frames = [], [], []
        for b in range(ceil(len(todo) / diff_batch_size)):
            chunk = todo[b * diff_batch_size:(b + 1) * diff_batch_size]
            idx = torch.tensor(chunk, dtype=torch.long, device=dev)
            bg = hetero.expand_complexes(enc, pocket_t[idx], size_t[idx], self.n_lig_features)
            if centers is None and not has_start:
                raise ValueError("init_lig_pos is required when the graphs have no 'rec' nodes (SURVEY N7)")
            frag_kw = (self._fragment_rows(fragments, [pocket_of[i] for i in chunk], [sizes[i] for i in chunk], resamplings)
                       if has_fragment else {})
            if has_start:
                owners = [pocket_of[i] for i in chunk]
                frag_kw.update(init_lig_pos=None, start_step=int(start_step),
                               start_pos=torch.cat([start_ligands[r][0].detach().float().cpu() for r in owners]),
                               start_feat=torch.cat([start_ligands[r][1].detach().float().cpu() for r in owners]))
            else:
                frag_kw.update(init_lig_pos=centers[pocket_t[idx]])
            res = self.sample_from_encoded_receptors(bg, visualize=visualize,
                                                     noise=None if noise is None else noise[b], **frag_kw, **sampler_kw)
            if visualize:
                *res, fr = res
                frames.extend(fr)
            p, f = res
            lig_pos.extend(p)
            lig_feat.extend(f)
        if complexes is not None:
            return lig_pos, lig_feat
        samples, end = [], 0
        for rec_idx in range(n_receptors):
            start, end = end, end + len(n_lig_atoms[rec_idx])
            samples.append({'positions': lig_pos[start:end], 'features': lig_feat[start:end]})
            if visualize:
                samples[-1]['frames'] = frames[start:end]
        return samples

    def _fragment_rows(self, fragments, receptors: List[int], sizes: List[int], resamplings: int) -> Dict:
        """fixed_mask / fixed_pos / fixed_feat (host tensors, batch ligand order) of one diffusion batch whose complexes
        belong to `receptors`; {} (the plain loop) when none of them has a fragment atom."""
        F = self.n_lig_features
        n = sum(sizes)
        mask = torch.zeros(n, dtype=torch.bool)
        pos = torch.zeros(n, 3)
        feat = torch.zeros(n, F)
        off = 0
        for r, size in zip(receptors, sizes):
            frag = fragments[r]
            if frag is not None and frag[0].shape[0] > 0:
                m = int(frag[0].shape[0])
                mask[off:off + m] = True
                pos[off:off + m] = frag[0].detach().float().cpu()
                feat[off:off + m] = frag[1].detach().float().cpu()
            off += size
        if not bool(mask.any()):
            return {}
        return dict(fixed_mask=mask, fixed_pos=pos, fixed_feat=feat, resamplings=resamplings)

    @torch.no_grad()
    def sample_sharded(self, ref_graphs: List, n_lig_atoms: List[List[int]], rec_enc_batch_size: int = 32,
                       diff_batch_size: int = 128, group=None, **kw):
        """_sample over every rank of the process group (one process per GPU): the requested (receptor, ligand size)
        pairs are dealt to the ranks by estimated cost (dist.shard_complexes), each rank samples its share with its own
        captured loops and no per-step communication, and ONE final all_gather (NCCL over NVLink; gloo in the CPU
        tests) brings coordinates + atom features back, so every rank returns the complete, receptor-major result of
        ``_sample``.  The reference's equivalent is a slurm array of independent single-GPU processes
        (gen_test_commands.py:36-40, test.py:143-184).  Noise follows this rank's torch generator / ``seed``.
        visualize=True is not supported (ValueError): trajectories are not gathered across ranks."""
        if kw.get("visualize"):
            raise ValueError("visualize=True is not supported by sample_sharded")
        import torch.distributed as dist
        from . import dist as kdist
        world = dist.get_world_size(group) if dist.is_initialized() else 1
        rank = dist.get_rank(group) if dist.is_initialized() else 0
        sizes = [int(n) for r in range(len(ref_graphs)) for n in n_lig_atoms[r]]
        kp_n = [int(g.num_nodes('kp')) or int(g.num_nodes('rec')) for g in ref_graphs]
        kp_of = [kp_n[r] for r in range(len(ref_graphs)) for _ in n_lig_atoms[r]]
        shards = kdist.shard_complexes(sizes, kp_of, world)
        mine = shards[rank]
        pos, feat = self._sample(ref_graphs, n_lig_atoms, rec_enc_batch_size, diff_batch_size, complexes=mine, **kw)
        dev = self.gamma.gamma.device
        F = self.n_lig_features
        x = torch.cat(pos).to(dev) if pos else torch.zeros(0, 3, device=dev)
        h = torch.cat(feat).to(dev) if feat else torch.zeros(0, F, device=dev)
        xs, hs, all_sizes = kdist.gather_ligands(x, h, [sizes[i] for i in mine], group=group)
        out_pos, out_feat = [None] * len(sizes), [None] * len(sizes)
        for r in range(world):
            px = torch.split(xs[r].cpu(), all_sizes[r])
            ph = torch.split(hs[r].cpu(), all_sizes[r])
            for j, i in enumerate(shards[r]):
                out_pos[i], out_feat[i] = px[j], ph[j]
        samples, end = [], 0
        for rec_idx in range(len(ref_graphs)):
            start, end = end, end + len(n_lig_atoms[rec_idx])
            samples.append({'positions': out_pos[start:end], 'features': out_feat[start:end]})
        return samples

    @torch.no_grad()
    def sample_given_pocket(self, rec_graph, n_lig_atoms: torch.Tensor, rec_enc_batch_size: int = 32,
                            diff_batch_size: int = 32, visualize=False, fragment=None, start_ligand=None,
                            start_step: Optional[int] = None, **kw):
        """fragment: optional ``(pos [m,3], feat [m,F])``: every ligand starts with these m atoms (see _sample).
        start_ligand / start_step: optional ``(pos [m,3], feat [m,F])`` and t0: every ligand (each of size m) is a
        variant of that ligand, noised to level t0 and denoised from there (see _sample).
        visualize=True: returns (positions, features, frames), one trajectory dict per ligand (see
        sample_from_encoded_receptors)."""
        samples = self._sample([rec_graph], n_lig_atoms=[n_lig_atoms.tolist()], rec_enc_batch_size=rec_enc_batch_size,
                               diff_batch_size=diff_batch_size, visualize=visualize,
                               fragments=None if fragment is None else [fragment],
                               start_ligands=None if start_ligand is None else [start_ligand], start_step=start_step,
                               **kw)
        if visualize:
            return samples[0]['positions'], samples[0]['features'], samples[0]['frames']
        return samples[0]['positions'], samples[0]['features']

    @torch.no_grad()
    def sample_random_sizes(self, ref_graphs: List, n_replicates: int = 10, rec_enc_batch_size: int = 32,
                            diff_batch_size: int = 32, **kw):
        n_nodes_rec = torch.tensor([max(g.num_nodes('rec'), g.num_nodes('kp') if self.rec_encoder_type == 'fixed' else 0)
                                    for g in ref_graphs])
        n_lig_atoms = self.lig_size_dist.sample(n_nodes_rec, n_replicates).tolist()
        return self._sample(ref_graphs=ref_graphs, n_lig_atoms=n_lig_atoms, rec_enc_batch_size=rec_enc_batch_size,
                            diff_batch_size=diff_batch_size, **kw)
