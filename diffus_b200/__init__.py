"""diffus_b200 -- B200-native DiffUS B-mode renderer hot path.

Drop-in for ``UltrasoundRenderer.plot_beam_frame`` (+ ``generate_cone_directions`` and
``ImpedanceEstimator``) of gduguey/DiffUS over hand-written sm_100a kernels behind a C ABI
(``include/diffus_b200.h``).  Importing the package is cheap and works without a GPU; the
first op call loads ``libdiffus_b200.so`` and fails loudly if it has not been built.
"""
from .cone import generate_cone_directions
from .impedance import ImpedanceEstimator
from .ops import fan_directions, probe_rays
from .renderer import (PreparedVolume, UltrasoundRenderer, compute_echo_traces, compute_gaussian_pulse, gaussian_pulse, custom_nearest_sampler, differentiable_splat,
                       propagate_full_rays_batched, render_frames, render_gauss_newton, render_gauss_newton_sweep, render_mse_loss,
                       rotate_around_apex, smooth_volume)
from .pose_recovery import (apply_fan_twist, apply_pose_twist, apply_probe_twist, recover_poses, recover_poses_coarse_to_fine,
                            register_sweep)

__all__ = ["UltrasoundRenderer", "render_frames", "render_mse_loss", "render_gauss_newton", "PreparedVolume", "compute_echo_traces", "compute_gaussian_pulse", "gaussian_pulse",
           "propagate_full_rays_batched", "custom_nearest_sampler", "differentiable_splat", "rotate_around_apex", "generate_cone_directions",
           "fan_directions", "ImpedanceEstimator", "apply_pose_twist", "apply_fan_twist", "recover_poses", "smooth_volume",
           "recover_poses_coarse_to_fine", "probe_rays", "apply_probe_twist", "render_gauss_newton_sweep", "register_sweep"]
