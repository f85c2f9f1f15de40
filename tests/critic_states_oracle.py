"""The critic state row (DESIGN.md section 4, "Critic states") restated in numpy float32, operation for operation in the
order of stage_critic_privileged (task_kernels.cu): the observation row's first 487 columns, the height-scan columns,
then 31 privileged columns, each clipped to [-5, 5]."""
import numpy as np

f32 = np.float32
NOBS, NPRIV = 487, 31


def privileged(root, net_contact_force, lfoot, rfoot, push_force, motor_constant_scale, total_mass, nominal_mass,
               friction, pd_gain_scale, epi_len):
    """(N, 31) privileged block. root (N, 13), net_contact_force (N, 38, 3), push_force (N, 3), motor_constant_scale
    (N, 12), total_mass (N), friction (N) or a scalar (the sim's), pd_gain_scale (N, 2) or None, epi_len (N)."""
    root = np.asarray(root, f32)
    n = root.shape[0]
    ncf = np.asarray(net_contact_force, f32).reshape(n, -1, 3)
    start = (np.asarray(epi_len, f32) == f32(0))[:, None]
    v = np.zeros((n, NPRIV), f32)
    v[:, 0:3] = root[:, 7:10] * f32(2.0)
    v[:, 3:6] = root[:, 10:13] * f32(0.25)
    v[:, 6:9] = np.where(start, f32(0), ncf[:, lfoot] * f32(1e-3))
    v[:, 9:12] = np.where(start, f32(0), ncf[:, rfoot] * f32(1e-3))
    v[:, 12:15] = np.where(start, f32(0), np.asarray(push_force, f32).reshape(n, 3) * f32(1e-2))
    v[:, 15:27] = np.asarray(motor_constant_scale, f32).reshape(n, 12) - f32(1)
    v[:, 27] = np.asarray(total_mass, f32).reshape(n) / f32(nominal_mass) - f32(1)
    v[:, 28] = np.broadcast_to(np.asarray(friction, f32), (n,)) - f32(1)
    if pd_gain_scale is not None:
        v[:, 29:31] = np.asarray(pd_gain_scale, f32).reshape(n, 2) - f32(1)
    return np.fmin(np.fmax(v, f32(-5)), f32(5))  # (fmin / fmax as fminf / fmaxf: a NaN becomes -5)


def state_rows(obs, height_columns, priv):
    """(N, 487 + P + 31): obs[:, :487] | the height-scan columns (N, P) or None | the privileged block."""
    obs = np.asarray(obs, f32)
    parts = [obs[:, :NOBS]] + ([np.asarray(height_columns, f32)] if height_columns is not None else []) + [priv]
    return np.concatenate(parts, axis=1)
