"""TEST INFRASTRUCTURE ONLY -- CPU restatement (numpy, float64) of the Crazyflie env step.

This is the *oracle* for the B200 stepping engine: a from-scratch restatement of what one
`env.reset()` / `env.step()` of the reference's six `Drone*Env-v0` ids computes, written
against the reference files cited below (paths relative to
/root/reference/phoenix_drone_simulation/).  It is pinned against the reference itself:
`oracle/gen_golden.py` runs the unmodified reference (through the stand-ins in
oracle/shim/) and `tests/test_oracle_golden.py` checks this file against the committed
vectors in tests/golden/.  Only tests/, __graft_entry__.smoke() and bench.py's CPU
baseline may import it; the product package never does.

Parity status:
  * `*SimpleEnv` ids: pinned -- the reference's own arithmetic is reproduced (<= 1e-13).
  * `*BulletEnv` ids: motor/latency/observation/reward logic pinned the same way; the
    rigid-body integrator behind `stepSimulation` is third-party Bullet (not vendored,
    version un-pinned, setup.py:32), restated here as a single rigid body (SURVEY.md
    Appendix A.4).  **Parity of that integrator with real Bullet is unpinned.**

Random numbers come from a *draw source*:
  * NumpyGlobalSource -- calls the global `np.random.*` functions in exactly the
    reference's order (so seeding `np.random` identically reproduces the reference);
  * TapeSource -- reads standard normals / unit uniforms from a recorded or synthetic
    tape laid out in the fixed per-step slot order the CUDA kernel uses in tape mode.
"""
from __future__ import annotations

import math
from collections import deque

import numpy as np

DEG = np.pi / 180.0


# =============================================================================================
#  Third-party PyBullet helpers (upstream Bullet3 pybullet.c / btMatrix3x3.h), SURVEY App. B
# =============================================================================================
def quat_from_euler(rpy):
    """pybullet.getQuaternionFromEuler: half-angle products followed by normalisation."""
    phi, the, psi = float(rpy[0]) / 2.0, float(rpy[1]) / 2.0, float(rpy[2]) / 2.0
    sphi, cphi = math.sin(phi), math.cos(phi)
    sthe, cthe = math.sin(the), math.cos(the)
    spsi, cpsi = math.sin(psi), math.cos(psi)
    q = np.array([sphi * cthe * cpsi - cphi * sthe * spsi,
                  cphi * sthe * cpsi + sphi * cthe * spsi,
                  cphi * cthe * spsi - sphi * sthe * cpsi,
                  cphi * cthe * cpsi + sphi * sthe * spsi])
    n = math.sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3])
    return q / n


def quat_from_euler_unnormalised(rpy):
    """envs/utils.py:32-56 (same products, no normalisation); used for init_quaternion."""
    hr, hp, hy = rpy[0] * 0.5, rpy[1] * 0.5, rpy[2] * 0.5
    cy, sy, cp, sp, cr, sr = np.cos(hy), np.sin(hy), np.cos(hp), np.sin(hp), np.cos(hr), np.sin(hr)
    return np.array([sr * cp * cy - cr * sp * sy, cr * sp * cy + sr * cp * sy,
                     cr * cp * sy - sr * sp * cy, cr * cp * cy + sr * sp * sy])


def rot_from_quat(q):
    """pybullet.getMatrixFromQuaternion (btMatrix3x3::setRotation), row-major 3x3."""
    x, y, z, w = float(q[0]), float(q[1]), float(q[2]), float(q[3])
    s = 2.0 / (x * x + y * y + z * z + w * w)
    xs, ys, zs = x * s, y * s, z * s
    wx, wy, wz = w * xs, w * ys, w * zs
    xx, xy, xz = x * xs, x * ys, x * zs
    yy, yz, zz = y * ys, y * zs, z * zs
    return np.array([[1.0 - (yy + zz), xy - wz, xz + wy],
                     [xy + wz, 1.0 - (xx + zz), yz - wx],
                     [xz - wy, yz + wx, 1.0 - (xx + yy)]])


def euler_from_quat(q):
    """pybullet.getEulerFromQuaternion incl. the gimbal-lock branches."""
    x, y, z, w = float(q[0]), float(q[1]), float(q[2]), float(q[3])
    sarg = -2.0 * (x * z - w * y)
    if sarg <= -0.99999:
        return np.array([0.0, -0.5 * math.pi, 2.0 * math.atan2(x, -y)])
    if sarg >= 0.99999:
        return np.array([0.0, 0.5 * math.pi, 2.0 * math.atan2(-x, y)])
    return np.array([math.atan2(2.0 * (y * z + w * x), w * w - x * x - y * y + z * z),
                     math.asin(sarg),
                     math.atan2(2.0 * (x * y + w * z), w * w + x * x - y * y - z * z)])


# =============================================================================================
#  Draw sources
# =============================================================================================
class NumpyGlobalSource:
    """Issues the same `np.random.*` calls, in the same order, as the reference."""

    def begin_init(self):
        pass

    def begin_reset(self, t):
        pass

    def begin_step(self, t):
        pass

    def normal(self, loc, scale, n):
        return np.random.normal(loc, scale, size=n)

    def uniform(self, lo, hi, n):
        return np.random.uniform(lo, hi, size=n)

    def uniform1(self, lo, hi):
        return np.random.uniform(lo, hi)

    def randn(self, n):
        return np.random.randn(n)

    def randint(self, hi):
        return int(np.random.randint(0, hi))


class TapeSource:
    """Reads standardised draws from a tape.

    `reset_tape[e]` (1-D) holds the draws of the e-th reset in consumption order and
    `step_tape[t]` those of the t-th step; `normal` = loc + scale*z and
    `uniform` = lo + (hi-lo)*u, the same arithmetic numpy's legacy generator applies.
    """

    def __init__(self, reset_tape, step_tape, init_tape=None):
        self.reset_tape = reset_tape
        self.step_tape = step_tape
        self.init_tape = np.zeros(64) if init_tape is None else init_tape
        self.cur = None
        self.pos = 0

    def begin_init(self):
        self.cur, self.pos = self.init_tape, 0

    def begin_reset(self, e):
        self.cur, self.pos = self.reset_tape[e], 0

    def begin_step(self, t):
        self.cur, self.pos = self.step_tape[t], 0

    def _take(self, n):
        out = np.asarray(self.cur[self.pos:self.pos + n], dtype=np.float64)
        assert out.shape[0] == n, 'tape exhausted'
        self.pos += n
        return out

    def normal(self, loc, scale, n):
        return loc + scale * self._take(n)

    def uniform(self, lo, hi, n):
        return lo + (hi - lo) * self._take(n)

    def uniform1(self, lo, hi):
        return float(lo + (hi - lo) * self._take(1)[0])

    def randn(self, n):
        return self._take(n)

    def randint(self, hi):
        return int(self._take(1)[0])


# =============================================================================================
#  Configuration (constants of envs/assets/*.urdf and the constructor defaults)
# =============================================================================================
MODELS = {
    # envs/assets/cf21x_sys_eq.urdf:10,16-17
    'cf21x_sys_eq': dict(M=0.027, L=0.0397, T2W=2.25, IXX=1.7e-5, IYY=1.7e-5, IZZ=2.9e-5),
    # envs/assets/cf21x_bullet.urdf:12,18,30 ; prop joints :59,85,111,136
    'cf21x_bullet': dict(M=0.030, L=0.0397, T2W=1.8, IXX=1.33e-5, IYY=1.33e-5, IZZ=2.64e-5),
}
KF, GND_EFF_COEFF, PROP_RADIUS = 3.16e-10, 11.36859, 2.31348e-2
DRAG_COEFF = np.array([9.1785e-7, 9.1785e-7, 10.311e-7])
PROP_XY = np.array([[0.028, -0.028], [-0.028, -0.028], [-0.028, 0.028], [0.028, 0.028]])
PROP_Z = 0.0108
COLLISION_HALF_HEIGHT = 0.0125          # cf21x_bullet.urdf collision cylinder length .025

TASK_DEFAULTS = {
    # hover.py:7-24 ; circle.py:7-35 ; takeoff.py:13-41
    'hover': dict(penalty_action=1e-4, penalty_angle=0.0, penalty_spin=1e-4,
                  penalty_terminal=100.0, penalty_velocity=0.0, ARP=0.0),
    'circle': dict(penalty_action=1e-4, penalty_angle=0.0, penalty_spin=1e-3,
                   penalty_terminal=100.0, penalty_velocity=1e-4, ARP=1e-3),
    'takeoff': dict(penalty_action=1e-4, penalty_angle=0.0, penalty_spin=1e-4,
                    penalty_terminal=100.0, penalty_velocity=0.0, ARP=0.0),
}

ENV_IDS = {
    'DroneHoverSimpleEnv-v0': ('hover', 'simple'),
    'DroneHoverBulletEnv-v0': ('hover', 'bullet'),
    'DroneCircleSimpleEnv-v0': ('circle', 'simple'),
    'DroneCircleBulletEnv-v0': ('circle', 'bullet'),
    'DroneTakeOffSimpleEnv-v0': ('takeoff', 'simple'),
    'DroneTakeOffBulletEnv-v0': ('takeoff', 'bullet'),
}


class OracleEnv:
    """One environment, reference semantics (quirks of SURVEY.md A.6 included)."""

    def __init__(self, env_id, source=None, *, domain_randomization=0.10, observation_noise=1,
                 observation_history_size=2, enable_reset_distribution=True,
                 aggregate_phy_steps=None, latency=0.015, motor_time_constant=0.080,
                 motor_thrust_noise=0.05, use_ground_effect=False,
                 lin_damping=0.04, ang_damping=0.04, control_mode='PWM',
                 observation_frequency=100, target_pos=(0, 0, 1), use_latency=None,
                 use_motor_dynamics=None, **penalties):
        """`use_latency` / `use_motor_dynamics`: None keeps the agent's default (agents.py:165,196); a bool
        stands for the reference's debug scripts assigning drone.use_latency / drone.use_motor_dynamics
        after construction (Bullet agent only; latency still needs latency >= TIME_STEP)."""
        self.task, self.physics = ENV_IDS[env_id]
        self.src = source if source is not None else NumpyGlobalSource()
        bullet = self.physics == 'bullet'
        mdl = MODELS['cf21x_bullet' if bullet else 'cf21x_sys_eq']
        self.M, self.L, self.T2W = mdl['M'], mdl['L'], mdl['T2W']
        self.J0 = np.array([mdl['IXX'], mdl['IYY'], mdl['IZZ']])
        self.sim_freq = 200 if bullet else 100                       # hover.py:263,280
        self.agg = aggregate_phy_steps if aggregate_phy_steps is not None else (2 if bullet else 1)
        if self.task == 'takeoff' and not bullet:
            self.agg = 1                                             # takeoff.py:224
        self.TIME_STEP = 1.0 / self.sim_freq                         # base.py:98
        self.obs_rate = int(self.sim_freq // observation_frequency)  # base.py:108
        self.dr = domain_randomization
        self.noise_on = observation_noise > 0
        self.H = observation_history_size
        self.reset_dist = enable_reset_distribution
        self.use_ground_effect = use_ground_effect
        self.lin_damping, self.ang_damping = lin_damping, ang_damping
        self.pen = dict(TASK_DEFAULTS[self.task])
        self.pen.update(penalties)

        # agents.py:142-206
        self.G = 9.81
        self.FTF0, self.FTF1 = 1.56e-5, 5.96e-3
        self.GRAVITY = self.G * self.M
        self.MAX_THRUST = self.GRAVITY * self.T2W / 4
        self.HOVER_X = np.sqrt(1 / self.T2W)
        self.HOVER_ACTION = 2 * 1 / self.T2W - 1
        max_rpm = np.sqrt((self.T2W * self.GRAVITY) / (4 * self.MAX_THRUST))
        self.GND_EFF_H_CLIP = 0.25 * PROP_RADIUS * np.sqrt(
            (15 * max_rpm ** 2 * KF * GND_EFF_COEFF) / self.MAX_THRUST)
        self.use_latency = bullet and latency >= self.TIME_STEP       # agents.py:165
        if use_latency is not None and bullet:
            self.use_latency = bool(use_latency) and latency >= self.TIME_STEP
        self.use_motor_dynamics = bullet
        if use_motor_dynamics is not None and bullet:
            self.use_motor_dynamics = bool(use_motor_dynamics)
        self.buf_size = int(max(1, int(latency // self.TIME_STEP)))  # agents.py:180
        self.MOTOR_T = motor_time_constant
        self.ou_sigma = 0.2 * motor_thrust_noise                     # agents.py:206
        self.ou_theta = 0.15
        # control.py:13-26,120-287: firmware PID gains; the controllers keep the NOMINAL time step
        # under domain randomisation (agents.py:74-78, quirk A.6-13)
        assert control_mode in ('PWM', 'AttitudeRate', 'Attitude')
        self.control_mode = control_mode
        self.rate_kp = np.array([250.0, 250.0, 120.0])
        self.rate_ki = np.array([500.0, 500.0, 16.7])
        self.rate_kd = np.array([2.5, 2.5, 0.0])
        self.rate_lim = np.array([33.3, 33.3, 166.7])
        self.att_kp = np.array([6.0, 6.0, 6.0])
        self.att_ki = np.array([3.0, 3.0, 1.0])
        self.att_kd = np.array([0.0, 0.0, 0.35])
        self.att_lim = np.array([20.0, 20.0, 360.0])
        self.rate_int, self.rate_err = np.zeros(3), np.zeros(3)
        self.att_int, self.att_err = np.zeros(3), np.zeros(3)

        # sensors.py:18-33,121-128 (dt is the *nominal* 1/SIM_FREQ, hover.py:144)
        sdt = 1 / self.sim_freq
        sg = 0.000175 / (sdt ** 0.5)
        self.gyro_sigma_b = (-(sg ** 2) * (1000. / 2) * (math.exp(-2 * sdt / 1000.) - 1)) ** 0.5
        self.gyro_pi = math.exp(-sdt / 1000.)
        self.gyro_rw = 0.0105
        self.gyro_turn_on = np.pi * 5 / 180
        self.quat_std = np.pi * 0.1 / 180
        self.quat_unif = np.pi * 0.05 / 180
        self.lpf_ratio = (1 / self.sim_freq) / (2 / self.sim_freq)   # base.py:109-110

        # reference trajectories: circle.py:46-56, takeoff.py:44-48
        if self.task == 'circle':
            n = 3 * 100
            ts = 2 * np.pi * np.arange(n) / n
            self.ref = np.zeros((n, 3))
            self.ref[:, 2] = 1.
            self.ref[:, 1] = 0.25 * np.sin(ts)
            self.ref[:, 0] = 0.25 * (1 - np.cos(ts))
        elif self.task == 'takeoff':
            self.ref = np.zeros((300, 3))
            self.ref[:, 2] = np.arange(300) / 300
        self.num_ref = 300
        self.ref_offset = 0
        self.target_pos = np.array(target_pos, dtype=np.float32)     # hover.py:14 (Circle / TakeOff overwrite it)

        z0 = 0.0125 if self.task == 'takeoff' else 1.0
        self.init_xyz = np.array([0, 0, z0], dtype=np.float32)       # float32! hover.py:44
        self.init_quat = quat_from_euler_unnormalised(np.zeros(3))
        self.init_xyz_dot, self.init_rpy_dot = np.zeros(3), np.zeros(3)      # base.py:117-118

        # --- persistent state (SURVEY A.8) ---
        self.xyz = np.array([0., 0., 1.])
        self.rpy = np.zeros(3)
        self.quat = quat_from_euler(self.rpy)
        self.vel = np.zeros(3)
        self.omega = np.zeros(3)                  # body rates (`rpy_dot`)
        self.omega_world = np.zeros(3)            # Bullet only
        self.dt = self.TIME_STEP
        self.m = self.M
        self.J = self.J0.copy()
        self.J_inv = 1.0 / self.J
        self.ftf0, self.ftf1 = self.FTF0, self.FTF1
        self.A = np.ones(4) * (1 - self.TIME_STEP / self.MOTOR_T)
        self.B = np.ones(4) * self.TIME_STEP / self.MOTOR_T
        self.K = self.MAX_THRUST
        self.x = np.zeros(4)
        self.ring = np.zeros((self.buf_size, 4))
        self.ring_idx = 0
        self.drone_last_action = np.zeros(4)
        self.env_last_action = np.zeros(4)
        self.ou = np.ones(4) * 0
        self.gyro_bias = np.zeros(3)
        self.lpf = 0
        self.cache = np.zeros(10)
        self.obs_hist = deque(maxlen=self.H)
        self.act_hist = deque(maxlen=self.H)
        self.iteration = 0
        self.n_resets = 0
        self.n_steps = 0
        # base.py:143 -- the constructor really calls compute_observation() once to size the
        # observation space: with noise on this consumes 33 draws and seeds the gyro bias.
        self.src.begin_init()
        self.obs_dim = self.H * (self._observe().size + 4)

    # ----------------------------------------------------------------------------------------
    #  control.act: control.py:94-100 (PWM), :120-191 (AttitudeRate), :194-287 (Attitude)
    # ----------------------------------------------------------------------------------------
    def set_latency(self, new_latency):
        """agents.py:388-404 (called by the simulation-optimisation objective): NOTE the true division, where the
        constructor (agents.py:180) floors -- 0.015 s is 3 sub-steps here and 2 there."""
        self.latency = new_latency
        if new_latency < self.TIME_STEP:
            self.use_latency = False
        else:
            self.use_latency = True
            self.buf_size = int(new_latency / self.TIME_STEP)
            assert self.buf_size > 0
            self.ring = np.zeros((self.buf_size, 4))
            self.ring_idx = 0

    def _rate_pid(self, rpy_dot_target):
        dt = self.TIME_STEP
        error = (rpy_dot_target - self.omega) * 180. / np.pi
        derivative = (error - self.rate_err) / dt
        self.rate_err = error
        self.rate_int = self.rate_int + error * dt
        self.rate_int = np.clip(self.rate_int, -self.rate_lim, self.rate_lim)
        return self.rate_kp * error + self.rate_ki * self.rate_int + self.rate_kd * derivative

    def _att_pid(self, rpy_target):
        dt = self.TIME_STEP
        error = (rpy_target - self.rpy) * 180. / np.pi
        derivative = (error - self.att_err) / dt
        self.att_err = error
        self.att_int = self.att_int + error * dt
        self.att_int = np.clip(self.att_int, -self.att_lim, self.att_lim)
        offs = self.att_kp * error + self.att_ki * self.att_int + self.att_kd * derivative
        return offs / 180. * np.pi

    @staticmethod
    def _mix(f, thrust):
        """rpy_control_factors_to_PWM, control.py:34-50 (QUAD_FORMATION_X)."""
        r, p, y = f[0] / 2.0, f[1] / 2.0, f[2]
        return np.array([np.clip(thrust - r - p - y, 0, 60000), np.clip(thrust - r + p + y, 0, 60000),
                         np.clip(thrust + r + p - y, 0, 60000), np.clip(thrust + r - p + y, 0, 60000)])

    def _control(self, action):
        """`action` keeps its dtype: float32 from the policy (Simple agent) or float64 out of the
        latency ring -- the leading arithmetic of every mode runs in that dtype (quirk A.6-3)."""
        clipped = np.clip(action, -1, 1)
        if self.control_mode == 'PWM':
            return 30000 + clipped * 30000
        if self.control_mode == 'AttitudeRate':
            thrust = 30000 + clipped[0] * 30000
            return self._mix(self._rate_pid(clipped[1:4] * np.pi / 3), thrust)
        thrust = 45000 + clipped[0] * 10000
        rate_targets = self._att_pid(clipped[1:4] * np.pi / 18)
        return self._mix(self._rate_pid(rate_targets), thrust)

    # ----------------------------------------------------------------------------------------
    #  motor model: agents.py:259-298, envs/utils.py:104-108
    # ----------------------------------------------------------------------------------------
    def _motor(self, action):
        self.drone_last_action = action.copy()
        if self.use_latency:
            delayed = self.ring[self.ring_idx].copy()
            self.ring[self.ring_idx] = action
            self.ring_idx = (self.ring_idx + 1) % self.buf_size
        else:
            delayed = action
        pwm = self._control(delayed)
        self.ou = self.ou + (self.ou_theta * (0 - self.ou) + self.ou_sigma * self.src.randn(4))
        u = pwm / 60000
        if self.use_motor_dynamics:
            self.x = self.A * self.x + self.B * np.sqrt(u)
            noisy = (1 + self.ou) * self.x ** 2
        else:
            noisy = (1 + self.ou) * u
        forces = self.K * np.clip(noisy, 0, 1)
        tq = self.ftf1 * forces + self.ftf0
        z_torque = (-tq[0] + tq[1] - tq[2] + tq[3])
        return forces, z_torque

    # ----------------------------------------------------------------------------------------
    #  ground effect: physics.py:27-58 (dead by default; SURVEY config 4 switches it on)
    # ----------------------------------------------------------------------------------------
    def _ground_effect(self, forces, R):
        prop_z = np.array([self.xyz[2] + R[2, 0] * PROP_XY[i, 0] + R[2, 1] * PROP_XY[i, 1]
                           + R[2, 2] * (PROP_Z if self.physics == 'bullet' else 0.0)
                           for i in range(4)])
        prop_z = np.clip(prop_z, self.GND_EFF_H_CLIP, np.inf)
        ge = forces * GND_EFF_COEFF * (PROP_RADIUS / (4 * prop_z)) ** 2
        if np.abs(self.rpy[0]) < np.pi / 2 and np.abs(self.rpy[1]) < np.pi / 2:
            return ge
        return np.zeros_like(ge)

    # ----------------------------------------------------------------------------------------
    #  SimplePhysics.step_forward: physics.py:130-200
    # ----------------------------------------------------------------------------------------
    def _physics_simple(self, action):
        forces, z_torque = self._motor(action)
        R = rot_from_quat(self.quat)
        if self.use_ground_effect:                       # extension (not in reference)
            forces = forces + self._ground_effect(forces, R)
        thrust = np.array([0, 0, np.sum(forces)])
        force_world = np.dot(R, thrust) - np.array([0, 0, self.G]) * self.m
        x_torque = (-forces[0] - forces[1] + forces[2] + forces[3]) * self.L / np.sqrt(2)
        y_torque = (-forces[0] + forces[1] + forces[2] - forces[3]) * self.L / np.sqrt(2)
        torques = np.array([x_torque, y_torque, z_torque])
        torques = torques - np.cross(self.omega, self.J * self.omega)
        alpha = self.J_inv * torques
        acc = force_world / self.m
        self.vel = self.vel + self.dt * acc
        self.omega = self.omega + self.dt * alpha
        self.xyz = self.xyz + self.dt * self.vel
        self.rpy = self.rpy + self.dt * self.omega
        self.quat = quat_from_euler(self.rpy)
        self.xyz[2] = np.clip(self.xyz[2], 0, np.inf)

    # ----------------------------------------------------------------------------------------
    #  PyBulletPhysics.step_forward: physics.py:91-124 + single-rigid-body stepSimulation
    #  (SURVEY A.4; integrator parity with real Bullet is UNPINNED)
    # ----------------------------------------------------------------------------------------
    def _physics_bullet(self, action):
        forces, z_torque = self._motor(action)
        R = rot_from_quat(self.quat)
        rpm = self.x ** 2 * 25000
        k = -1 * DRAG_COEFF * np.sum(2 * np.pi * rpm / 60)
        drag_link = np.dot(R, k * self.vel)              # physics.py:113 (quirk: R applied...
        f_eff = forces
        if self.use_ground_effect:
            f_eff = forces + self._ground_effect(forces, R)
        # ... and LINK_FRAME application rotates it once more, agents.py:300-309)
        f_body = np.array([0.0, 0.0, np.sum(f_eff)]) + drag_link
        t_body = np.array([np.sum(PROP_XY[:, 1] * f_eff), -np.sum(PROP_XY[:, 0] * f_eff), z_torque])
        v_body = R.T @ self.vel
        w_body = R.T @ self.omega_world
        f_body = f_body + R.T @ (np.array([0.0, 0.0, -9.81]) * self.m)
        Jw = self.J * w_body
        f_body = f_body - self.m * v_body * (self.lin_damping + self.lin_damping * np.linalg.norm(v_body))
        t_body = t_body - Jw * (self.ang_damping + self.ang_damping * np.linalg.norm(w_body))
        t_body = t_body - np.cross(w_body, Jw)
        self.vel = self.vel + self.dt * (R @ (f_body / self.m))
        self.omega_world = self.omega_world + self.dt * (R @ (t_body / self.J))
        self.xyz = self.xyz + self.dt * self.vel
        wn = np.linalg.norm(self.omega_world)
        if wn * self.dt > 1e-12:
            half = 0.5 * wn * self.dt
            ax = self.omega_world / wn * math.sin(half)
            dq = np.array([ax[0], ax[1], ax[2], math.cos(half)])
            q = _quat_mul(dq, self.quat)
            self.quat = q / np.linalg.norm(q)
        if self.xyz[2] < COLLISION_HALF_HEIGHT:          # crude ground plane (see shim)
            self.xyz[2] = COLLISION_HALF_HEIGHT
            self.vel[2] = max(self.vel[2], 0.0)
        self._readback()

    def _readback(self):
        """agents.py:434-453 for the Bullet integrator state."""
        self.rpy = euler_from_quat(self.quat)
        self.omega = rot_from_quat(self.quat).T @ self.omega_world

    # ----------------------------------------------------------------------------------------
    #  observation: hover.py:131-163, circle.py:128-177, takeoff.py:107-149, sensors.py:75-134
    # ----------------------------------------------------------------------------------------
    def _noisy_gyro(self):
        self.gyro_bias = self.gyro_pi * self.gyro_bias + self.gyro_sigma_b * self.src.normal(0, 1, 3)
        return self.omega + self.gyro_bias + self.gyro_rw * self.src.normal(0, 1, 3) \
            + self.gyro_turn_on * self.src.normal(0, 1, 3)

    def _observe(self):
        if self.task == 'circle':
            t = (self.iteration // self.agg + self.ref_offset) % self.num_ref
            self.target_pos = self.ref[t]
        elif self.task == 'takeoff':
            t = int(min(self.iteration, self.num_ref - 1))
            self.target_pos = self.ref[t]
        if not self.noise_on:
            state = np.concatenate([self.xyz, self.quat, self.vel, self.omega])
            if self.task == 'hover':
                return np.concatenate([state, self.drone_last_action])
            err = self.target_pos - self.xyz
            if self.task == 'circle':
                return np.concatenate([state, err])
            return np.concatenate([state, self.drone_last_action, err])
        s = self.src
        if self.iteration % self.obs_rate == 0:
            xyz = self.xyz + (s.normal(0., 0.002, 3) + s.uniform(-0.001, 0.001, 3))
            vel = self.vel + s.normal(0., 0.01, 3) + s.uniform(-0., 0., 3)
            omega = self._noisy_gyro()
            theta = s.normal(0, self.quat_std, 3) + s.uniform(-self.quat_unif, self.quat_unif, 3)
            rpy = np.clip(self.rpy + theta, [-np.pi, -np.pi / 2, -np.pi], [np.pi, np.pi / 2, np.pi])
            s.normal(0., 0.002, 3)                   # accelerometer noise: drawn, discarded
            s.normal(0., 0.005, 3)
            quat = quat_from_euler(rpy)
            self.cache = np.concatenate([xyz, quat, vel])
        else:
            xyz, quat, vel = self.cache[0:3], self.cache[3:7], self.cache[7:10]
            omega = self._noisy_gyro()
        self.lpf = (1 - self.lpf_ratio) * self.lpf + 1. * self.lpf_ratio * omega
        core = [xyz, quat, vel, self.lpf]
        if self.task == 'takeoff':
            core.append(self.drone_last_action)
        if self.task != 'hover':
            core.append(self.target_pos - xyz)
        return np.concatenate(core)

    def _history(self):
        """base.py:303-319: emit [o(k-H+1), a(k-H), ..., o(k), a(k-1)], then push a(k)."""
        self.obs_hist.append(self._observe())
        hist = np.concatenate([np.concatenate([o, a]) for o, a in zip(self.obs_hist, self.act_hist)])
        self.act_hist.append(self.drone_last_action)
        return hist

    # ----------------------------------------------------------------------------------------
    #  done / reward / cost
    # ----------------------------------------------------------------------------------------
    def _done(self):
        if self.task == 'hover':                     # hover.py:89-101
            d = np.pi * 60 / 180
            rp = self.rpy[:2]
            z_limit = self.xyz[2] < 0.2
            rpy_limit = bool((np.abs(rp) > d).any())
            rate_limit = bool((180 * np.abs(self.omega) / np.pi > 300).any())
            return bool(rpy_limit or rate_limit or z_limit)
        if self.task == 'circle':                    # circle.py:116-120
            return bool(np.linalg.norm(self.xyz - self.target_pos) > 0.25)
        return False                                 # takeoff.py:96-100

    def _reward(self, action):
        p = self.pen
        if self.task == 'circle':
            act_diff = action - self.env_last_action               # circle.py:186
        else:
            act_diff = action - self.drone_last_action             # hover.py:171 (== 0)
        nca = 0.5 * (np.clip(action, -1, 1) + 1)
        penalty_action = p['penalty_action'] * np.linalg.norm(nca)
        penalty_action_rate = p['ARP'] * np.linalg.norm(act_diff)
        penalty_rpy = p['penalty_angle'] * np.linalg.norm(self.rpy)
        penalty_spin = p['penalty_spin'] * np.linalg.norm(self.omega)
        penalty_terminal = p['penalty_terminal'] if self._done() else 0.
        cvel = p['penalty_action'] if self.task == 'takeoff' else p['penalty_velocity']  # takeoff.py:165
        penalty_velocity = cvel * np.linalg.norm(self.vel)
        penalties = np.sum([penalty_rpy, penalty_action_rate, penalty_spin,
                            penalty_velocity, penalty_action, penalty_terminal])
        dist = np.linalg.norm(self.xyz - self.target_pos)
        reward = -dist - penalties
        if self.task == 'takeoff' and self.xyz[2] < 0.08:
            reward -= 1.
        return reward

    def _cost(self):
        if self.task != 'hover':
            return 0.
        c = 0.                                       # hover.py:103-129
        x, y, z = self.xyz
        if np.abs(x) > 0.10 or np.abs(y) > 0.10 or z > 1.20:
            c = 1.
        if (np.abs(self.rpy[:2]) > np.pi * 10 / 180).any():
            c = 1.
        # Quirk (hover.py:118-124): the 17-vector of get_state() is [xyz, quat(4), vel, rates,
        # last_action], so `state[10:13]` -- meant as the linear velocity -- is really the
        # body rates, and `state[13:16]` -- meant as the rates -- is last_action[0:3].
        if (np.abs(self.omega) > 0.25).any():
            c = 1.
        if (np.abs(self.drone_last_action[0:3]) > np.pi * 200 / 180).any():
            c = 1.
        return c

    # ----------------------------------------------------------------------------------------
    #  reset: base.py:382-431, task_specific_reset, apply_domain_randomization
    # ----------------------------------------------------------------------------------------
    def _task_reset(self):
        s = self.src
        pos = self.init_xyz.copy()                   # float32 array (A.6-6)
        vel = np.array(self.init_xyz_dot, dtype=np.float64)          # hover.py:196-197 (zeros unless a caller set
        omega_s = np.array(self.init_rpy_dot, dtype=np.float64)      # them: simopt/pybullet.py:147-154)
        quat = self.init_quat.copy()
        if self.task == 'takeoff':                   # takeoff.py:179-212
            if self.reset_dist:
                pos[:2] += s.uniform(-0.25, 0.25, 2)
                quat = quat_from_euler(np.array([0, 0, s.uniform1(-np.pi, np.pi)]))
            self.x[:] = 0.
            self.ring[:] = -1
            self.drone_last_action[:] = -1
            return pos, quat, vel, omega_s
        if self.reset_dist:
            if self.task == 'hover':                 # hover.py:192-243
                pos += s.uniform(-0.25, 0.25, 3)     # in-place on float32
                rpy = s.uniform(-np.pi / 6, np.pi / 6, 3)
                rpy[2] = s.uniform1(-2 * np.pi, 2 * np.pi)
                quat = quat_from_euler(rpy)
                vel = vel + s.uniform(-0.1, 0.1, 3)
                lim = np.pi * 200 / 180
                omega_s = omega_s + s.uniform(-lim, lim, 3)
                omega_s[2] = s.uniform1(-(np.pi * 20 / 180), np.pi * 20 / 180)
            else:                                    # circle.py:213-277
                self.ref_offset = s.randint(self.num_ref)
                self.target_pos = self.ref[self.ref_offset]
                pos = self.target_pos.copy()
                pos += s.uniform(-0.05, 0.05, 3)
                a0 = np.pi * 20 / 180
                rpy = s.uniform(-a0, a0, 3)
                rpy[2] = s.uniform1(-0.1 * np.pi, 0.1 * np.pi)
                quat = quat_from_euler(rpy)
                vel = vel + s.uniform(-0.1, 0.1, 3)
                lim = np.pi * 50 / 180
                omega_s[:2] = s.uniform(-lim, lim, 2)
                omega_s[2] = s.uniform1(-(np.pi * 20 / 180), np.pi * 20 / 180)
            self.x = s.normal(self.HOVER_X, 0.02, 4)
            self.ring = np.clip(s.normal(self.HOVER_ACTION, 0.02, self.ring.size).reshape(
                self.ring.shape), -1, 1)
            self.drone_last_action = self.ring[-1, :]        # a *view* (aliasing quirk)
        return pos, quat, vel, omega_s

    def _domain_randomize(self):
        """base.py:239-296 ; agents.py:208-224."""
        if not self.dr > 0:
            return
        s, f = self.src, self.dr

        def draw(v, n=None):
            b = f * v
            return s.uniform1(v - b, v + b) if n is None else s.uniform(v - b, v + b, n)

        self.dt = draw(self.TIME_STEP)
        self.m = draw(self.M)
        self.J = draw(self.J0, 3)
        self.J_inv = 1.0 / self.J                    # np.linalg.inv of a diagonal matrix
        self.ftf0 = draw(self.FTF0)
        self.ftf1 = draw(self.FTF1)
        if self.use_motor_dynamics:
            mtc = draw(self.MOTOR_T, 4)
            t2w = draw(self.T2W, 4)
            T = np.clip(mtc, self.dt, np.inf)
            self.A = 1 - self.dt / T
            self.B = self.dt / T
            self.K = 0.028 * self.G * t2w / 4        # hard-coded mass (A.6-7)

    def reset(self):
        self.src.begin_reset(self.n_resets)
        self.n_resets += 1
        self.iteration = 0
        # drone.reset(): agents.py:377-386 (control.reset(): control.py:182-191,282-287)
        self.rate_int, self.rate_err = np.zeros(3), np.zeros(3)
        self.att_int, self.att_err = np.zeros(3), np.zeros(3)
        self.x = np.zeros(4)
        self.ring_idx = 0
        self.ring = np.zeros_like(self.ring)
        self.drone_last_action = self.ring[-1, :]
        pos, quat, vel, omega_s = self._task_reset()
        R = rot_from_quat(quat)
        omega_world = R.T @ omega_s                  # hover.py:242: R^T w written as world rate
        self._domain_randomize()
        self.lpf = self.omega                        # base.py:411: stale body rates (A.6-5)
        # update_information(): agents.py:434-453
        self.xyz = np.array(pos, dtype=np.float64)
        self.quat = np.array(quat, dtype=np.float64)
        self.rpy = euler_from_quat(self.quat)
        self.vel = np.array(vel, dtype=np.float64)
        self.omega_world = omega_world
        self.omega = rot_from_quat(self.quat).T @ omega_world        # R^T again (A.6-4)
        obs = self._observe()
        for _ in range(self.H):
            self.obs_hist.append(obs)
        action = self.drone_last_action
        for _ in range(self.H):
            self.act_hist.append(action)
        self.env_last_action = action
        return self._history(), {}

    def step(self, action):
        self.src.begin_step(self.n_steps)
        self.n_steps += 1
        for _ in range(self.agg):
            if self.physics == 'simple':
                self._physics_simple(action)
            else:
                self._physics_bullet(action)
            self._observe()                          # discarded; advances RNG + gyro LPF
            self.iteration += 1
        obs = self._history()
        r = self._reward(action)
        cost = self._cost()
        terminated = self._done()
        self.env_last_action = action
        return obs, r, terminated, False, {'cost': cost}

    # --- helpers for the parity harness -----------------------------------------------------
    def snapshot(self):
        return dict(xyz=self.xyz.copy(), rpy=self.rpy.copy(), quat=self.quat.copy(),
                    vel=self.vel.copy(), omega=self.omega.copy())


def _quat_mul(a, b):
    ax, ay, az, aw = a
    bx, by, bz, bw = b
    return np.array([aw * bx + ax * bw + ay * bz - az * by,
                     aw * by - ax * bz + ay * bw + az * bx,
                     aw * bz + ax * by - ay * bx + az * bw,
                     aw * bw - ax * bx - ay * by - az * bz])


def draws_per_phase(env_id, **kwargs):
    """(reset_slots, step_slots): tape widths, counted by dry-running one reset + one step of an OracleEnv
    built with `kwargs`."""
    class _Count(TapeSource):
        def __init__(self):
            self.n = 0
            self.counts = {}
            self.phase = None

        def begin_init(self):
            self.phase, self.counts['init'] = 'init', 0

        def begin_reset(self, e):
            self.phase, self.counts['reset'] = 'reset', 0

        def begin_step(self, t):
            self.phase, self.counts['step'] = 'step', 0

        def _take(self, n):
            self.counts[self.phase] += n
            return np.zeros(n)

    c = _Count()
    env = OracleEnv(env_id, c, **kwargs)
    env.reset()
    env.step(np.zeros(4, dtype=np.float32))
    return c.counts['reset'], c.counts['step']
