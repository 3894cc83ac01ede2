"""ctypes binding of libphoenix_b200.so (C ABI declared in include/phoenix_b200.h).

The product path is CUDA only: if the shared library is missing, or a compute entry point
reports an error (e.g. no CUDA device), a `PhoenixB200Error` is raised -- there is no CPU
fallback and nothing here imports the test oracle.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# PDX_LIB: another build of the same library (kernel A/B experiments); default: the in-tree build
LIB_PATH = os.environ.get('PDX_LIB') or os.path.join(HERE, 'libphoenix_b200.so')
ABI_VERSION = 8
PDX_BUF_STATE_STABLE = 1          # PdxBuffers.flags
PDX_POLICY_TC_OVERLAP = 0x100     # or-ed into pdx_policy_step_tc's precision

PDX_TASK = {'hover': 0, 'circle': 1, 'takeoff': 2}
PDX_PHYSICS = {'SimplePhysics': 0, 'PyBulletPhysics': 1}
PDX_DTYPE_F32, PDX_DTYPE_F64 = 0, 1
PDX_RNG_PHILOX, PDX_RNG_TAPE = 0, 1
PDX_CTRL = {'PWM': 0, 'AttitudeRate': 1, 'Attitude': 2}


class PhoenixB200Error(RuntimeError):
    pass


class PdxConfig(C.Structure):
    _fields_ = [
        ('task', C.c_int32), ('physics', C.c_int32), ('dtype', C.c_int32), ('rng_mode', C.c_int32),
        ('observation_noise', C.c_int32), ('history', C.c_int32), ('agg', C.c_int32),
        ('obs_rate', C.c_int32), ('use_latency', C.c_int32), ('buf_size', C.c_int32),
        ('use_motor_dynamics', C.c_int32), ('reset_distribution', C.c_int32),
        ('ground_effect', C.c_int32), ('max_episode_steps', C.c_int32), ('core_dim', C.c_int32),
        ('obs_dim', C.c_int32), ('reset_on_nonfinite', C.c_int32), ('auto_reset', C.c_int32), ('control_mode', C.c_int32),
        ('reserved_i', C.c_int32 * 1),
        ('domain_randomization', C.c_double), ('time_step', C.c_double), ('sensor_dt', C.c_double),
        ('mass', C.c_double), ('inertia', C.c_double * 3), ('arm', C.c_double),
        ('gravity', C.c_double), ('thrust2weight', C.c_double), ('max_thrust', C.c_double),
        ('k_mass_dr', C.c_double), ('ftf0', C.c_double), ('ftf1', C.c_double),
        ('hover_x', C.c_double), ('hover_action', C.c_double), ('motor_time_constant', C.c_double),
        ('ou_theta', C.c_double), ('ou_sigma', C.c_double), ('lpf_ratio', C.c_double),
        ('pos_norm_std', C.c_double), ('pos_unif_range', C.c_double), ('vel_norm_std', C.c_double),
        ('quat_norm_std', C.c_double), ('quat_unif_range', C.c_double),
        ('gyro_pi', C.c_double), ('gyro_sigma_b', C.c_double), ('gyro_random_walk', C.c_double),
        ('gyro_turn_on', C.c_double),
        ('penalty_action', C.c_double), ('penalty_angle', C.c_double), ('penalty_spin', C.c_double),
        ('penalty_terminal', C.c_double), ('penalty_velocity', C.c_double),
        ('action_rate_penalty', C.c_double),
        ('target_pos', C.c_double * 3), ('init_xyz', C.c_double * 3), ('drag_coeff', C.c_double * 3),
        ('prop_xy', (C.c_double * 2) * 4), ('prop_z', C.c_double),
        ('gnd_eff_coeff', C.c_double), ('prop_radius', C.c_double), ('gnd_eff_h_clip', C.c_double),
        ('lin_damping', C.c_double), ('ang_damping', C.c_double), ('ground_z', C.c_double),
        ('reserved_d', C.c_double * 8),
    ]


class PdxBuffers(C.Structure):
    _fields_ = [
        ('n_envs', C.c_int64), ('env_offset', C.c_int64), ('device', C.c_int32), ('flags', C.c_int32),
        ('state', C.c_void_p), ('obs', C.c_void_p), ('reward', C.c_void_p), ('cost', C.c_void_p),
        ('terminated', C.c_void_p), ('truncated', C.c_void_p), ('final_obs', C.c_void_p),
        ('episode_return', C.c_void_p), ('episode_length', C.c_void_p), ('episode_stats', C.c_void_p),
        ('tape_step', C.c_void_p), ('tape_reset', C.c_void_p), ('tape_init', C.c_void_p),
    ]


class PdxMlp(C.Structure):
    _fields_ = [('hidden', C.c_int32 * 2), ('n_out', C.c_int32), ('reserved', C.c_int32),
                ('weight', C.c_void_p * 3), ('bias', C.c_void_p * 3)]


class PdxPolicy(C.Structure):
    _fields_ = [('obs_dim', C.c_int32), ('precision', C.c_int32), ('mean', C.c_void_p), ('std', C.c_void_p),
                ('eps', C.c_float), ('reserved', C.c_int32), ('pi', C.POINTER(PdxMlp)), ('v', C.POINTER(PdxMlp)),
                ('log_std', C.c_void_p), ('packed', C.c_void_p), ('seed', C.c_uint64), ('counter', C.c_uint64)]


class PdxRollout(C.Structure):
    _fields_ = [('n_steps', C.c_int32), ('reserved', C.c_int32), ('obs0', C.c_void_p), ('act', C.c_void_p),
                ('val', C.c_void_p), ('logp', C.c_void_p), ('last_val', C.c_void_p), ('scratch', C.c_void_p),
                ('scratch_bytes', C.c_int64), ('obs_moments', C.c_void_p)]


class PdxPolicySet(C.Structure):
    _fields_ = [('n_policies', C.c_int32), ('episodes', C.c_int32), ('obs_dim', C.c_int32), ('hidden', C.c_int32 * 2),
                ('n_out', C.c_int32), ('stride', C.c_int64), ('packed', C.c_void_p), ('mean', C.c_void_p),
                ('std', C.c_void_p), ('eps', C.c_float), ('reserved', C.c_int32)]


class PdxEvaluation(C.Structure):
    _fields_ = [('ret', C.c_void_p), ('cost', C.c_void_p), ('length', C.c_void_p), ('rec_obs', C.c_void_p),
                ('rec_act', C.c_void_p), ('rec_reward', C.c_void_p), ('rec_cost', C.c_void_p),
                ('rec_terminated', C.c_void_p), ('rec_truncated', C.c_void_p)]


class PdxMlpGrad(C.Structure):
    _fields_ = [('weight', C.c_void_p * 3), ('bias', C.c_void_p * 3)]


class PdxPpoBatch(C.Structure):
    _fields_ = [('n', C.c_int64), ('obs_dim', C.c_int32), ('reserved', C.c_int32), ('obs', C.c_void_p),
                ('index', C.c_void_p), ('act', C.c_void_p), ('adv', C.c_void_p), ('logp_old', C.c_void_p),
                ('target_v', C.c_void_p)]


_lib = None


def load():
    """Load (once) and type the shared library.  Raises PhoenixB200Error if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PhoenixB200Error(
            f'{LIB_PATH} not found: build it with `python -m phoenix_drone_simulation_b200.build` '
            '(nvcc, sm_100a).  There is no CPU fallback.')
    lib = C.CDLL(LIB_PATH)
    P = C.POINTER
    lib.pdx_abi_version.restype = C.c_int
    lib.pdx_last_error.restype = C.c_char_p
    lib.pdx_config_size.restype = C.c_int
    lib.pdx_buffers_size.restype = C.c_int
    lib.pdx_config_finalize.argtypes = [P(PdxConfig)]
    lib.pdx_state_quads.argtypes = [P(PdxConfig)]
    lib.pdx_state_field.argtypes = [P(PdxConfig), C.c_char_p, P(C.c_int), P(C.c_int)]
    lib.pdx_tape_slots.argtypes = [P(PdxConfig), P(C.c_int), P(C.c_int), P(C.c_int)]
    lib.pdx_step_bytes.argtypes = [P(PdxConfig)]
    lib.pdx_step_bytes.restype = C.c_int64
    lib.pdx_rollout_bytes.argtypes = [P(PdxConfig), C.c_int32]
    lib.pdx_rollout_bytes.restype = C.c_int64
    lib.pdx_device_count.restype = C.c_int
    lib.pdx_init.argtypes = [P(PdxConfig), P(PdxBuffers), C.c_uint64, C.c_uint64, C.c_void_p]
    lib.pdx_reset.argtypes = [P(PdxConfig), P(PdxBuffers), C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p]
    lib.pdx_step.argtypes = [P(PdxConfig), P(PdxBuffers), C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p]
    lib.pdx_step_many.argtypes = [P(PdxConfig), P(PdxBuffers), C.c_void_p, C.c_int32, C.c_uint64, C.c_uint64, C.c_void_p]
    lib.pdx_dump_draws.argtypes = [P(PdxConfig), P(PdxBuffers), C.c_void_p, C.c_uint64, C.c_uint64,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.pdx_gae.argtypes = [C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                            C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_int, C.c_void_p,
                            C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.pdx_moments.argtypes = [C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.pdx_policy_step.argtypes = [C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, P(PdxMlp), P(PdxMlp),
                                    C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p]
    lib.pdx_policy_pack_words.argtypes = [C.c_int32, P(PdxMlp), P(PdxMlp)]
    lib.pdx_policy_pack_words.restype = C.c_int64
    lib.pdx_policy_pack.argtypes = [C.c_int32, P(PdxMlp), P(PdxMlp), C.c_void_p, C.c_void_p]
    lib.pdx_oms_update.argtypes = [C.c_int32, C.c_void_p, C.c_void_p, C.c_double, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
    lib.pdx_stats_combine.argtypes = [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.pdx_policy_step_tc.argtypes = [C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, P(PdxMlp), P(PdxMlp),
                                       C.c_void_p, C.c_void_p, C.c_int32, C.c_uint64, C.c_uint64, C.c_int64, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p]
    lib.pdx_collect_scratch_bytes.argtypes = [C.c_int32]
    lib.pdx_collect_scratch_bytes.restype = C.c_int64
    lib.pdx_collect.argtypes = [P(PdxConfig), P(PdxBuffers), P(PdxPolicy), P(PdxRollout), C.c_uint64, C.c_uint64, C.c_void_p]
    lib.pdx_policy_tc_pack_words.argtypes = [C.c_int32, P(PdxMlp), P(PdxMlp), C.c_int32]
    lib.pdx_policy_tc_pack_words.restype = C.c_int64
    lib.pdx_policy_tc_pack.argtypes = [C.c_int32, P(PdxMlp), P(PdxMlp), C.c_int32, C.c_void_p, C.c_void_p]
    lib.pdx_evaluate.argtypes = [P(PdxConfig), P(PdxBuffers), P(PdxPolicySet), P(PdxEvaluation), C.c_uint64, C.c_uint64,
                                 C.c_void_p]
    lib.pdx_ppo_scratch_bytes.argtypes = [C.c_int32, C.c_int32, P(PdxMlp)]
    lib.pdx_ppo_scratch_bytes.restype = C.c_int64
    lib.pdx_ppo_pi_grad.argtypes = [P(PdxPpoBatch), P(PdxMlp), C.c_void_p, C.c_float, P(PdxMlpGrad), C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    lib.pdx_ppo_v_grad.argtypes = [P(PdxPpoBatch), P(PdxMlp), P(PdxMlpGrad), C.c_void_p, C.c_void_p, C.c_int64,
                                   C.c_void_p]
    lib.pdx_ppo_pi_fvp.argtypes = [P(PdxPpoBatch), P(PdxMlp), C.c_void_p, P(PdxMlp), C.c_float, C.c_float,
                                   P(PdxMlpGrad), C.c_void_p, C.c_int64, C.c_void_p]
    lib.pdx_policy_step_members.argtypes = [C.c_int32, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float,
                                            P(PdxMlp), P(PdxMlp), C.c_void_p, C.c_void_p, C.c_int64, C.c_uint64,
                                            C.c_uint64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p]
    lib.pdx_gae_members.argtypes = [C.c_int32, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_int, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p]
    lib.pdx_moments_members.argtypes = [C.c_int32, C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p]
    lib.pdx_ppo_pi_grad_members.argtypes = [C.c_int32, P(PdxPpoBatch), C.c_int64, C.c_void_p, P(PdxMlp), C.c_void_p,
                                            C.c_float, P(PdxMlpGrad), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_int64, C.c_void_p]
    lib.pdx_ppo_v_grad_members.argtypes = [C.c_int32, P(PdxPpoBatch), C.c_int64, C.c_void_p, P(PdxMlp), P(PdxMlpGrad),
                                           C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    lib.pdx_ppo_pi_fvp_members.argtypes = [C.c_int32, P(PdxPpoBatch), C.c_int64, C.c_void_p, P(PdxMlp), C.c_void_p,
                                           P(PdxMlp), C.c_float, C.c_float, P(PdxMlpGrad), C.c_int64, C.c_void_p,
                                           C.c_int64, C.c_void_p]
    lib.pdx_adam_members.argtypes = [C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_float, C.c_void_p]
    if lib.pdx_abi_version() != ABI_VERSION:
        raise PhoenixB200Error(f'ABI mismatch: library {lib.pdx_abi_version()} != binding {ABI_VERSION}')
    if lib.pdx_config_size() != C.sizeof(PdxConfig) or lib.pdx_buffers_size() != C.sizeof(PdxBuffers):
        raise PhoenixB200Error('struct layout mismatch between phoenix_b200.h and lib.py')
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise PhoenixB200Error(f'libphoenix_b200 error {rc}: {load().pdx_last_error().decode()}')


EXPORTED_SYMBOLS = [
    'pdx_abi_version', 'pdx_last_error', 'pdx_config_size', 'pdx_buffers_size',
    'pdx_config_finalize', 'pdx_state_quads', 'pdx_state_field', 'pdx_tape_slots',
    'pdx_step_bytes', 'pdx_rollout_bytes', 'pdx_device_count', 'pdx_init', 'pdx_reset', 'pdx_step',
    'pdx_step_many', 'pdx_dump_draws',
    'pdx_gae', 'pdx_moments', 'pdx_stats_combine', 'pdx_policy_step', 'pdx_policy_pack', 'pdx_policy_pack_words',
    'pdx_policy_step_tc', 'pdx_policy_tc_pack', 'pdx_policy_tc_pack_words', 'pdx_collect', 'pdx_collect_scratch_bytes', 'pdx_oms_update',
    'pdx_evaluate', 'pdx_ppo_scratch_bytes', 'pdx_ppo_pi_grad', 'pdx_ppo_v_grad', 'pdx_ppo_pi_fvp',
    'pdx_policy_step_members', 'pdx_gae_members', 'pdx_moments_members', 'pdx_ppo_pi_grad_members',
    'pdx_ppo_v_grad_members', 'pdx_adam_members', 'pdx_ppo_pi_fvp_members',
]
