"""ctypes binding of libsimba_b200.so (include/simba_b200.h).

The library is built in-tree by `__graft_entry__.build()` (or `make -C csrc`). There is no CPU
fallback: if the shared object is missing, importing a compute class raises with the build
command; if no sm_100 GPU is present, the first compute call raises SimbaError.
"""
import ctypes as C
import os
import pathlib

SIMBA_MAX_ACT = 16
SIMBA_MAX_CONSTRAINTS = 4
SIMBA_MAX_HORIZON = 1024   # and horizon * act_dim <= 1024

OBJ_REWARD, OBJ_SAFE_PENALTY, OBJ_LEAST_COST, OBJ_FEASIBLE_FIRST = 0, 1, 2, 3
PREC_FP32, PREC_BF16_TC = 0, 1
ACT_RELU, ACT_SWISH = 0, 1
UPDATE_CEM, UPDATE_MPPI = 0, 1
MAP_SPLIT, MAP_PARTICLE = 0, 1
(BUF_ACTIONS, BUF_ROW_RETURN, BUF_ROW_COSTMASK, BUF_ROW_COSTSUM, BUF_PAIRS_LOCAL, BUF_PAIRS_ALL,
 BUF_ELITE, BUF_MU, BUF_SIGMA, BUF_BEST_ACTION, BUF_BEST_SCORE, BUF_ACTIVE, BUF_SCORES) = range(13)

(ROLLOUT_FP32, ROLLOUT_TC_ONE_CTA, ROLLOUT_TC_PAIR, ROLLOUT_TC_TWO_TILE, ROLLOUT_TC_WIDE,
 ROLLOUT_TC_WIDE_OBS) = range(6)

PRECISIONS = {'fp32': PREC_FP32, 'bf16': PREC_BF16_TC}
MEMBER_MAPS = {'split': MAP_SPLIT, 'particle': MAP_PARTICLE}


class SimbaError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("simba_b200 error %d: %s" % (code, message))
        self.code = code


class ModelConfig(C.Structure):
    _fields_ = [('obs_dim', C.c_int32), ('act_dim', C.c_int32), ('ensemble_size', C.c_int32),
                ('n_layers', C.c_int32), ('units', C.c_int32)]


class Scorer(C.Structure):
    _fields_ = [('goal_begin', C.c_int32), ('goal_end', C.c_int32), ('goal_dist_index', C.c_int32),
                ('n_constraints', C.c_int32),
                ('con_begin', C.c_int32 * SIMBA_MAX_CONSTRAINTS),
                ('con_end', C.c_int32 * SIMBA_MAX_CONSTRAINTS),
                ('con_size', C.c_float * SIMBA_MAX_CONSTRAINTS),
                ('lidar_max_dist', C.c_float), ('goal_threshold', C.c_float),
                ('reward_distance', C.c_float), ('reward_goal', C.c_float),
                ('reward_clip', C.c_float), ('constrain_indicator', C.c_int32)]


class PlannerConfig(C.Structure):
    _fields_ = [('horizon', C.c_int32), ('iterations', C.c_int32), ('n_samples', C.c_int32),
                ('n_elite', C.c_int32), ('particles', C.c_int32), ('n_states', C.c_int32),
                ('smoothing', C.c_float), ('stddev_threshold', C.c_float),
                ('noise_stddev', C.c_float), ('posterior_mean_threshold', C.c_float),
                ('prior_mu', C.c_float), ('prior_sigma', C.c_float),
                ('objective', C.c_int32), ('sampling_propagation', C.c_int32),
                ('precision', C.c_int32), ('member_map', C.c_int32),
                ('rank', C.c_int32), ('world_size', C.c_int32),
                ('act_low', C.c_float * SIMBA_MAX_ACT), ('act_high', C.c_float * SIMBA_MAX_ACT),
                ('init_mean', C.c_float * SIMBA_MAX_ACT), ('init_stddev', C.c_float * SIMBA_MAX_ACT),
                ('scorer', Scorer)]


class TrainerConfig(C.Structure):
    _fields_ = [('batch_size', C.c_int32), ('max_eval_rows', C.c_int32),
                ('learning_rate', C.c_float), ('lr_schedule', C.c_int32),
                ('steps_per_epoch', C.c_int32), ('train_epochs', C.c_int32),
                ('beta1', C.c_float), ('beta2', C.c_float), ('epsilon', C.c_float),
                ('clipvalue', C.c_float), ('dropout_rate', C.c_float), ('dropout_seed', C.c_uint64),
                ('precision', C.c_int32)]


_vp, _i32, _u64, _f = C.c_void_p, C.c_int32, C.c_uint64, C.c_float
_i64 = C.c_int64
_P = C.POINTER

# name -> argtypes (every function returns int unless listed in _RESTYPES)
_SIGNATURES = {
    'simba_model_create': [_P(ModelConfig), _P(_vp)],
    'simba_model_destroy': [_vp],
    'simba_model_set_layer': [_vp, _i32, _i32, _vp, _vp],
    'simba_model_set_scaler': [_vp, _vp, _vp, _i32],
    'simba_model_commit': [_vp],
    'simba_model_set_activation': [_vp, _i32],
    'simba_planner_create': [_vp, _P(PlannerConfig), _P(_vp)],
    'simba_planner_destroy': [_vp],
    'simba_planner_set_external_draws': [_vp, _vp, _vp, _vp],
    'simba_sample_actions': [_vp, _vp, _vp, _vp, _u64, _i32, _vp, _vp, _vp],
    'simba_rollout_score': [_vp, _vp, _vp, _vp, _u64, _i32, _vp, _vp, _vp, _vp, _vp],
    'simba_score_reduce': [_vp, _vp, _vp, _vp, _vp, _vp, _vp],
    'simba_allgather_scores': [_vp, _vp, _vp, _vp],
    'simba_select_elites': [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    'simba_refit': [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    'simba_finalize_action': [_vp, _vp, _vp, _u64, _vp, _vp],
    'simba_planner_set_update_rule': [_vp, _i32, _f],
    'simba_mppi_update': [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    'simba_plan': [_vp, _vp, _u64, _vp, _vp, _vp, _vp],
    'simba_plan_host': [_vp, _vp, _u64, _vp, _vp, _vp],
    'simba_planner_buffer': [_vp, _i32, _P(_vp), _P(_u64)],
    'simba_planner_copy_buffer': [_vp, _i32, _vp, _vp],
    'simba_planner_launches_per_plan': [_vp, _P(_i32)],
    'simba_planner_count_threshold': [_vp, _P(_i32)],
    'simba_planner_rollout_kernel': [_vp, _P(_i32), _P(_i32)],
    'simba_nccl_unique_id': [_vp],
    'simba_planner_init_nccl': [_vp, _vp],
    'simba_unfold': [_vp, _vp, _vp, _vp, _u64, _i32, _i32, _i32, _vp, _vp],
    'simba_unfold_tc': [_vp, _vp, _vp, _vp, _u64, _i32, _i32, _i32, _vp, _vp],
    'simba_unfold_tc_kernel': [_vp, _i32, _i32, _P(_i32), _P(_i32)],
    'simba_ensemble_forward': [_vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp],
    'simba_ensemble_forward_tc': [_vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp],
    'simba_ensemble_forward_tc_kernel': [_vp, _i32, _P(_i32), _P(_i32)],
    'simba_scale': [_vp, _vp, _i32, _vp, _vp],
    'simba_score_trajectories': [_vp, _vp, _vp, _vp, _vp],
    'simba_scorer_eval': [_P(Scorer), _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp],
    'simba_trainer_create': [_vp, _P(TrainerConfig), _P(_vp)],
    'simba_trainer_destroy': [_vp],
    'simba_trainer_step': [_vp, _vp, _vp, _i32, _vp, _vp],
    'simba_trainer_fit': [_vp, _vp, _vp, _i64, _vp, _vp, _i32, _vp, _vp],
    'simba_trainer_validation': [_vp, _vp, _vp, _i64, _vp, _vp],
    'simba_trainer_sync_model': [_vp, _vp],
    'simba_trainer_get': [_vp, _i32, _i32, _i32, _vp, _vp],
    'simba_trainer_iterations': [_vp],
    'simba_trainer_launches_per_step': [_vp],
    'simba_model_get_layer': [_vp, _i32, _i32, _vp, _vp],
    'simba_philox_raw': [_P(C.c_uint32 * 4), _P(C.c_uint32 * 2), _P(C.c_uint32 * 4)],
    'simba_philox_normals': [_u64, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp],
    'simba_last_error': [],
    'simba_version': [],
    'simba_device_check': [],
}
_RESTYPES = {'simba_last_error': C.c_char_p, 'simba_version': C.c_char_p,
             'simba_trainer_iterations': C.c_int64}

LIB_PATH = pathlib.Path(__file__).resolve().parent / 'libsimba_b200.so'
_lib = None


def load():
    """Load libsimba_b200.so and declare every prototype. Raises ImportError if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get('SIMBA_B200_LIB', str(LIB_PATH))
    if not os.path.exists(path):
        raise ImportError(
            "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C ethz-safe-learning_b200/csrc`). There is no CPU fallback." % path)
    lib = C.CDLL(path)
    for name, argtypes in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = _RESTYPES.get(name, C.c_int)
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise SimbaError(rc, load().simba_last_error().decode('utf-8', 'replace'))


def exported_names():
    return list(_SIGNATURES)
