"""ctypes binding of include/b200rl.h (the drop-in boundary).

PyTorch tensors only provide device memory (`.data_ptr()`) and the current stream; every
computation on the hot path happens inside `libb200rl.so`.  There is no CPU fallback: if the
library is missing or the device is not an sm_100 part, calls raise.
"""

from __future__ import annotations

import ctypes as C
import os

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'lib', 'libb200rl.so')

c_i32, c_i64, c_u64, c_f32, c_f64, c_vp, c_int = (C.c_int32, C.c_int64, C.c_uint64, C.c_float,
                                                  C.c_double, C.c_void_p, C.c_int)


class ReplayCfg(C.Structure):
  _fields_ = [('max_items', c_i64), ('slot_capacity', c_i64), ('obs_bytes', c_i32),
              ('act_bytes', c_i32), ('max_window', c_i32), ('shard_count', c_i32),
              ('shard_rank', c_i32), ('device', c_i32), ('stage_slots', c_i32),
              ('frame_stack', c_i32), ('gamma', c_f32), ('reserved_f', c_f32), ('alpha', c_f64)]


class DpCfg(C.Structure):
  _fields_ = [('world', c_i32), ('rank', c_i32), ('device', c_i32), ('reserved', c_i32), ('n_params', c_i64)]


class ConvGeom(C.Structure):
  _fields_ = [(n, c_i32) for n in ('B', 'H', 'W', 'C', 'kh', 'kw', 'stride', 'pad_top',
                                   'pad_left', 'OH', 'OW', 'Cout')]


# name -> (restype, argtypes); every symbol declared in include/b200rl.h
PROTOTYPES = {
    'b200rl_version': (c_int, []),
    'b200rl_launch_count': (c_u64, []),
    'b200rl_last_error': (C.c_char_p, []),
    'b200rl_device_check': (c_int, [c_int]),
    'b200rl_replay_create': (c_int, [C.POINTER(c_vp), C.POINTER(ReplayCfg)]),
    'b200rl_replay_destroy': (c_int, [c_vp]),
    'b200rl_replay_reset': (c_int, [c_vp, c_vp]),
    'b200rl_writer_open': (c_int, [c_vp, C.POINTER(c_i32)]),
    'b200rl_writer_append': (c_int, [c_vp, c_i32, c_vp, c_vp, c_f32, c_f32, c_vp]),
    'b200rl_writer_create_item': (c_int, [c_vp, c_i32, c_i32, c_f64, C.POINTER(c_u64)]),
    'b200rl_writer_close': (c_int, [c_vp, c_i32]),
    'b200rl_writer_append_stream': (c_int, [c_vp, c_i32, c_i64, c_vp, c_int, c_vp, c_vp, c_vp, c_vp,
                                            c_vp, c_i32, c_f64, c_vp]),
    'b200rl_writer_append_multi': (c_int, [c_vp, c_i64, c_vp, c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_f64, c_vp]),
    'b200rl_replay_flush': (c_int, [c_vp, c_vp]),
    'b200rl_replay_sample': (c_int, [c_vp, c_i32, c_vp, c_int, c_vp, c_vp, c_vp, c_vp]),
    'b200rl_replay_sample_philox': (c_int, [c_vp, c_i32, c_u64, c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'b200rl_replay_gather': (c_int, [c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'b200rl_replay_gather_rows': (c_int, [c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, C.POINTER(ConvGeom), c_vp]),
    'b200rl_demo_mix': (c_int, [c_i32, c_vp, c_i32, c_vp, c_i32, c_vp, c_vp, c_vp, c_i32, c_i32, c_f32, c_vp, c_f32, c_vp, c_vp, c_vp,
                        c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'b200rl_replay_gather_sequences': (c_int, [c_vp, c_i32, c_vp, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'b200rl_replay_update_priorities': (c_int, [c_vp, c_i32, c_vp, c_vp, c_vp]),
    'b200rl_replay_info': (c_int, [c_vp, C.POINTER(c_i64), C.POINTER(c_u64), C.POINTER(c_u64),
                                   C.POINTER(c_f32), c_vp]),
    'b200rl_replay_tree_levels': (c_int, [c_vp, C.POINTER(c_i32), C.POINTER(c_i32), C.POINTER(c_i32)]),
    'b200rl_replay_tree_level_width': (c_int, [c_vp, c_i32, C.POINTER(c_i64)]),
    'b200rl_replay_tree_read': (c_int, [c_vp, c_i32, c_vp, c_i64, c_vp]),
    'b200rl_replay_tree_read_prefix': (c_int, [c_vp, c_i32, c_vp, c_i64, c_vp]),
    'b200rl_replay_mass_ptr': (c_int, [c_vp, C.POINTER(c_vp)]),
    'b200rl_replay_host_state': (c_int, [c_vp, c_vp, c_i64, C.POINTER(c_i64), c_vp]),
    'b200rl_replay_set_host_state': (c_int, [c_vp, c_vp, c_i64]),
    'b200rl_replay_segment': (c_int, [c_vp, c_i32, C.POINTER(c_vp), C.POINTER(c_i64)]),
    'b200rl_replay_set_global_mass': (c_int, [c_vp, c_vp]),
    'b200rl_replay_set_weights': (c_int, [c_vp, c_i64, c_vp, c_vp]),
    'b200rl_uniform': (c_int, [c_vp, c_i32, c_u64, c_vp, c_i64, c_vp]),
    'b200rl_epsilon_greedy': (c_int, [c_i32, c_i32, c_vp, c_i64, c_f32, c_u64, c_vp, c_vp, c_vp, c_vp]),
    'b200rl_gaussian_explore': (c_int, [c_i32, c_i32, c_vp, c_f32, c_vp, c_vp, c_u64, c_vp, c_vp, c_vp, c_vp]),
    'b200rl_dqn_td': (c_int, [c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_f32, c_f32,
                              c_f64, c_f32, c_vp, c_f32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp]),
    'b200rl_is_weight_max': (c_int, [c_i32, c_vp, c_f64, c_vp, c_i32, c_vp]),
    'b200rl_seq_priority': (c_int, [c_i32, c_i32, c_vp, C.c_float, c_vp, c_vp]),
    'b200rl_seq_is_weights': (c_int, [c_i32, c_vp, c_f64, c_f64, c_vp, c_vp]),
    'b200rl_c51_loss': (c_int, [c_i32, c_i32, c_f32, c_f32, c_vp, c_vp, c_vp, c_vp, c_f32, c_f32,
                                c_vp, c_vp, c_vp, c_vp, c_vp]),
    'b200rl_td_learning': (c_int, [c_i32, c_vp, c_vp, c_vp, c_vp, c_f32, c_f32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'b200rl_c51_loss_weighted': (c_int, [c_i32, c_i32, c_f32, c_f32, c_vp, c_vp, c_vp, c_vp, c_f32, c_vp, c_f64, c_vp, c_f32,
                                         c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'b200rl_td_learning_weighted': (c_int, [c_i32, c_vp, c_vp, c_vp, c_vp, c_f32, c_vp, c_f64, c_vp, c_f32, c_vp, c_vp, c_vp, c_vp,
                                            c_vp, c_vp, c_vp]),
    'b200rl_c51_mean_fwd': (c_int, [c_i32, c_i32, c_f32, c_f32, c_vp, c_vp, c_vp]),
    'b200rl_c51_mean_bwd': (c_int, [c_i32, c_i32, c_f32, c_f32, c_vp, c_vp, c_vp, c_vp]),
    'b200rl_dpg_action_grad': (c_int, [c_i32, c_i32, c_vp, c_f32, c_int, c_f32, c_vp, c_vp, c_vp, c_vp]),
    'b200rl_adam': (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_f32, c_f64, c_f64, c_f32, c_int,
                            c_vp, c_vp, c_vp]),
    'b200rl_learner_tail': (c_int, [c_i64, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp]),
    'b200rl_global_norm_scale': (c_int, [c_i64, c_vp, c_f32, c_vp, c_vp, c_vp, c_vp]),
    'b200rl_copy_if_period': (c_int, [c_i64, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp]),
    'b200rl_step_increment': (c_int, [c_vp, c_vp]),
    'b200rl_conv2d_fwd': (c_int, [c_vp, c_int, c_vp, c_vp, c_vp, C.POINTER(ConvGeom), c_int, c_int,
                                  c_vp, c_i64, c_vp]),
    'b200rl_conv2d_wgrad': (c_int, [c_vp, c_int, c_vp, c_vp, c_vp, C.POINTER(ConvGeom), c_int, c_vp,
                                    c_i64, c_vp]),
    'b200rl_conv2d_dgrad': (c_int, [c_vp, c_vp, c_vp, C.POINTER(ConvGeom), c_vp, c_int, c_int, c_vp,
                                    c_i64, c_vp]),
    'b200rl_linear_fwd': (c_int, [c_i32, c_i32, c_i32, c_vp, c_i32, c_vp, c_vp, c_vp, c_i32, c_int,
                                  c_int, c_vp, c_i64, c_vp]),
    'b200rl_linear_dgrad': (c_int, [c_i32, c_i32, c_i32, c_vp, c_i32, c_vp, c_vp, c_i32, c_vp, c_int,
                                    c_int, c_vp, c_i64, c_vp]),
    'b200rl_linear_wgrad': (c_int, [c_i32, c_i32, c_i32, c_vp, c_i32, c_vp, c_i32, c_vp, c_vp, c_int,
                                    c_vp, c_i64, c_vp]),
    'b200rl_act_bwd': (c_int, [c_i64, c_vp, c_vp, c_int, c_vp]),
    'b200rl_duelling_fwd': (c_int, [c_i32, c_i32, c_vp, c_vp, c_vp, c_vp]),
    'b200rl_duelling_bwd': (c_int, [c_i32, c_i32, c_vp, c_vp, c_vp, c_vp]),
    'b200rl_duelling_head_fwd': (c_int, [c_i32, c_i32, c_i32, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'b200rl_duelling_head_bwd': (c_int, [c_i32, c_i32, c_i32, c_vp, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp,
                                          c_vp, c_vp, c_vp, c_i64, c_vp]),
    'b200rl_dqn_head_td': (c_int, [c_i32, c_i32, c_i32, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                   c_vp, c_vp, c_vp, c_vp, c_f32, c_f32, c_f64, c_f32, c_vp, c_f32, c_i32, c_vp, c_vp, c_vp, c_vp,
                                   c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_vp]),
    'b200rl_mean': (c_int, [c_i32, c_vp, c_vp, c_vp]),
    'b200rl_duelling_head_wgrad': (c_int, [c_i32, c_i32, c_i32, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    'b200rl_bf16_from_f32': (c_int, [c_i64, c_vp, c_vp, c_vp]),
    'b200rl_conv2d_rows_bf16_bytes': (c_i64, [C.POINTER(ConvGeom)]),
    'b200rl_conv2d_rows_bf16_from_u8': (c_int, [c_vp, C.POINTER(ConvGeom), c_vp, c_i64, c_vp]),
    'b200rl_conv2d_fwd_bf16': (c_int, [c_vp, c_int, c_vp, c_vp, c_vp, c_int, C.POINTER(ConvGeom), c_int, c_vp, c_i64, c_vp]),
    'b200rl_conv2d_wgrad_bf16': (c_int, [c_vp, c_int, c_vp, c_vp, c_vp, C.POINTER(ConvGeom), c_vp, c_i64, c_vp]),
    'b200rl_conv2d_dgrad_bf16': (c_int, [c_vp, c_vp, c_vp, c_int, C.POINTER(ConvGeom), c_vp, c_int, c_int, c_vp]),
    'b200rl_linear_fwd_bf16': (c_int, [c_i32, c_i32, c_i32, c_vp, c_i32, c_vp, c_vp, c_vp, c_i32, c_int, c_int, c_vp, c_i64, c_vp]),
    'b200rl_linear_dgrad_bf16': (c_int, [c_i32, c_i32, c_i32, c_vp, c_i32, c_vp, c_vp, c_i32, c_int, c_vp, c_int, c_int, c_vp,
                                         c_i64, c_vp]),
    'b200rl_colsum_bf16': (c_int, [c_i32, c_i32, c_vp, c_i32, c_vp, c_vp, c_i64, c_vp]),
    'b200rl_linear_wgrad_bf16': (c_int, [c_i32, c_i32, c_i32, c_vp, c_i32, c_vp, c_i32, c_vp, c_vp, c_vp, c_i64, c_vp]),
    'b200rl_layernorm_tanh_fwd_bf16': (c_int, [c_i32, c_i32, c_vp, c_vp, c_vp, c_f32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'b200rl_dense_head_bwd_bf16': (c_int, [c_i32, c_i32, c_i32, c_vp, c_i32, c_vp, c_i32, c_vp, c_vp, c_i32, c_vp, c_int, c_vp,
                                           c_vp, c_vp, c_i64, c_vp]),
    'b200rl_layernorm_tanh_fwd': (c_int, [c_i32, c_i32, c_vp, c_vp, c_vp, c_f32, c_vp, c_vp, c_vp, c_vp]),
    'b200rl_layernorm_tanh_bwd': (c_int, [c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'b200rl_feature_layer_fwd': (c_int, [c_i32, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_f32, c_vp, c_vp, c_vp, c_vp,
                                         c_vp]),
    'b200rl_feature_layer_bwd': (c_int, [c_i32, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                         c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    'b200rl_tanh_to_spec_fwd': (c_int, [c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'b200rl_tanh_to_spec_bwd': (c_int, [c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'b200rl_concat2': (c_int, [c_i32, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp]),
    'b200rl_split_second': (c_int, [c_i32, c_i32, c_i32, c_vp, c_vp, c_vp]),
    'b200rl_workspace_bytes': (c_i64, [c_i64]),
    'b200rl_conv2d_rows_bytes': (c_i64, [C.POINTER(ConvGeom)]),
    'b200rl_conv2d_rows_from_u8': (c_int, [c_vp, C.POINTER(ConvGeom), c_vp, c_i64, c_vp]),
    'b200rl_frames_pad_u8': (c_int, [c_vp, c_i64, c_i32, c_i32, c_vp, c_vp]),
    'b200rl_x3_ws_bytes': (c_i64, [c_int, c_i32, c_i32, c_i32, C.POINTER(ConvGeom), c_int]),
    'b200rl_linear_fwd_x3': (c_int, [c_i32, c_i32, c_i32, c_vp, c_i32, c_vp, c_vp, c_vp, c_i32, c_int, c_vp, c_i64, c_vp]),
    'b200rl_linear_dgrad_x3': (c_int, [c_i32, c_i32, c_i32, c_vp, c_i32, c_vp, c_vp, c_i32, c_vp, c_int, c_vp, c_i64, c_vp]),
    'b200rl_linear_wgrad_x3': (c_int, [c_i32, c_i32, c_i32, c_vp, c_i32, c_vp, c_i32, c_vp, c_vp, c_vp, c_i64, c_vp]),
    'b200rl_conv2d_fwd_x3': (c_int, [c_vp, c_int, c_vp, c_vp, c_vp, C.POINTER(ConvGeom), c_int, c_vp, c_i64, c_vp]),
    'b200rl_conv2d_wgrad_x3': (c_int, [c_vp, c_int, c_vp, c_vp, c_vp, C.POINTER(ConvGeom), c_vp, c_i64, c_vp]),
    'b200rl_conv2d_dgrad_x3': (c_int, [c_vp, c_vp, c_vp, C.POINTER(ConvGeom), c_vp, c_int, c_vp, c_i64, c_vp]),
    'b200rl_dp_create': (c_int, [C.POINTER(c_vp), C.POINTER(DpCfg)]),
    'b200rl_dp_destroy': (c_int, [c_vp]),
    'b200rl_dp_buffers': (c_int, [c_vp, C.POINTER(c_vp), C.POINTER(c_vp)]),
    'b200rl_dp_export': (c_int, [c_vp, c_vp]),
    'b200rl_dp_import': (c_int, [c_vp, c_i32, c_vp]),
    'b200rl_dp_max_f64': (c_int, [c_vp, c_vp, c_vp, c_vp]),
    'b200rl_dp_adam': (c_int, [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, C.c_float, C.c_double, C.c_double, C.c_float, c_int,
                               c_i32, c_i32, c_vp]),
    'b200rl_dp_reduce_adam_ce': (c_int, [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, C.c_float, C.c_double, C.c_double, C.c_float, c_int,
                                 c_i32, c_vp, c_i32, c_vp]),
    'b200rl_dp_region_bytes': (c_i64, [c_i64]),
    'b200rl_dp_create_external': (c_int, [C.POINTER(c_vp), C.POINTER(DpCfg), C.POINTER(c_vp), c_vp]),
    'b200rl_dp_has_multicast': (c_int, [c_vp]),
    'b200rl_dp_adam_mc': (c_int, [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, C.c_float, C.c_double, C.c_double, C.c_float, c_int,
                          c_i32, c_i32, c_i32, c_vp]),
    'b200rl_dp_reduce_adam_mc': (c_int, [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, C.c_float, C.c_double, C.c_double, C.c_float, c_int,
                                 c_i32, c_vp, c_i32, c_vp]),
    'b200rl_dp_broadcast_mc': (c_int, [c_vp, c_i64, c_i64, c_vp, c_i32, c_i32, c_i32, c_vp]),
    'b200rl_dp_broadcast_ce': (c_int, [c_vp, c_i64, c_i64, c_vp, c_i32, c_i32, c_vp]),
    'b200rl_dp_status': (c_int, [c_vp]),
}

ACT_NONE, ACT_RELU, ACT_ELU, ACT_TANH = 0, 1, 2, 3
TD_IS_WEIGHTS_F32 = 1
# precision of the network layers (K6):
#   0  fp32 FFMA: the 1e-5 parity mode
#   1  tcgen05 with fp32 tensors: tf32 operands fetched by TMA where eligible, bf16 operands converted on the fly otherwise
#   2  bf16 dataflow: activations, weight shadows and back-propagated gradients in bf16 (kind::f16), fp32 master weights /
#      accumulation / optimizer (DQNAtariNetwork and the LayerNormMLP networks)
#   3  fp32-accurate layers on the bf16 tensor cores: fp32 tensors as in mode 0, every layer call through the `*_x3` entry
#      points (each operand split into three bf16 planes, six products per fp32 product; the precision-0 tolerance)
PRECISION_FP32, PRECISION_TC, PRECISION_BF16FLOW, PRECISION_FP32X3 = 0, 1, 2, 3
# `op` of b200rl_x3_ws_bytes
X3_LINEAR_FWD, X3_LINEAR_DGRAD, X3_LINEAR_WGRAD, X3_CONV_FWD, X3_CONV_WGRAD, X3_CONV_DGRAD = range(6)
PRECISION_BF16 = PRECISION_TC      # historical name of mode 1

_lib = None


class B200RLError(RuntimeError):
  pass


def load():
  """Loads libb200rl.so (once).  Raises if it has not been built: there is no fallback path."""
  global _lib
  if _lib is not None:
    return _lib
  if not os.path.exists(_LIB_PATH):
    raise ImportError(
        f'{_LIB_PATH} is missing: build it with `python -c "import __graft_entry__ as g; g.build()"` '
        '(or `make -C acme_b200/csrc`).  acme_b200 has no CPU fallback.')
  lib = C.CDLL(_LIB_PATH)
  for name, (res, args) in PROTOTYPES.items():
    fn = getattr(lib, name)  # AttributeError here = header / library mismatch
    fn.restype = res
    fn.argtypes = args
  _lib = lib
  return lib


def check(rc: int):
  if rc == 0:
    return
  msg = load().b200rl_last_error().decode('utf-8', 'replace')
  if rc == -1:
    raise ValueError(msg)
  raise B200RLError(f'b200rl error {rc}: {msg}')


def call(name: str, *args):
  check(getattr(load(), name)(*args))


def ptr(t):
  """Device (or host) address of a torch tensor / numpy array, None -> NULL."""
  if t is None:
    return None
  if hasattr(t, 'data_ptr'):
    return t.data_ptr()
  return t.ctypes.data


def current_stream() -> int:
  import torch
  return torch.cuda.current_stream().cuda_stream


def require_device(device: int = 0):
  """Fails loudly unless `device` is a B200-class (sm_100) GPU."""
  import torch
  if not torch.cuda.is_available():
    raise B200RLError('no CUDA device: acme_b200 runs on sm_100a GPUs only and has no CPU fallback')
  check(load().b200rl_device_check(device))
