/* go2policy -- C ABI of the B200-native Go2 policy hot path.
 *
 * This is the drop-in boundary: everything the reference does between
 * ONNXController::publish() gathering its inputs and handing joint targets to the
 * robot interface, i.e.
 *     A1-A6  observation assembly          reference: onnx_controller/src/controller.cpp:173-212
 *     A7     ONNXActor::act()              reference: onnx_inference/src/cpp/onnx_actor.cpp:38-48
 *                                          (Ort::Session::Run on onnx_inference/data/model.onnx)
 *     A9     clamp + dead-man mask         reference: controller.cpp:217-223
 *     A11    joint targets / gains         reference: controller.cpp:235-248
 * re-implemented as hand-written sm_100a CUDA kernels.  Plain C types only -- no
 * CUDA, torch or ONNX Runtime type crosses this boundary (streams are void*).
 *
 * There is NO CPU fallback: go2p_create fails (GO2P_ERR_NO_DEVICE) when no
 * sm_100 device is present, and every compute entry point fails loudly rather than
 * computing on the host.
 *
 * All functions return 0 (GO2P_OK) on success or a go2p_status error code;
 * go2p_last_error() returns a thread-local human-readable message.
 */
#ifndef GO2POLICY_H
#define GO2POLICY_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GO2P_ABI_VERSION 2
#define GO2P_DOF 12            /* reference: controller.hpp:13 kDimDOF   */
#define GO2P_FRAME 49          /* reference: controller.hpp:14 kDimObs   */
#define GO2P_MAX_HISTORY 8     /* reference uses kHistory = 2 (controller.hpp:15) */
#define GO2P_MAX_LAYERS 8

typedef struct go2p_handle go2p_handle;

typedef enum go2p_status {
  GO2P_OK = 0,
  GO2P_ERR_INVALID = 1,      /* bad argument                                   */
  GO2P_ERR_IO = 2,           /* model file cannot be read                      */
  GO2P_ERR_MODEL = 3,        /* .onnx is malformed or uses an unsupported op   */
  GO2P_ERR_CUDA = 4,         /* a CUDA runtime call failed                     */
  GO2P_ERR_NO_DEVICE = 5,    /* no sm_100 GPU: there is no CPU fallback        */
  GO2P_ERR_UNSUPPORTED = 6,  /* valid request the kernels cannot serve         */
  GO2P_ERR_STATE = 7,        /* call not valid in the current state            */
  GO2P_ERR_TIMEOUT = 8       /* persistent kernel did not answer               */
} go2p_status;

/* arithmetic used for the Gemm operands of the batched path (accumulation is always fp32) */
typedef enum go2p_precision {
  GO2P_PREC_FP32 = 0,        /* CUDA-core FFMA; agrees with ORT-CPU semantics to 1e-5 */
  GO2P_PREC_BF16 = 1,        /* tcgen05 kind::f16, bf16 operands                        */
  GO2P_PREC_FP16 = 2,        /* tcgen05 kind::f16, fp16 operands (saturating convert)   */
  /* 3 was reserved for kind::tf32 and is rejected: fp32 weights of the policy do not fit in shared memory beside the
   * observation ring, and fp16 operands have the same 11-bit significand (see DESIGN.md, precision contract) */
  GO2P_PREC_FP32_TC = 4      /* fp32 accuracy on the tensor cores: every operand split into three bf16 pieces (24
                              * significand bits, fp32 range), six tcgen05 kind::f16 products per K step, fp32
                              * accumulation, bias and ELU.  Same contract as GO2P_PREC_FP32 against an fp64
                              * reference (|a - ref| <= 1e-5 * max(|ref|, 1), row rel-L2 <= 1e-5), no saturation,
                              * the reference's NaN pattern for +-Inf / NaN inputs, results independent of batch
                              * size and entry point; not bit-identical to GO2P_PREC_FP32 (other summation order).
                              * Serves 2-8 layers, hidden widths that are multiples of 64, at most 16 outputs;
                              * other shapes: GO2P_ERR_UNSUPPORTED.  GO2P_F_SAT_COUNT counts nothing. */
} go2p_precision;

/* how the batch-1 control-loop step reaches the GPU */
typedef enum go2p_b1_mode {
  GO2P_B1_PERSISTENT = 0,    /* one resident kernel polls a host-mapped mailbox: launch-free */
  GO2P_B1_GRAPH = 1,         /* one CUDA-graph launch per step, zero-copy mailbox I/O        */
  GO2P_B1_LAUNCH = 2         /* plain kernel launch per step                                 */
} go2p_b1_mode;

/* flags of go2p_infer_batch_ex */
#define GO2P_F_CLAMP_MASK 1u   /* apply A9 (clamp to +-action_limit, multiply by button0==0) */
#define GO2P_F_QDES 2u         /* also emit A11 q_des = q0 + (double)a * action_scale        */
#define GO2P_F_MOTOR_CMD 4u    /* also emit the send_command arguments in Unitree motor order (go2p_motor_cmd) */
#define GO2P_F_SAT_COUNT 8u    /* GO2P_PREC_FP16 only: count operand blocks clipped at +-65504 (go2p_saturation_count) */

/* Compile-time constants of the reference exposed as one POD; go2p_config_default()
 * fills in the reference's values. */
typedef struct go2p_config {
  uint32_t struct_size;        /* = sizeof(go2p_config), for ABI evolution                    */
  int32_t device;              /* CUDA device ordinal (default 0)                             */
  int32_t b1_mode;             /* go2p_b1_mode (default: env GO2P_B1_MODE or PERSISTENT)      */
  int32_t history;             /* H; obs width must be 49*H for the fused step (default 2)    */
  float action_limit;          /* controller.hpp:16  kActionLimit = 1000                      */
  double action_scale;         /* controller.cpp:244 0.25                                     */
  double q0[GO2P_DOF];         /* controller.hpp:165                                          */
  int32_t foot_threshold;      /* controller.hpp:100-103  22                                  */
  float kp, kd;                /* controller.hpp:119-120  28.0, 0.5                           */
  float kp_deadman;            /* controller.cpp:246  5                                       */
  int32_t log_level;           /* OrtLoggingLevel numbering (onnx_actor.hpp:33), 2 = WARNING  */
  int32_t timeout_ms;          /* persistent-mailbox answer timeout (default 2000)            */
  int32_t idle_exit_ms;        /* resident kernel leaves its SM after this long without a     *
                                * request and is relaunched on demand (default 30000, 0=never)*/
} go2p_config;

/* Everything publish() reads from the outside world in one control step. */
typedef struct go2p_raw_state {
  float quat[4];               /* w,x,y,z  controller.hpp:95-97                               */
  float gyro[3];               /* controller.hpp:109                                          */
  float q[GO2P_DOF];           /* (float)robot_interface_->get_q()[i]   controller.cpp:189    */
  float dq[GO2P_DOF];          /* (float)robot_interface_->get_dq()[i]  controller.cpp:190    */
  float axes[4];               /* joy axes; 0,1,3 are read  controller.cpp:176-178            */
  int16_t foot_force[4];       /* unitree order; swapped + thresholded  controller.hpp:100-103*/
  int32_t joy_valid;           /* joy_ && !joy_->axes.empty()  controller.cpp:173             */
  int32_t button0;             /* joy_->buttons[0]  controller.cpp:221,246                    */
} go2p_raw_state;

/* What publish() hands on: the ObservationAction message payload
 * (onnx_interfaces/msg/ObservationAction.msg:1-2) and the send_command arguments. */
typedef struct go2p_step_out {
  float observation[GO2P_FRAME * GO2P_MAX_HISTORY]; /* first 49*H valid                       */
  float action_raw[GO2P_DOF];  /* policy output before clamp/mask                             */
  float action[GO2P_DOF];      /* published action (post clamp+mask, pre scaling)             */
  double q_des[GO2P_DOF];      /* controller.cpp:244                                          */
  double kp, kd;               /* controller.cpp:246-247 (same value for all 12 joints)       */
  uint64_t device_ns;          /* in-kernel time from inputs-seen to outputs-written          */
} go2p_step_out;

/* What Go2RobotInterface::send_command receives from publish() (controller.cpp:235-251), in UNITREE motor order:
 * motor u = leg*3 + joint with legs FR, FL, RR, RL and joints hip, thigh, calf; the policy works in Isaac order
 * (controller.hpp:168-170: joint*4 + leg with legs FL, FR, RL, RR).  dq_des and tau_ff are zero in the reference. */
typedef struct go2p_motor_cmd {
  double q_des[GO2P_DOF];      /* controller.cpp:244, permuted to motor order                  */
  double kp, kd;               /* controller.cpp:246-247: one value for all 12 joints          */
} go2p_motor_cmd;

typedef struct go2p_model_info_t {
  int32_t in_dim, out_dim, n_layers;
  int32_t dims[GO2P_MAX_LAYERS + 1];
  int32_t has_elu[GO2P_MAX_LAYERS];
  float elu_alpha[GO2P_MAX_LAYERS];
  const char* input_name;      /* owned by the handle                                         */
  const char* output_name;
  int64_t n_params;
  int32_t sm_count, cc_major, cc_minor;
  int32_t tensor_core_path;    /* 1 if the tcgen05 kernels can serve this model               */
} go2p_model_info_t;

typedef struct go2p_b1_stats {
  uint64_t steps;
  uint64_t device_ns_min, device_ns_max, device_ns_sum;
} go2p_b1_stats;

/* ---- lifecycle -- replaces Ort::Env / Ort::Session construction, onnx_actor.cpp:6-36 ---- */
void go2p_config_default(go2p_config* cfg);
int go2p_create(const char* onnx_path, const go2p_config* cfg, go2p_handle** out);
int go2p_destroy(go2p_handle* h);
/* replaces session_.GetInputNameAllocated / GetInputTypeInfo ..., onnx_actor.cpp:23-28 */
int go2p_model_info(const go2p_handle* h, go2p_model_info_t* info);
/* the same facts straight from a file, without a device (what print_model_info needs, onnx_actor.cpp:60-66):
 * parses the graph, fills dims / activations / names (strings owned by the library, valid until the calling
 * thread's next go2p_inspect_model) and, if checksum != NULL, a positional checksum of every layer's
 * [out][in] weights and bias: sum over elements of ((i mod 97) + 1) * value in double, layer after layer. */
int go2p_inspect_model(const char* onnx_path, go2p_model_info_t* info, double* checksum);
const char* go2p_last_error(void);
int go2p_abi_version(void);

/* ---- batch-1 control loop ---- */
/* replaces Ort::Value::CreateTensor over the caller's buffers, onnx_actor.cpp:31-35:
 * the spans are captured; every go2p_act reads obs[0..n_obs) and overwrites act[0..n_act). */
int go2p_bind(go2p_handle* h, float* obs, size_t n_obs, float* act, size_t n_act);
/* replaces session_.Run, onnx_actor.cpp:47 (A7 only, synchronous) */
int go2p_act(go2p_handle* h);
/* A1-A6 + A7 + A9 + A11 in one device round trip; history lives on the device */
int go2p_step_fused(go2p_handle* h, const go2p_raw_state* raw, go2p_step_out* out);
/* `steps` consecutive go2p_step_fused calls over raws[i % n_raws] (closed loop: the device feeds its own
 * previous action back), each timed on the host with a monotonic clock from request-written to
 * answer-read.  host_ns / device_ns (may be NULL) receive one entry per step; last (may be NULL) the
 * final step's output.  Measurement helper for BASELINE.json configs[1]. */
int go2p_b1_closed_loop(go2p_handle* h, const go2p_raw_state* raws, int n_raws, int steps,
                        uint64_t* host_ns, uint64_t* device_ns, go2p_step_out* last);
/* Profiling twin of the resident kernel: ONE bounded launch that runs `steps` closed-loop control steps with
 * the raw states read from device memory (cycled) and weights/history in shared memory -- what a profiler
 * can measure of the resident design (a kernel that never exits cannot be profiled): per-step device time =
 * elapsed_ms/steps, DRAM bytes per step from ncu.  last_action: host float[12] (may be NULL). */
int go2p_b1_selfdriven(go2p_handle* h, const go2p_raw_state* raws, int n_raws, int steps,
                       float* last_action, float* elapsed_ms);
/* controller.hpp:132-162 initial member state: histories 0, action 0, vel_cmd 0 */
int go2p_reset_history(go2p_handle* h);
/* ROS params kp/kd, controller.cpp:254-277 */
int go2p_set_gains(go2p_handle* h, float kp, float kd);
int go2p_b1_stats_get(go2p_handle* h, go2p_b1_stats* out, int reset);
/* start/stop the resident kernel explicitly (create starts it lazily on first use) */
int go2p_persistent_start(go2p_handle* h);
int go2p_persistent_stop(go2p_handle* h);

/* ---- batched inference: many robots / rollouts through the same policy ---- */
/* d_obs [B,in_dim] and d_act [B,out_dim] are DEVICE pointers, row-major fp32, the layout of
 * ObservationAction.msg repeated B times.  Asynchronous on `stream` (a cudaStream_t, may be NULL). */
int go2p_infer_batch(go2p_handle* h, const float* d_obs, float* d_act, int64_t B,
                     int precision, void* stream);
/* + fused A9/A11 epilogue. d_button0 [B] int32 (may be NULL = all 0), d_qdes [B,12] double (may be NULL) */
int go2p_infer_batch_ex(go2p_handle* h, const float* d_obs, const int32_t* d_button0,
                        float* d_act, double* d_qdes, int64_t B, int precision,
                        uint32_t flags, void* stream);
/* HOST buffers: chunked H2D -> kernel -> D2H pipeline inside the call, synchronous.
 * h_obs/h_act should be pinned (go2p_host_alloc) for full PCIe rate. */
int go2p_infer_batch_host(go2p_handle* h, const float* h_obs, float* h_act, int64_t B, int precision);
/* batched A1-A6 front-end (SURVEY 8f-1): B robots' raw state -> obs rows, history kept per robot.
 * d_raw [B] go2p_raw_state, d_prev_action [B,12] (the robots' previous published action),
 * d_obs [B,49*H] is read (old frames) and rewritten in place. */
int go2p_assemble_batch(go2p_handle* h, const go2p_raw_state* d_raw, const float* d_prev_action,
                        float* d_vel_cmd, float* d_obs, int64_t B, void* stream);
/* batched publish() for B robots (reference: controller.cpp:173-251 once per robot): A1-A6 -> A7 -> A9 -> A11 on
 * device buffers, two launches (assembly, fused policy kernel).  Per-robot state lives in the caller's buffers:
 * d_obs [B,49*H] history (in/out), d_vel_cmd [B,3] last joystick command (in/out), d_action [B,12] previous
 * published action on entry, new published (clamped, masked) action on return; d_qdes [B,12] double out.
 * kp/kd are per-robot functions of button0 alone (controller.cpp:246) and stay with the caller. */
int go2p_step_batch(go2p_handle* h, const go2p_raw_state* d_raw, float* d_vel_cmd, float* d_obs,
                    float* d_action, double* d_qdes, int64_t B, int precision, void* stream);
/* + the send_command arguments in Unitree motor order: d_cmd [B] go2p_motor_cmd (flag GO2P_F_MOTOR_CMD).  kp follows
 * d_button0 (controller.cpp:246) with the handle's gains (go2p_config.kp/kd, go2p_set_gains). */
int go2p_infer_batch_cmd(go2p_handle* h, const float* d_obs, const int32_t* d_button0, float* d_act,
                         double* d_qdes, go2p_motor_cmd* d_cmd, int64_t B, int precision,
                         uint32_t flags, void* stream);
/* go2p_step_batch ending in motor commands (SURVEY 8f-2): d_qdes or d_cmd may be NULL, not both */
int go2p_step_batch_cmd(go2p_handle* h, const go2p_raw_state* d_raw, float* d_vel_cmd, float* d_obs,
                        float* d_action, double* d_qdes, go2p_motor_cmd* d_cmd, int64_t B,
                        int precision, void* stream);
/* go2p_step_batch_cmd with per-robot resets, for fleets whose robots end their episodes at different times.
 * d_reset [B] uint8 on the device (NULL = no resets, any alignment; a torch.bool tensor qualifies).  A robot whose
 * byte is non-zero starts this step from the controller's initial state (controller.hpp:132-162): its H-1 older frames
 * of every term are 0, its previous action is 0 and its stored joystick command is 0; then the step runs as usual (the
 * newest frame is appended; without joy_valid its command is 0, and 0 is written back to d_vel_cmd).  Its outputs do not
 * depend on what its rows of d_obs / d_vel_cmd / d_action held on entry (NaN included).  Robots with a zero byte step
 * exactly as with go2p_step_batch_cmd, which is this call with d_reset = NULL.  Same argument rules and launch count
 * as go2p_step_batch_cmd. */
int go2p_step_batch_ex(go2p_handle* h, const go2p_raw_state* d_raw, const uint8_t* d_reset, float* d_vel_cmd,
                       float* d_obs, float* d_action, double* d_qdes, go2p_motor_cmd* d_cmd, int64_t B,
                       int precision, void* stream);
/* The raw states of B robots as one DEVICE array per field, the way a GPU simulator keeps them: row-major, contiguous,
 * B rows each, every pointer aligned to its element type.  Meaning of each field as in go2p_raw_state. */
typedef struct go2p_raw_fields {
  const float* quat;           /* [B,4]  w,x,y,z                                              */
  const float* gyro;           /* [B,3]                                                       */
  const float* q;              /* [B,12]                                                      */
  const float* dq;             /* [B,12]                                                      */
  const float* axes;           /* [B,4]                                                       */
  const int16_t* foot_force;   /* [B,4]  unitree order                                        */
  const uint8_t* joy_valid;    /* [B]    non-zero = joy_ && !axes.empty() (a torch.bool qualifies) */
  const uint8_t* button0;      /* [B]    non-zero = dead-man button pressed                  */
} go2p_raw_fields;
/* go2p_step_batch_ex with the raw states read from per-field device arrays instead of go2p_raw_state records: it
 * computes exactly what go2p_step_batch_ex computes from records that hold the same values (flags compared with 0), with
 * the same argument rules, reset rule and launch count.  The one-launch path (fp16 / bf16) needs every field pointer
 * 16-byte aligned where the record form needs d_raw so; otherwise the step takes the two-kernel chain, as records do.
 * A NULL handle, f or field is GO2P_ERR_INVALID. */
int go2p_step_batch_fields(go2p_handle* h, const go2p_raw_fields* f, const uint8_t* d_reset, float* d_vel_cmd,
                           float* d_obs, float* d_action, double* d_qdes, go2p_motor_cmd* d_cmd, int64_t B,
                           int precision, void* stream);
/* T consecutive go2p_step_batch_fields steps of B robots in one call, e.g. to replay recorded sensor streams
 * closed-loop.  Every field of f points at T*B rows, step-major ([T,B,w]: step t's array starts t*B rows in).
 * d_reset: [T,B] uint8 or NULL.  State in/out exactly as in the single step: d_vel_cmd [B,3], d_obs [B,49*H],
 * d_action [B,12] hold the state before step 0 on entry and after step T-1 on return.  Per-step outputs:
 * d_action_seq [T,B,12] float (required) = the published action of every step; d_qdes_seq [T,B,12] double, d_cmd_seq
 * [T,B] go2p_motor_cmd, d_obs_seq [T,B,49*H] float (the ObservationAction observation of every step): each may be NULL
 * (unlike the single step, d_qdes and d_cmd may both be NULL).
 * The call leaves exactly the bytes that T calls of go2p_step_batch_fields leave on the step-t slices, with d_action
 * copied to d_action_seq[t] and d_obs to d_obs_seq[t] after each.  fp16 / bf16 take ONE launch (go2p_last_launch_count
 * 1) where the one-launch single step would serve step 0 and every step's slices are 16-byte aligned (B % 16 == 0,
 * aligned bases); the history then stays in shared memory from step 0 to step T-1.  Every other case steps T times,
 * each step by the single step's rules (the launch count is the sum of their kernels).  Argument rules as in
 * go2p_step_batch_fields; T or B = 0 does nothing; a negative T or B, or T*B*49*H beyond int64 for
 * the largest history (H = 8), is GO2P_ERR_INVALID. */
int go2p_step_batch_fields_seq(go2p_handle* h, const go2p_raw_fields* f, int64_t T, const uint8_t* d_reset,
                               float* d_vel_cmd, float* d_obs, float* d_action, float* d_action_seq,
                               double* d_qdes_seq, go2p_motor_cmd* d_cmd_seq, float* d_obs_seq,
                               int64_t B, int precision, void* stream);
/* go2p_step_fused + the same step's send_command arguments in motor order (out may be NULL) */
int go2p_step_fused_cmd(go2p_handle* h, const go2p_raw_state* raw, go2p_step_out* out, go2p_motor_cmd* cmd);
/* isaac_of_motor[u] = Isaac joint index of Unitree motor u */
int go2p_motor_order(int32_t isaac_of_motor[GO2P_DOF]);
/* Closed-loop control step for B robots from HOST buffers (pinned for full PCIe rate): the robots' observation
 * history, joystick command and previous action live on the device inside the handle (zeroed when B changes or after
 * go2p_step_batch_host_reset), so a step moves 156 B/robot in and 48 B/robot out (+112 B with h_cmd) instead of the
 * 392 + 48 B of go2p_infer_batch_host.  h_action [B,12] out, h_cmd [B] out or NULL.  Synchronous. */
int go2p_step_batch_host(go2p_handle* h, const go2p_raw_state* h_raw, float* h_action, go2p_motor_cmd* h_cmd,
                         int64_t B, int precision);
int go2p_step_batch_host_reset(go2p_handle* h);
/* go2p_step_batch_host with per-robot resets (the rule of go2p_step_batch_ex) applied to the state the handle keeps:
 * h_reset [B] uint8 in host memory, NULL = no resets.  1 B more per robot on the way in. */
int go2p_step_batch_host_ex(go2p_handle* h, const go2p_raw_state* h_raw, const uint8_t* h_reset, float* h_action,
                            go2p_motor_cmd* h_cmd, int64_t B, int precision);
/* ---- replacing the policy weights of a live handle (a new checkpoint, a running observation normaliser, an A/B
 * comparison) without losing robot state.
 * Replace the weights and biases of every layer.  The topology of the handle is fixed at create: n_layers, dims,
 * activations and ELU alpha must match.
 * weight[l]: [dims[l+1]][dims[l]] fp32 row-major (the layout of torch nn.Linear.weight and of ONNX Gemm transB=1).
 * bias[l]: [dims[l+1]] fp32, or NULL for zeros (the bias array itself may be NULL: every bias zero).
 * obs_mean / obs_std: [in_dim] fp32 or both NULL.  They describe an observation normaliser x' = (x - mean) / std and are
 *   folded into layer 0 exactly as the reader folds a Sub(mean) -> Div(std) prefix.
 * After the call, every path computes what a handle created from an .onnx holding these tensors would compute, bit for
 *   bit.  Robot state is untouched: batch-1 history, the host-step fleet state, caller buffers, gains, log ring and
 *   saturation counter.
 * The pointer arrays are host arrays.  GO2P_ERR_INVALID: null handle, n_layers that does not match, a null weight
 * pointer, or exactly one of mean / std given.
 *
 * go2p_set_weights: the tensors are on the handle's device; the weight images are rebuilt in place by a device packer
 *   on `stream`, so "step, update, step" can be written on one stream.  The caller's tensors may be reused once
 *   `stream` has passed the update.  A resident batch-1 kernel is stopped first (its state is saved; the next batch-1
 *   call relaunches it), so the call may wait on the host for that.  The handle's own streams (batch-1, host-buffer
 *   steps) wait for the update: every go2p_* call issued after this returns sees the new weights.  Kernels the caller
 *   queued on OTHER streams are the caller's to order, as for any stream-ordered write: work that may still read the
 *   handle's weights must complete before `stream` reaches the update, and work that must see the new weights has to
 *   wait for `stream` (an event) -- the images are rewritten in place, not double-buffered. */
int go2p_set_weights(go2p_handle* h, const float* const* d_weight, const float* const* d_bias, int n_layers,
                     const float* d_obs_mean, const float* d_obs_std, void* stream);
/* the same from host memory; synchronous (the packer has completed when it returns) */
int go2p_set_weights_host(go2p_handle* h, const float* const* h_weight, const float* const* h_bias, int n_layers,
                          const float* h_obs_mean, const float* h_obs_std);

/* fp16 operands saturate at +-65504 where the fp32 reference does not.  Launches with GO2P_F_SAT_COUNT count the
 * (row, 32-column operand block) pairs in which an observation or a hidden activation was clipped on its way into a
 * Gemm; this reads (and optionally resets) the total once `stream` has drained.  0 means the fp16 path never left the
 * reference's range; otherwise use GO2P_PREC_FP32 (or bf16, which has the fp32 range) for those inputs. */
int go2p_saturation_count(go2p_handle* h, uint64_t* count, int reset, void* stream);
/* number of kernels the previous batched call launched (for bench.py's gpu_launches) */
int go2p_last_launch_count(const go2p_handle* h);

/* ---- ObservationAction log (SURVEY 8f-3; reference: onnx_interfaces/msg/ObservationAction.msg:1-2, filled at
 * controller.cpp:226-229): every go2p_step_fused appends float32[in_dim] observation + float32[12] published action to
 * a ring of `capacity` records in device memory; go2p_log_drain copies the records written since the last drain,
 * oldest first, tightly packed ((in_dim + 12) floats each), without stopping the resident kernel.  capacity 0 turns
 * logging off (the default: a control step then touches no device memory at all). */
int go2p_log_enable(go2p_handle* h, int capacity);
int go2p_log_drain(go2p_handle* h, float* out, int max_records, int* n_records, uint64_t* dropped);

/* ---- one process, several GPUs (SURVEY 7 step 7): the rows of a batch are split into contiguous shards, one per
 * device, each served by its own handle, host thread and stream set; weights are replicated at create time and no
 * data crosses between devices (no collective on this path). */
typedef struct go2p_fleet go2p_fleet;
int go2p_fleet_create(const char* onnx_path, const go2p_config* cfg, const int32_t* devices, int n_devices,
                      go2p_fleet** out);
int go2p_fleet_destroy(go2p_fleet* f);
int go2p_fleet_device_count(const go2p_fleet* f);
/* rows [begin, end) of a B-row batch that shard `i` of `n` serves (contiguous, sizes differ by at most one) */
int go2p_shard_rows(int64_t B, int n, int i, int64_t* begin, int64_t* end);
int go2p_fleet_infer_host(go2p_fleet* f, const float* h_obs, float* h_act, int64_t B, int precision);
int go2p_fleet_step_host(go2p_fleet* f, const go2p_raw_state* h_raw, float* h_action, go2p_motor_cmd* h_cmd,
                         int64_t B, int precision);
/* + per-robot resets (go2p_step_batch_host_ex): h_reset [B] uint8 in host memory, NULL = no resets, sharded like h_raw */
int go2p_fleet_step_host_ex(go2p_fleet* f, const go2p_raw_state* h_raw, const uint8_t* h_reset, float* h_action,
                            go2p_motor_cmd* h_cmd, int64_t B, int precision);
/* go2p_set_weights_host on every device of the fleet, one after the other.  On failure the devices before the failing
 * one already hold the new weights; the message names the device. */
int go2p_fleet_set_weights_host(go2p_fleet* f, const float* const* h_weight, const float* const* h_bias, int n_layers,
                                const float* h_obs_mean, const float* h_obs_std);

/* ---- small device / pinned-memory helpers so non-CUDA hosts can drive the batched path ---- */
int go2p_dev_alloc(go2p_handle* h, size_t bytes, void** dptr);
int go2p_dev_free(go2p_handle* h, void* dptr);
int go2p_host_alloc(go2p_handle* h, size_t bytes, void** hptr);   /* pinned */
int go2p_host_free(go2p_handle* h, void* hptr);
int go2p_memcpy_h2d(go2p_handle* h, void* dptr, const void* hptr, size_t bytes, void* stream);
int go2p_memcpy_d2h(go2p_handle* h, void* hptr, const void* dptr, size_t bytes, void* stream);
int go2p_stream_sync(go2p_handle* h, void* stream);
/* time `iters` back-to-back go2p_infer_batch_ex launches with CUDA events on `stream` */
int go2p_time_batch(go2p_handle* h, const float* d_obs, const int32_t* d_button0, float* d_act,
                    double* d_qdes, int64_t B, int precision, uint32_t flags, void* stream,
                    int iters, float* total_ms);

#ifdef __cplusplus
}
#endif
#endif /* GO2POLICY_H */
