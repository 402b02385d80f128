/*
 * ppo_core.h — C ABI of the B200-native PPO training core (libppo_core.so).
 *
 * This is the drop-in boundary for the data-parallel hot path of Antymon/ppo_cpp.  The reference has
 * no FFI of its own: the path sits behind C++ classes that call tensorflow::Session::Run.  Each entry
 * point below names the reference interface it replaces (file:line in the reference tree); the C++
 * classes in ppo_cpp_b200/host/ (same names and signatures as the reference's) and the Python ctypes
 * mirror in ppo_cpp_b200/core.py call ONLY these functions.
 *
 * Conventions
 *   - plain pointers and sizes; no C++/torch types.  Every function returns 0 on success or a
 *     negative ppo_status; ppo_last_error() gives the message (thread-local).
 *   - `mem` says where caller buffers live: PPO_HOST (pageable or pinned host memory; the call does
 *     the H2D/D2H copies on the core's stream and returns after they completed — with one exception:
 *     PINNED input buffers of ppo_runner_observe are DMA'd in place and the call returns once the copies are
 *     enqueued; they must stay valid and unmodified until the next call that returns data to the host
 *     (ppo_runner_act, ppo_train_update with losses, ppo_core_sync ...)) or PPO_DEVICE
 *     (device pointers on the core's device; the call only enqueues work on the core's stream —
 *     use ppo_core_sync or your own event to wait).
 *   - all matrices are row-major fp32, shapes as in the reference (obs [n,O], actions [n,A], per-env
 *     scalars [n]).  Rollout buffers are exported in the reference's flat layout row = env*n_steps+t
 *     (ppo2/runner.hpp:136-152); internally they are time-major.
 *   - there is no CPU fallback: without a CUDA device ppo_core_create fails with PPO_ERR_CUDA.
 */
#ifndef PPO_CORE_H
#define PPO_CORE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PPO_CORE_ABI_VERSION 1

typedef enum {
    PPO_OK = 0,
    PPO_ERR_INVALID = -1,     /* bad argument / shape mismatch (the reference would assert) */
    PPO_ERR_CUDA = -2,        /* CUDA runtime error or no device */
    PPO_ERR_IO = -3,          /* file missing / unparsable */
    PPO_ERR_UNSUPPORTED = -4, /* configuration outside what the kernels cover */
    PPO_ERR_COMM = -5         /* NCCL error */
} ppo_status;

typedef enum { PPO_HOST = 0, PPO_DEVICE = 1 } ppo_mem;

typedef struct ppo_core ppo_core; /* opaque */

/* Everything PPO2's constructor + EnvNormalize's constructor take (ppo2/ppo2.hpp:33-47,
 * env/env_normalize.hpp:20-28) plus what the reference reads from the graph file (SURVEY §3.5:
 * ent_coef, vf_coef, max_grad_norm and Adam's constants are baked into the .meta.txt). */
typedef struct {
    int abi_version; /* PPO_CORE_ABI_VERSION */
    int device;      /* CUDA ordinal */
    int obs_dim, act_dim;   /* 1..64 each.  Reference envs: 18/18 closed loop (36/18 with velocities), 1/18 open loop */
    int hidden1, hidden2;   /* MLP [h1,h2] for both towers; overwritten by ppo_core_load_meta_txt */
    int n_envs;             /* envs owned by THIS rank */
    int n_steps;            /* --batch_steps: steps per env per update (ppo2.cpp:114) */
    int nminibatches;       /* 32 (ppo2.cpp:216) */
    int noptepochs;         /* --num_epochs */
    float gamma, lam;       /* 0.99, 0.95 (ppo2.cpp:216) */
    float ent_coef, vf_coef, max_grad_norm;          /* graph constants */
    float adam_beta1, adam_beta2, adam_epsilon;      /* graph constants */
    /* VecNormalize */
    int norm_obs, norm_reward, training;
    float clip_obs, clip_reward, norm_gamma, norm_epsilon;
    /* RNG: Philox4x32-10 key for action noise (and, xor 0x1234, the synthetic env) */
    uint64_t seed;
    /* sharding: this rank owns global envs [env_offset, env_offset + n_envs) of n_envs_global */
    int rank, world_size;
    int env_offset, n_envs_global;
} ppo_core_desc;

const char *ppo_last_error(void);
int ppo_abi_version(void);
/* fills the reference's defaults (ppo2.cpp:215-217, env_normalize.hpp:20-28, graph constants of the shipped graph) */
int ppo_core_desc_default(ppo_core_desc *desc);

/* ---- graph file (replaces SessionCreator::load_graph, ppo2/session_creator.hpp:23-57) ---- */
typedef struct {
    int obs_dim, act_dim, hidden1, hidden2;
    float ent_coef, vf_coef, max_grad_norm, adam_beta1, adam_beta2, adam_epsilon;
    int n_params_trainable, n_params_total; /* 13 tensors / 15 tensors (with the unused q head) */
} ppo_meta_info;
/* Parse a TF-1.14 text MetaGraphDef: shapes, baked constants.  params_out (may be NULL) receives the
 * n_params_total initial values in core order (see ppo_core_tensor_name). */
int ppo_meta_parse(const char *meta_txt_path, ppo_meta_info *info, float *params_out, size_t params_capacity);

/* Value-function loss of Stable-Baselines' PPO2 (SURVEY §3.5), fixed by `cliprange_vf` when the graph was exported:
 *   SHARED    vc = old_v + clip(v - old_v, -cliprange, cliprange)        (cliprange_vf None: the shipped graph)
 *   NONE      vc = v, no clipping                                         (cliprange_vf < 0: the original PPO loss)
 *   SEPARATE  vc = old_v + clip(v - old_v, -cliprange_vf, cliprange_vf)   (cliprange_vf >= 0: placeholder loss/clip_range_vf_ph)
 * vf_loss = 0.5 * mean(max((v - R)^2, (vc - R)^2)) in every mode. */
typedef enum { PPO_VF_CLIP_SHARED = 0, PPO_VF_CLIP_NONE = 1, PPO_VF_CLIP_SEPARATE = 2 } ppo_vf_clip;
/* the ppo_vf_clip of a graph file, read from the data flow of its loss sub-graph (a file without one, as written by
 * meta_graph.write_meta_txt without vf_clip, is SHARED); PPO_ERR_UNSUPPORTED if the value loss is of no known form */
int ppo_meta_vf_clip(const char *meta_txt_path);

/* Hidden-layer activation of the MLP (Stable-Baselines' policy_kwargs act_fun: tf.tanh, the default, or tf.nn.relu), the
 * same for both hidden layers of both towers.  ReLU's gradient is TensorFlow's ReluGrad: a unit whose pre-activation is
 * exactly 0 gets none. */
typedef enum { PPO_ACT_TANH = 0, PPO_ACT_RELU = 1 } ppo_activation;
/* the ppo_activation of a graph file, read from the data flow into each layer that reads a hidden layer (a file without
 * forward nodes, as written by meta_graph.write_meta_txt without activation, is TANH); PPO_ERR_UNSUPPORTED for any other
 * activation, mixed activations, or a deeper / shared-trunk net_arch.  ppo_meta_parse fails the same way. */
int ppo_meta_activation(const char *meta_txt_path);

/* Action space of the policy head (Stable-Baselines' probability distribution of the env's action space):
 *   BOX       DiagGaussianProbabilityDistribution: mean = model/pi, std = exp(model/pi/logstd); actions are act_dim floats
 *   DISCRETE  CategoricalProbabilityDistribution over act_dim = n logits (model/pi, no logstd): an action is ONE index
 *             0 .. n-1, stored as fp32 wherever actions are passed (action width 1); it is sampled as
 *             argmax_j (l_j - log(-log(u_j))) with u uniform in [0, 1), and ppo_policy_step's eps holds those n uniforms per env.
 *   MULTI_DISCRETE  MultiCategoricalProbabilityDistribution: k categoricals side by side over slices of act_dim = sum(nvec)
 *             logits (nvec[i] logits each, in order); an action is k indices (action width k, column i in 0 .. nvec[i]-1),
 *             each sampled as DISCRETE samples its slice from the uniforms of the flat logit index, so MultiDiscrete([n]) draws
 *             what Discrete(n) draws; neglogp and entropy are the sums over the slices.
 *   MULTI_BINARY    BernoulliProbabilityDistribution over act_dim = n logits: an action is n columns of 0 / 1, sampled as
 *             [u_j < sigmoid(l_j)] (eps: n uniforms per env); neglogp = sum_j sigmoid_cross_entropy_with_logits(l_j, x_j),
 *             entropy = sum_j sigmoid_cross_entropy_with_logits(l_j, sigmoid(l_j)) with its gradient through sigmoid(l_j);
 *             the deterministic action is round(sigmoid(l)) with ties to even (l = 0 gives 0).
 *             An action column outside its choices (or not an integer) is PPO_ERR_INVALID in ppo_rollout_set and ppo_loss_grad.
 *             Every head but BOX has no logstd: ppo_meta_parse counts 14 tensors; checkpoints hold them in sorted-name order.
 *             The S / U / W kernel families, the persistent rollout and the synthetic env are continuous-only: a core with
 *             another head runs the F or T family, and the synthetic-env entry points return PPO_ERR_UNSUPPORTED. */
typedef enum { PPO_ACTION_BOX = 0, PPO_ACTION_DISCRETE = 1, PPO_ACTION_MULTI_DISCRETE = 2, PPO_ACTION_MULTI_BINARY = 3 } ppo_action_space;
/* the ppo_action_space of a graph file: BOX with model/pi/logstd; without it DISCRETE, unless PPO2's placeholder loss/action_ph is
 * int32 / int64 [?, k]: then MULTI_DISCRETE when a SplitV under model/ reads the pi head's output (the Add / BiasAdd over
 * model/pi/b) with k size_splits summing to the pi width; without such a SplitV, MULTI_BINARY when a Sigmoid under model/ reads the
 * pi head's output (Bernoulli's tf.sigmoid of the logits) and k is the pi width.  An int [?, k] placeholder with neither op is
 * refused, so a Discrete graph with a rank-2 placeholder is not read as MultiBinary.  When the file has loss/action_ph it must
 * agree (float [?, n] for BOX, int32 / int64 [?] for DISCRETE), otherwise PPO_ERR_UNSUPPORTED naming the node; ppo_meta_parse
 * fails the same way. */
int ppo_meta_action_space(const char *meta_txt_path);
/* the choices per action column of a graph file's head: {n} (DISCRETE), nvec (MULTI_DISCRETE), 2s (MULTI_BINARY); returns the
 * action width (nvec may be NULL to ask for it alone) or a negative ppo_status: PPO_ERR_INVALID for BOX or a capacity below the width */
int ppo_meta_action_nvec(const char *meta_txt_path, int *nvec, int capacity);

int ppo_core_create(const ppo_core_desc *desc, ppo_core **out); /* ppo_core_create_ex(desc, PPO_ACTION_BOX, out) */
/* a core whose policy head is of the given ppo_action_space (fixed for the core's lifetime); MULTI_DISCRETE is PPO_ERR_INVALID
 * here (it needs an nvec: ppo_core_create_nvec) */
int ppo_core_create_ex(const ppo_core_desc *desc, int action_space, ppo_core **out);
/* a MULTI_DISCRETE core with k action columns of nvec[i] >= 1 choices: sum(nvec) == desc->act_dim <= 64, k <= 64 */
int ppo_core_create_nvec(const ppo_core_desc *desc, const int *nvec, int k, ppo_core **out);
int ppo_core_action_space(ppo_core *core); /* the core's ppo_action_space, or a negative ppo_status */
/* the core's choices per action column, as ppo_meta_action_nvec; returns the action width */
int ppo_core_action_nvec(ppo_core *core, int *nvec, int capacity);
/* Invalid-action masks (sb3-contrib's MaskableCategorical), DISCRETE and MULTI_DISCRETE cores only: ppo_core_set_action_masking on
 * a BOX or MULTI_BINARY core is PPO_ERR_UNSUPPORTED.  Off at create; must be the same on every rank.  Turning it on allocates the
 * "action_masks" rollout buffer (every row all allowed) and, on or off, drops the captured CUDA graphs.
 *   A mask is const uint8_t [n][act_dim]: per row one entry per logit in logit order (act_dim for DISCRETE, sum(nvec) for
 *   MULTI_DISCRETE), 1 allowed, 0 forbidden; any other value is PPO_ERR_INVALID, as is a categorical (the row, or a slice) that
 *   allows nothing.  Internally a row is one 64-bit word (bit j = logit j allowed), 8 bytes per transition.
 *   Over the allowed logits S of each categorical: the sample is argmax_{j in S} (l_j - log(-log u_j)) with the unmasked head's
 *   uniforms (forbidden indices skipped, ties to the first index), so all-allowed draws what the unmasked head draws; neglogp =
 *   log z_S - (l_a - m_S) with m_S = max_S l, z_S = sum_S exp(l - m_S) (summed over the slices); entropy = sum_S p (log z_S - (l - m_S));
 *   dL/dl_j is exactly 0 for a forbidden j; the deterministic action is argmax_S l.  The value loss, clip and Adam are unchanged.
 *   These equal sb3-contrib's results with -1e8 in the forbidden logits.
 *   The plain entry points (ppo_policy_step, ppo_runner_reset / act / observe, ppo_rollout_set of "actions", ppo_loss_grad ...)
 *   allow every action of the rows they touch; the _masked ones fail with PPO_ERR_INVALID while masking is off.
 *   A mask in device memory (PPO_DEVICE) is checked on the device: its first bad row (every logit then allowed for it) is reported
 *   as PPO_ERR_INVALID by the next ppo_runner_finish, ppo_train_update*, ppo_train_minibatch* or ppo_core_sync of the core.  With
 *   more than one rank, ppo_train_update* and ppo_train_minibatch* first sum every rank's count of bad masks (one ncclAllReduce of
 *   one float per call, on masking cores only), so a bad mask on one rank fails the call on every rank before any collective of it.
 *   ppo_runner_rollout_host / _replay take no masks: PPO_ERR_UNSUPPORTED on a masking core. */
int ppo_core_set_action_masking(ppo_core *core, int enable);
int ppo_core_action_masking(ppo_core *core); /* 1 on, 0 off, or a negative ppo_status */
void ppo_core_destroy(ppo_core *core);
/* load initial weights from the graph file; its shapes and its ppo_action_space (and nvec) must match the core's (ppo2.hpp:90-105 reset());
 * sets the core's ppo_vf_clip and ppo_activation */
int ppo_core_load_meta_txt(ppo_core *core, const char *meta_txt_path);
/* the value loss of a graph-less core (default SHARED); ppo_core_load_meta_txt sets it from the graph */
int ppo_core_set_vf_clip(ppo_core *core, int mode);
int ppo_core_vf_clip(ppo_core *core); /* the core's ppo_vf_clip, or a negative ppo_status */
/* the hidden-layer activation of a graph-less core (default TANH); ppo_core_load_meta_txt sets it from the graph.  A change
 * drops the captured CUDA graphs (they are re-captured on their next use). */
int ppo_core_set_activation(ppo_core *core, int act);
int ppo_core_activation(ppo_core *core); /* the core's ppo_activation, or a negative ppo_status */
/* Stable-Baselines' orthogonal init for graph-less configs (synthetic benchmarks with [64,64], [256,256]) */
int ppo_core_init_orthogonal(ppo_core *core, uint64_t seed);
/* TF Saver V2 bundle written by PPO2::save (ppo2.hpp:107-131): `<prefix>.data-00000-of-00001` holds the 15
 * model tensors as raw fp32 in sorted-name order.  load() restores weights only — Adam restarts (ppo2.hpp:169-223). */
int ppo_core_load_checkpoint_data(ppo_core *core, const char *prefix);
/* writes `<prefix>.data-00000-of-00001` and `<prefix>.index` (the bundle's table of name -> dtype / shape / offset / size / crc32c),
 * so the reference's PPO2::load (ppo2.hpp:169-189, `save/restore_all`) and TensorFlow read the checkpoint back */
int ppo_core_save_checkpoint_data(ppo_core *core, const char *prefix);
/* the `.index` alone, for a `.data` payload held by the caller (the 15 tensors of an MLP [hidden1, hidden2] policy in ascending name
 * order, n_floats values); no device needed.  Byte-identical to TensorFlow 1.14's BundleWriter on the reference's shipped checkpoint. */
int ppo_checkpoint_write_index(const char *prefix, int obs_dim, int act_dim, int hidden1, int hidden2, const float *data, size_t n_floats);
/* ... for either layout: PPO_ACTION_DISCRETE leaves model/pi/logstd out (14 tensors), the layout of every head but BOX, which
 * ppo_core_save_checkpoint_data writes for MULTI_DISCRETE and MULTI_BINARY cores too; other values are PPO_ERR_INVALID */
int ppo_checkpoint_write_index_ex(const char *prefix, int action_space, int obs_dim, int act_dim, int hidden1, int hidden2,
                                  const float *data, size_t n_floats);

/* tensors by TF variable name: "model/pi_fc0/w" ... "model/q/b"; Adam slots "<name>/Adam", "<name>/Adam_1";
 * "beta1_power", "beta2_power"; "params" = the whole flat vector (n_params_total). Host buffers. */
int ppo_core_num_tensors(void);
const char *ppo_core_tensor_name(int index);
int ppo_core_tensor_size(ppo_core *core, const char *name);
int ppo_core_get_tensor(ppo_core *core, const char *name, float *out, size_t capacity);
int ppo_core_set_tensor(ppo_core *core, const char *name, const float *in, size_t count);
int ppo_core_sync(ppo_core *core);
/* the core's CUDA stream (cudaStream_t) for callers that enqueue their own device work */
void *ppo_core_stream(ppo_core *core);

/* ---- policy (MlpPolicy::step/value/get_deterministic_action, ppo2/policies.hpp:33-77) ---- */
/* eps: [n,A] standard-normal noise to use (parity tests) or NULL to draw Philox noise for
 * (seed, env_offset+i, internal step counter).  Outputs may be NULL. */
int ppo_policy_step(ppo_core *core, const float *obs, int n, const float *eps, float *action, float *value,
                    float *neglogp, ppo_mem mem);
int ppo_policy_value(ppo_core *core, const float *obs, int n, float *value, ppo_mem mem);
int ppo_policy_mean(ppo_core *core, const float *obs, int n, float *action, ppo_mem mem); /* PPO2::eval, ppo2.hpp:225-237 */
/* ... over the actions mask [n][act_dim] allows (see ppo_core_set_action_masking); mask lives where `mem` says */
int ppo_policy_step_masked(ppo_core *core, const float *obs, int n, const float *eps, const uint8_t *mask, float *action, float *value,
                           float *neglogp, ppo_mem mem);
int ppo_policy_mean_masked(ppo_core *core, const float *obs, int n, const uint8_t *mask, float *action, ppo_mem mem);

/* ---- VecNormalize (EnvNormalize, env/env_normalize.hpp:64-116) on the core's running statistics ---- */
int ppo_vecnorm_reset(ppo_core *core, const float *raw_obs, float *obs_out, ppo_mem mem);
int ppo_vecnorm_step(ppo_core *core, const float *raw_obs, const float *raw_rew, const float *done, float *obs_out,
                     float *rew_out, ppo_mem mem);
/* The same as n_steps consecutive ppo_vecnorm_step calls on a recorded trajectory (raw_obs [n_steps][n_envs][O],
 * raw_rew / done [n_steps][n_envs]; env/env_normalize.hpp:64-92 applied step by step, running statistics and the
 * discounted return carried on), evaluated as four HBM-bound launches.  rew_out may be NULL.  Single rank only. */
int ppo_vecnorm_replay(ppo_core *core, const float *raw_obs, const float *raw_rew, const float *done, int n_steps,
                       float *obs_out, float *rew_out, ppo_mem mem);
/* obs_rms / ret_rms as serialised by RunningStatistics (common/running_statistics.hpp:57-86) */
int ppo_vecnorm_get_stats(ppo_core *core, float *obs_mean, float *obs_var, double *obs_count, float *ret_mean,
                          float *ret_var, double *ret_count);
int ppo_vecnorm_set_stats(ppo_core *core, const float *obs_mean, const float *obs_var, double obs_count,
                          const float *ret_mean, const float *ret_var, double ret_count);
int ppo_vecnorm_set_training(ppo_core *core, int training);
/* stateless pieces (RunningStatistics::update, running_statistics.hpp:26-35; MatrixClamp::clamp, matrix_clamp.hpp:32-35);
 * mean/var/count are host state owned by the caller */
int ppo_running_stats_update(ppo_core *core, float *mean, float *var, double *count, int dim, const float *batch,
                             int rows, ppo_mem batch_mem);
int ppo_matrix_clamp(ppo_core *core, const float *x, size_t n, float lo, float hi, float *out, ppo_mem mem);

/* ---- GAE (Runner::set_returns, ppo2/runner.hpp:159-191); time-major [n_steps,n_envs] ---- */
int ppo_gae(ppo_core *core, const float *rewards, const float *values, const float *dones, const float *last_values,
            const float *last_dones, int n_steps, int n_envs, float gamma, float lam, float *advs, float *returns,
            ppo_mem mem);

/* ---- rollout (Runner::run, ppo2/runner.hpp:56-157) ---- */
/* host-env protocol, one call pair per env step:
 *   ppo_runner_reset(raw_obs0)                      Runner ctor: obs = env.reset() through EnvNormalize::reset
 *   for t in 0..n_steps-1:
 *       ppo_runner_act(t, actions_out)              store obs/dones, policy step, store action/value/neglogp
 *       ppo_runner_observe(t, raw_obs, raw_rew, done)   EnvNormalize::step post-processing, store rewards
 *   ppo_runner_finish()                             bootstrap value + GAE */
int ppo_runner_reset(ppo_core *core, const float *raw_obs, ppo_mem mem);
int ppo_runner_act(ppo_core *core, int t, float *actions_out, ppo_mem mem);
int ppo_runner_observe(ppo_core *core, int t, const float *raw_obs, const float *raw_rew, const float *done, ppo_mem mem);
int ppo_runner_finish(ppo_core *core);
/* ... on a masking core: the mask [n_envs][act_dim] travels with the observation it belongs to; the next ppo_runner_act samples over
 * it and stores it at rollout row t (the mask after the last observe is that of the next rollout's step 0, as the observation is).
 * With PPO_HOST, ppo_runner_observe_masked copies the observation, reward, done and the mask's packed words through the core's
 * pinned staging buffer and returns without waiting for the copies (the caller's buffers may be reused at once). */
int ppo_runner_reset_masked(ppo_core *core, const float *raw_obs, const uint8_t *mask, ppo_mem mem);
int ppo_runner_observe_masked(ppo_core *core, int t, const float *raw_obs, const float *raw_rew, const float *done, const uint8_t *mask,
                              ppo_mem mem);
/* The same protocol as ONE call (the loop of Runner::run, ppo2/runner.hpp:75-129, in C): per env step the actions are
 * copied to `actions` (host, [n_envs][A]), `step` advances the host env and hands back pointers to its raw
 * observation / reward / done arrays (host, valid until the next call), which are copied to the device and
 * normalised; then bootstrap value + GAE.  `step` returns 0 to continue, anything else aborts the rollout.
 * On one GPU the rollout runs as ONE persistent kernel that trades actions / observations with this loop once per env
 * step (flags in mapped pinned memory; up to 512 envs the env's answer is read by the kernel from mapped memory, beyond
 * that the observations go through the copy engine with a 4-byte flag copy behind them); `raw_obs` should be pinned
 * memory for the copy-engine path to be asynchronous. */
typedef int (*ppo_env_step_fn)(void *user, int t, const float *actions, const float **raw_obs, const float **raw_rew,
                               const float **done);
int ppo_runner_rollout_host(ppo_core *core, ppo_env_step_fn step, void *user, float *actions);
/* ... with a recorded trajectory as the env: raw_obs [n_steps][n_envs][O], raw_rew / done [n_steps][n_envs] (host);
 * actions_out [n_steps][n_envs][A] (host) receives the actions the policy took, or NULL; when it is pinned memory the kernel
 * stores the actions into it directly (PCIe writes), no staging copy */
int ppo_runner_rollout_replay(ppo_core *core, const float *raw_obs, const float *raw_rew, const float *done,
                              float *actions_out);
/* GPU-resident synthetic env (SURVEY §8d): whole rollout on the device, no host round trips */
int ppo_synth_env_reset(ppo_core *core);
int ppo_rollout_synthetic(ppo_core *core);
/* rollout buffers in the reference's flat layout: "obs","returns","dones","actions","values","neglogpacs",
 * "true_rewards","unnormalized_rewards" ([n_batch,18] or [n_batch]); host pointers.  A masking core adds "action_masks" as fp32
 * 0 / 1 [n_batch, act_dim]; setting it refuses a mask that forbids its row's recorded action (set the actions first: setting
 * "actions" makes those rows' masks all allowed) */
int ppo_rollout_get(ppo_core *core, const char *name, float *out, size_t capacity);
int ppo_rollout_set(ppo_core *core, const char *name, const float *in, size_t count);

/* ---- update (PPO2::learn epoch/minibatch loop + _train_step, ppo2/ppo2.hpp:264-335,380-471) ---- */
/* std::srand / std::random_shuffle restated bit-exactly (glibc TYPE_3 + libstdc++ stl_algo.h:4581) */
int ppo_shuffle_seed(ppo_core *core, unsigned seed);
int ppo_host_srand_rand(unsigned seed, int count, int *out);                       /* rand() stream */
int ppo_host_random_shuffle(unsigned seed, int n, int epochs, int *perms_out);     /* [epochs,n] compounded */
/* one whole update over the current rollout: noptepochs x nminibatches train steps with the
 * reference's permutation semantics; mean_losses[5] = pg, vf, entropy, approxkl, clipfrac (ppo2.hpp:335) */
int ppo_train_update(ppo_core *core, float lr, float cliprange, float *mean_losses);
/* ... with the value clip range of a SEPARATE graph (>= 0; ignored in the other modes).  The calls without _vf fail with
 * PPO_ERR_INVALID on a SEPARATE core, as TensorFlow does on the unfed loss/clip_range_vf_ph.  lr, cliprange and
 * cliprange_vf live in device memory, written on the core's stream before each call's work: the captured update graphs
 * are replayed, not rebuilt, when they change from update to update (schedules, ppo2.hpp:264-335) */
int ppo_train_update_vf(ppo_core *core, float lr, float cliprange, float cliprange_vf, float *mean_losses);
/* finer grain for parity tests: set this epoch's permutation (perm.indices, n_batch ints) and run minibatch k;
 * losses[5] of that step; grads (may be NULL) = the unclipped gradient, n_params_trainable floats */
int ppo_train_set_permutation(ppo_core *core, const int *perm, int n);
/* perm.indices of epoch `epoch` of the LAST ppo_train_update (n_batch ints, compounded over the epochs as in
 * ppo2.hpp:274-288) — lets a test compare the device-built permutations with std::random_shuffle bit for bit.
 * Valid until the next rollout starts: the permutations of the NEXT update are then built beside the rollout
 * (they depend on the rand() stream only) and this call returns PPO_ERR_INVALID. */
int ppo_train_get_permutation(ppo_core *core, int epoch, int *out, int n);
int ppo_train_minibatch(ppo_core *core, int k, float lr, float cliprange, float *losses, float *grads);
int ppo_train_minibatch_vf(ppo_core *core, int k, float lr, float cliprange, float cliprange_vf, float *losses, float *grads);
/* standalone pieces on caller data (host pointers): advantage normalisation (ppo2.hpp:401-406) and loss+grad */
int ppo_advnorm(ppo_core *core, const float *returns, const float *values, int n, float *advs);
int ppo_loss_grad(ppo_core *core, const float *obs, const float *actions, const float *advs, const float *returns,
                  const float *old_neglogp, const float *old_values, int B, float cliprange, float *grads, float *losses);
int ppo_loss_grad_vf(ppo_core *core, const float *obs, const float *actions, const float *advs, const float *returns,
                     const float *old_neglogp, const float *old_values, int B, float cliprange, float cliprange_vf, float *grads,
                     float *losses);
/* ... with masks [B][act_dim] on a masking core (host pointers): the loss over the allowed actions; a recorded action its mask
 * forbids is PPO_ERR_INVALID.  cliprange_vf is read only in SEPARATE mode. */
int ppo_loss_grad_masked(ppo_core *core, const float *obs, const float *actions, const uint8_t *masks, const float *advs,
                         const float *returns, const float *old_neglogp, const float *old_values, int B, float cliprange,
                         float cliprange_vf, float *grads, float *losses);
/* rollout + update on the synthetic env; env-steps/s accounting is the caller's (ppo2.hpp:337-341) */
int ppo_learn_update_synthetic(ppo_core *core, float lr, float cliprange, float *mean_losses);

/* ---- multi-GPU (no counterpart in the reference; SURVEY §8e) ---- */
#define PPO_COMM_ID_BYTES 128
int ppo_comm_get_unique_id(char id[PPO_COMM_ID_BYTES]);
int ppo_comm_init(ppo_core *core, const char id[PPO_COMM_ID_BYTES], int rank, int world_size);
/* Peer-memory mailboxes (one process per GPU, one NVLink/NVSwitch node): every rank exports the cudaIpc handle of its
 * mailbox, the host gathers the world_size handles (rank order) and every rank maps them.  Once mapped, the
 * per-env-step VecNormalize moment exchange and the per-minibatch gradient allreduce run INSIDE the persistent rollout
 * kernel / the cooperative reduce+Adam kernel as NVLink P2P stores + flags (no NCCL call on those paths; NCCL remains
 * for the once-per-update allgather of the rollout buffers).  Without this call the NCCL path is used. */
#define PPO_IPC_HANDLE_BYTES 64
int ppo_comm_ipc_handle(ppo_core *core, char out[PPO_IPC_HANDLE_BYTES]);
int ppo_comm_ipc_open(ppo_core *core, const char *handles /* [world_size][PPO_IPC_HANDLE_BYTES] */, int world_size);
/* switch the mailbox path off (NCCL for every exchange) or back on; must be the same on every rank */
int ppo_comm_set_p2p(ppo_core *core, int enable);
/* 1 if a mailbox wait timed out (a peer never arrived); 0 otherwise */
int ppo_comm_error(ppo_core *core);

/* ---- introspection for the bench: kernels launched / device time of the dominant kernel ---- */
typedef struct {
    uint64_t kernel_launches; /* since create or last reset */
    uint64_t graph_launches;
    uint64_t h2d_bytes, d2h_bytes;
} ppo_counters;
int ppo_core_counters(ppo_core *core, ppo_counters *out, int reset);
/* CUDA graphs captured and instantiated since create (rollout, permutations, update / epochs) */
int ppo_core_graph_builds(ppo_core *core, uint64_t *out);
/* which kernel family the core selected for this MLP shape: "which" = "train" | "policy";
 * returns e.g. "train_umma_kernel (tcgen05, bf16x3 split)", "train_fused_kernel (fp32 FFMA, weights in smem)",
 * "train_tile_kernel (fp32 FFMA, generic)"; NULL on bad arguments */
const char *ppo_core_kernel_family(ppo_core *core, const char *which);
/* average device time (ms, CUDA events on the core's stream) of `iters` back-to-back launches of one kernel of
 * the path on the core's current rollout buffers: "train_fwdbwd" (rotating over the minibatches of the current
 * permutation), "grad_reduce", "adam" (lr = 0: weights unchanged), "policy_step", "norm_moments", "norm_apply",
 * "gae", "synth_env".  Used by bench.py for the roofline object; launches counts the kernel launches timed. */
int ppo_profile_kernel(ppo_core *core, const char *which, int iters, float *avg_ms, int *launches);

#ifdef __cplusplus
}
#endif
#endif /* PPO_CORE_H */
