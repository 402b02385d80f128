// Minimal reader for TensorFlow-1.14 text-proto MetaGraphDef files (.meta.txt).
// Replaces SessionCreator::load_graph (reference ppo2/session_creator.hpp:23-57): the graph is read,
// never executed.  Extracts variable shapes, initial values, the constants the graph bakes in and which value loss
// the graph builds and the hidden-layer activation of its forward pass.
#pragma once
#include <map>
#include <string>
#include <vector>

namespace ppo {

struct MetaTensor {
    std::vector<int> shape;
    std::vector<float> data;
};

struct MetaGraph {
    int obs_dim = 0, act_dim = 0, hidden1 = 0, hidden2 = 0;
    float ent_coef = 0, vf_coef = 0, clip_norm = 0, beta1 = 0, beta2 = 0, adam_eps = 0;
    // value loss of the graph (ppo_vf_clip: 0 shared clip range, 1 no clipping, 2 own range loss/clip_range_vf_ph), or -1
    // when the loss sub-graph is there but matches none of them (vf_clip_error says why)
    int vf_clip = 0;
    std::string vf_clip_error;
    // hidden-layer activation (ppo_activation: 0 tanh, 1 relu), or -1 when the forward pass is not two tanh or two relu
    // hidden layers per tower (activation_error says why)
    int activation = 0;
    std::string activation_error;
    // action space of the policy head (ppo_action_space: 0 Box, a Gaussian with model/pi/logstd; without it 1 Discrete,
    // 2 MultiDiscrete, 3 MultiBinary), or -1 when loss/action_ph contradicts the head (action_space_error says why)
    int action_space = 0;
    std::string action_space_error;
    std::vector<int> nvec;  // MultiDiscrete: the choices per action column (size_splits of the SplitV)
    std::map<std::string, MetaTensor> tensors;  // the model/* variables with their initial values (14 without logstd)
};

// Returns empty string on success, otherwise the error message.
std::string parse_meta_txt(const std::string& path, MetaGraph& out);

// Tensor order of the core's flat parameter vector: the graph's gradient order
// (GRAPH:23738-24074) followed by the untrained q head.
extern const char* const kTensorNames[15];
constexpr int kNumTrainableTensors = 13;
constexpr int kNumTensors = 15;
constexpr int kLogstdTensor = 12;  // "model/pi/logstd": absent in a graph with a categorical head

}  // namespace ppo
