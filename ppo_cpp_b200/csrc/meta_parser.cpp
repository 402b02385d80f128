// See meta_parser.h.  A ~150-line recursive-descent reader for protobuf text format, enough for
// MetaGraphDef: nested messages, string literals with C escapes, numbers and enum identifiers.
#include "meta_parser.h"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <memory>
#include <sstream>

namespace ppo {

const char* const kTensorNames[15] = {
    "model/pi_fc0/w", "model/pi_fc0/b", "model/vf_fc0/w", "model/vf_fc0/b", "model/pi_fc1/w",
    "model/pi_fc1/b", "model/vf_fc1/w", "model/vf_fc1/b", "model/vf/w",     "model/vf/b",
    "model/pi/w",     "model/pi/b",     "model/pi/logstd", "model/q/w",     "model/q/b"};

namespace {

struct Msg;
struct Field {
    std::string key;
    std::string scalar;         // string bytes / number / identifier
    std::unique_ptr<Msg> msg;   // non-null for nested messages
};
struct Msg {
    std::vector<Field> fields;
    const Field* find(const char* key) const {
        for (const auto& f : fields)
            if (f.key == key) return &f;
        return nullptr;
    }
    const Msg* sub(const char* key) const {
        const Field* f = find(key);
        return f && f->msg ? f->msg.get() : nullptr;
    }
    std::string str(const char* key) const {
        const Field* f = find(key);
        return f ? f->scalar : std::string();
    }
};

struct Parser {
    const char* p;
    const char* end;
    std::string err;

    void skip_ws() {
        while (p < end) {
            if (*p == '#') {
                while (p < end && *p != '\n') ++p;
            } else if (*p == ' ' || *p == '\n' || *p == '\t' || *p == '\r') {
                ++p;
            } else {
                break;
            }
        }
    }
    bool parse_string(std::string& out) {
        ++p;  // opening quote
        while (p < end && *p != '"') {
            if (*p != '\\') {
                out.push_back(*p++);
                continue;
            }
            ++p;
            if (p >= end) return false;
            char c = *p;
            if (c >= '0' && c <= '7') {
                int v = 0, n = 0;
                while (p < end && n < 3 && *p >= '0' && *p <= '7') {
                    v = v * 8 + (*p - '0');
                    ++p;
                    ++n;
                }
                out.push_back(static_cast<char>(v & 0xFF));
                continue;
            }
            ++p;
            switch (c) {
                case 'n': out.push_back('\n'); break;
                case 't': out.push_back('\t'); break;
                case 'r': out.push_back('\r'); break;
                case 'a': out.push_back('\a'); break;
                case 'b': out.push_back('\b'); break;
                case 'f': out.push_back('\f'); break;
                case 'v': out.push_back('\v'); break;
                case 'x': {
                    int v = 0, n = 0;
                    while (p < end && n < 2 && isxdigit(static_cast<unsigned char>(*p))) {
                        char h = *p++;
                        v = v * 16 + (h <= '9' ? h - '0' : (h | 32) - 'a' + 10);
                        ++n;
                    }
                    out.push_back(static_cast<char>(v));
                    break;
                }
                default: out.push_back(c); break;  // \" \' \\ ...
            }
        }
        if (p >= end) return false;
        ++p;  // closing quote
        return true;
    }
    bool parse_msg(Msg& m, bool top) {
        for (;;) {
            skip_ws();
            if (p >= end) return top;
            if (*p == '}') {
                ++p;
                return !top;
            }
            const char* k0 = p;
            while (p < end && (isalnum(static_cast<unsigned char>(*p)) || *p == '_')) ++p;
            if (p == k0) {
                err = "text-proto: field name expected";
                return false;
            }
            Field f;
            f.key.assign(k0, p);
            skip_ws();
            if (p < end && *p == ':') {
                ++p;
                skip_ws();
            }
            if (p >= end) return false;
            if (*p == '{') {
                ++p;
                f.msg.reset(new Msg());
                if (!parse_msg(*f.msg, false)) return false;
            } else if (*p == '"') {
                if (!parse_string(f.scalar)) {
                    err = "text-proto: unterminated string";
                    return false;
                }
            } else {
                const char* v0 = p;
                while (p < end && !isspace(static_cast<unsigned char>(*p)) && *p != '}') ++p;
                f.scalar.assign(v0, p);
            }
            m.fields.push_back(std::move(f));
        }
    }
};

const Msg* attr_value(const Msg& node, const char* key) {
    for (const auto& f : node.fields) {
        if (f.key != "attr" || !f.msg) continue;
        if (f.msg->str("key") == key) return f.msg->sub("value");
    }
    return nullptr;
}

std::vector<int> shape_dims(const Msg* shape) {
    std::vector<int> d;
    if (!shape) return d;
    for (const auto& f : shape->fields)
        if (f.key == "dim" && f.msg) d.push_back(std::atoi(f.msg->str("size").c_str()));
    return d;
}

bool const_tensor(const Msg& node, MetaTensor& t) {
    const Msg* v = attr_value(node, "value");
    const Msg* ten = v ? v->sub("tensor") : nullptr;
    if (!ten) return false;
    t.shape = shape_dims(ten->sub("tensor_shape"));
    size_t count = 1;
    for (int d : t.shape) count *= static_cast<size_t>(d);
    const Field* content = ten->find("tensor_content");
    if (content) {
        if (content->scalar.size() != count * 4) return false;
        t.data.resize(count);
        std::memcpy(t.data.data(), content->scalar.data(), count * 4);  // little-endian fp32
        return true;
    }
    std::vector<float> vals;
    for (const auto& f : ten->fields)
        if (f.key == "float_val") vals.push_back(std::strtof(f.scalar.c_str(), nullptr));
    if (vals.empty()) {
        t.data.assign(count, 0.f);  // all-zero tensors carry no value field
    } else if (vals.size() == 1) {
        t.data.assign(count, vals[0]);
    } else {
        if (vals.size() != count) return false;
        t.data = vals;
    }
    return true;
}

using NodeMap = std::map<std::string, const Msg*>;

// data inputs of a node ("name:0" -> "name"; control inputs "^name" skipped)
std::vector<std::string> node_inputs(const Msg& node) {
    std::vector<std::string> in;
    for (const auto& f : node.fields) {
        if (f.key != "input" || f.scalar.empty() || f.scalar[0] == '^') continue;
        const size_t colon = f.scalar.find(':');
        in.push_back(colon == std::string::npos ? f.scalar : f.scalar.substr(0, colon));
    }
    return in;
}

// Stable-Baselines' PPO2 builds vf_loss = 0.5 * mean(max(square(vpred - R), square(vpred_clipped - R))) with
//   vpred_clipped = vpred                                                      (cliprange_vf < 0: no clipping)
//   vpred_clipped = old_vpred_ph + clip_by_value(vpred - old_vpred_ph, -b, b)  (b = loss/clip_range_ph or loss/clip_range_vf_ph)
// Classified by following the data flow from the second operand of loss/Maximum back through its Square and Sub.
int classify_vf_clip(const NodeMap& nodes, std::string& err) {
    auto node = [&](const std::string& name, const char* op) -> const Msg* {
        auto it = nodes.find(name);
        return it != nodes.end() && it->second->str("op") == op ? it->second : nullptr;
    };
    auto sub_of_square = [&](const std::string& sq, std::vector<std::string>& ins) -> bool {
        const Msg* s = node(sq, "Square");
        if (!s || node_inputs(*s).size() != 1) return false;
        const Msg* d = node(node_inputs(*s)[0], "Sub");
        if (!d) return false;
        ins = node_inputs(*d);
        return ins.size() == 2;
    };
    if (nodes.find("loss/Maximum") == nodes.end()) return 0;  // no loss sub-graph (files of write_meta_txt): the shipped graph's form
    const Msg* mx = node("loss/Maximum", "Maximum");
    const std::vector<std::string> mi = mx ? node_inputs(*mx) : std::vector<std::string>();
    std::vector<std::string> s1, s2;
    if (mi.size() != 2 || !sub_of_square(mi[0], s1) || !sub_of_square(mi[1], s2) || s1[1] != s2[1]) {
        err = "loss/Maximum is not max(square(vpred - R), square(vpred_clipped - R))";
        return -1;
    }
    if (s2[0] == s1[0]) return 1;  // vpred_clipped is vpred itself
    const Msg* add = node(s2[0], "Add");
    std::vector<std::string> ai = add ? node_inputs(*add) : std::vector<std::string>();
    if (ai.size() == 2 && ai[1] == "loss/old_vpred_ph") std::swap(ai[0], ai[1]);
    const Msg* clip = ai.size() == 2 && ai[0] == "loss/old_vpred_ph" ? node(ai[1], "Maximum") : nullptr;  // clip_by_value = max(min(x, b), -b)
    const std::vector<std::string> ci = clip ? node_inputs(*clip) : std::vector<std::string>();
    const Msg* mn = ci.size() == 2 ? node(ci[0], "Minimum") : nullptr;
    const Msg* neg = ci.size() == 2 ? node(ci[1], "Neg") : nullptr;
    const std::vector<std::string> ni = mn ? node_inputs(*mn) : std::vector<std::string>();
    const std::vector<std::string> gi = neg ? node_inputs(*neg) : std::vector<std::string>();
    if (ni.size() != 2 || gi.size() != 1 || ni[1] != gi[0]) {
        err = "the clipped value " + s2[0] + " is neither vpred nor old_vpred_ph + clip_by_value(..., -b, b)";
        return -1;
    }
    if (ni[1] == "loss/clip_range_ph") return 0;
    if (ni[1] == "loss/clip_range_vf_ph") return 2;
    err = "the value clip bound " + ni[1] + " is neither loss/clip_range_ph nor loss/clip_range_vf_ph";
    return -1;
}

// Stable-Baselines' MlpPolicy builds every hidden layer as act(matmul(x, w) + b) (policies.py mlp_extractor / a2c/utils.py
// linear), with act the policy's act_fun.  The activation is classified by following the data flow into the layer that reads
// it: for each (hidden layer L, reader N) pair, every forward MatMul (in the model/ or train_model/ scope, neither operand
// transposed) whose weight operand is the read of model/N/w must take a Tanh or Relu of Add(MatMul(., read of model/L/w),
// read of model/L/b), and every pair has such a reader in both scopes.  The gradient sub-graph's MatMuls (under
// loss/gradients/, dY * W^T with transpose_b, X^T * dY with transpose_a) also read the weights and are not readers.  Node
// names of the activations are not relied on (model/Tanh, model/Tanh_1, ... in construction order).  Returns ACT_TANH (0)
// or ACT_RELU (1); a file with no forward nodes (files of write_meta_txt) is tanh; -1 with err naming the node otherwise.
int classify_activation(const NodeMap& nodes, std::string& err) {
    for (const char* v : {"model/pi_fc2/w", "model/vf_fc2/w", "model/shared_fc0/w"})
        if (nodes.count(v)) {
            err = std::string("variable ") + v + ": only two hidden layers per tower, without a shared trunk, are supported";
            return -1;
        }
    auto op_of = [&](const std::string& name) -> std::string {
        auto it = nodes.find(name);
        return it == nodes.end() ? std::string() : it->second->str("op");
    };
    auto is_read_of = [&](const std::string& name, const std::string& var) -> bool {
        auto it = nodes.find(name);
        if (it == nodes.end() || it->second->str("op") != "Identity") return false;
        const std::vector<std::string> in = node_inputs(*it->second);
        return in.size() == 1 && in[0] == var;
    };
    auto attr_true = [](const Msg& node, const char* key) -> bool {
        const Msg* v = attr_value(node, key);
        return v && v->str("b") == "true";
    };
    // 0: model/, 1: train_model/, -1: neither or not a plain x * W product
    auto forward_scope = [&](const std::string& name, const Msg& node) -> int {
        if (node.str("op") != "MatMul" || attr_true(node, "transpose_a") || attr_true(node, "transpose_b")) return -1;
        if (name.compare(0, 6, "model/") == 0) return 0;
        if (name.compare(0, 12, "train_model/") == 0) return 1;
        return -1;
    };
    static const char* const kPairs[4][2] = {{"pi_fc0", "pi_fc1"}, {"pi_fc1", "pi"}, {"vf_fc0", "vf_fc1"}, {"vf_fc1", "vf"}};
    std::string first_op, first_node;
    int found = 0, per_scope[4][2] = {};
    for (int pi = 0; pi < 4; ++pi) {
        const std::string L = kPairs[pi][0], N = kPairs[pi][1];
        for (const auto& kv : nodes) {
            const Msg& mm = *kv.second;
            const int scope = forward_scope(kv.first, mm);
            if (scope < 0) continue;
            const std::vector<std::string> mi = node_inputs(mm);
            if (mi.size() != 2 || !is_read_of(mi[1], "model/" + N + "/w")) continue;
            ++found;
            ++per_scope[pi][scope];
            const std::string act = mi[0], aop = op_of(act);
            if (aop != "Tanh" && aop != "Relu") {
                err = "node " + kv.first + " reads " + act + " (op " + (aop.empty() ? std::string("missing") : aop) +
                      "), not a Tanh or Relu of layer " + L;
                return -1;
            }
            const std::vector<std::string> ai = node_inputs(*nodes.at(act));
            const std::string add = ai.size() == 1 ? ai[0] : std::string(), addop = op_of(add);
            std::vector<std::string> di;
            if (addop == "Add" || addop == "AddV2" || addop == "BiasAdd") di = node_inputs(*nodes.at(add));
            bool ok = false;
            for (int s = 0; s < 2 && di.size() == 2; ++s) {
                const std::string &m = di[s], &b = di[1 - s];
                if (op_of(m) != "MatMul" || forward_scope(m, *nodes.at(m)) < 0 || !is_read_of(b, "model/" + L + "/b")) continue;
                const std::vector<std::string> li = node_inputs(*nodes.at(m));
                ok = li.size() == 2 && is_read_of(li[1], "model/" + L + "/w");
            }
            if (!ok) {
                err = "activation node " + act + " (read by " + kv.first + ") is not act(matmul(x, model/" + L + "/w) + model/" + L + "/b)";
                return -1;
            }
            if (first_op.empty()) {
                first_op = aop;
                first_node = act;
            } else if (aop != first_op) {
                err = "the graph mixes activations: " + first_node + " is " + first_op + ", " + act + " is " + aop;
                return -1;
            }
        }
    }
    if (found == 0) return 0;
    for (int pi = 0; pi < 4; ++pi)
        for (int scope = 0; scope < 2; ++scope)
            if (per_scope[pi][scope] == 0) {
                err = std::string("no forward MatMul under ") + (scope ? "train_model/" : "model/") + " reads model/" + kPairs[pi][1] + "/w";
                return -1;
            }
    return first_op == "Relu" ? 1 : 0;
}

// Stable-Baselines' policy head follows the action space: a Box gets DiagGaussianProbabilityDistribution (model/pi/w, model/pi/b
// and model/pi/logstd), a Discrete(n) gets CategoricalProbabilityDistribution (n logits from model/pi/w, model/pi/b, no logstd).
// PPO2's action placeholder loss/action_ph (pdtype.sample_placeholder([None])), when the file has it, must agree: float [?, n]
// for Box, int32 / int64 [?] for Discrete.  Returns 0 (Box) or 1 (Discrete); -1 with err naming the node otherwise.
int classify_action_space(const NodeMap& nodes, int n, std::string& err) {
    const bool box = nodes.count("model/pi/logstd") != 0;
    auto it = nodes.find("loss/action_ph");
    if (it == nodes.end()) return box ? 0 : 1;
    const Msg* dt = attr_value(*it->second, "dtype");
    const std::string dtype = dt ? dt->str("type") : std::string();
    const Msg* shp = attr_value(*it->second, "shape");
    const std::vector<int> dims = shape_dims(shp ? shp->sub("shape") : nullptr);
    const bool ok = box ? (dtype == "DT_FLOAT" && dims.size() == 2 && dims[1] == n)
                        : ((dtype == "DT_INT32" || dtype == "DT_INT64") && dims.size() == 1);
    if (ok) return box ? 0 : 1;
    err = "node loss/action_ph (" + (dtype.empty() ? std::string("no dtype") : dtype) + ", rank " + std::to_string(dims.size()) + ") contradicts the " +
          (box ? "Gaussian head (model/pi/logstd present): a Box space needs a float [?, " + std::to_string(n) + "] placeholder"
               : "categorical head (no model/pi/logstd): a Discrete space needs an int32 / int64 [?] placeholder");
    return -1;
}

}  // namespace

std::string parse_meta_txt(const std::string& path, MetaGraph& out) {
    std::ifstream in(path, std::ios::binary);
    if (!in) return "cannot open graph file: " + path;
    std::stringstream ss;
    ss << in.rdbuf();
    const std::string text = ss.str();
    Parser ps{text.data(), text.data() + text.size(), {}};
    Msg root;
    if (!ps.parse_msg(root, true)) return "cannot parse " + path + ": " + (ps.err.empty() ? "unbalanced braces" : ps.err);
    const Msg* graph = root.sub("graph_def");
    if (!graph) return "no graph_def in " + path;
    NodeMap nodes;
    for (const auto& f : graph->fields)
        if (f.key == "node" && f.msg) nodes[f.msg->str("name")] = f.msg.get();
    out.vf_clip = classify_vf_clip(nodes, out.vf_clip_error);
    out.activation = classify_activation(nodes, out.activation_error);

    for (int i = 0; i < kNumTensors; ++i) {
        const std::string name = kTensorNames[i];
        auto it = nodes.find(name);
        if (i == kLogstdTensor && it == nodes.end()) continue;  // categorical head
        if (it == nodes.end() || it->second->str("op") != "VariableV2") return "graph has no variable " + name;
        const Msg* shp = attr_value(*it->second, "shape");
        MetaTensor t;
        std::vector<int> vshape = shape_dims(shp ? shp->sub("shape") : nullptr);
        bool found = false;
        for (const char* suffix : {"initial_value", "Const", "zeros"}) {
            auto init = nodes.find(name + "/Initializer/" + suffix);
            if (init != nodes.end() && init->second->str("op") == "Const") {
                if (!const_tensor(*init->second, t)) return "bad initializer for " + name;
                found = true;
                break;
            }
        }
        if (!found) return "no Const initializer for " + name;
        size_t count = 1;
        for (int d : vshape) count *= static_cast<size_t>(d);
        if (t.data.size() != count) return "initializer/variable size mismatch for " + name;
        t.shape = vshape;
        out.tensors[name] = std::move(t);
    }
    auto scalar = [&](const char* name, float& dst) -> bool {
        auto it = nodes.find(name);
        MetaTensor t;
        if (it == nodes.end() || !const_tensor(*it->second, t) || t.data.empty()) return false;
        dst = t.data[0];
        return true;
    };
    if (!scalar("loss/mul_4/y", out.ent_coef)) return "graph has no loss/mul_4/y (entropy coefficient)";
    if (!scalar("loss/mul_5/y", out.vf_coef)) return "graph has no loss/mul_5/y (value coefficient)";
    if (!scalar("loss/clip_by_global_norm/mul/x", out.clip_norm)) return "graph has no clip norm constant";
    if (!scalar("ppo2/_train/beta1", out.beta1) || !scalar("ppo2/_train/beta2", out.beta2) ||
        !scalar("ppo2/_train/epsilon", out.adam_eps))
        return "graph has no Adam constants";
    const auto& w0 = out.tensors["model/pi_fc0/w"].shape;
    const auto& w1 = out.tensors["model/pi_fc1/w"].shape;
    const auto& wp = out.tensors["model/pi/w"].shape;
    if (w0.size() != 2 || w1.size() != 2 || wp.size() != 2 || w0[1] != w1[0] || w1[1] != wp[0])
        return "unexpected MLP variable shapes in " + path;
    out.obs_dim = w0[0];
    out.hidden1 = w0[1];
    out.hidden2 = w1[1];
    out.act_dim = wp[1];
    out.action_space = classify_action_space(nodes, out.act_dim, out.action_space_error);
    return std::string();
}

}  // namespace ppo
