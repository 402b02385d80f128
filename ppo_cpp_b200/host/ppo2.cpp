// CLI with the reference's flags (ppo2.cpp:93-128) driving the B200 core.  Envs: the DART hexapod cannot be
// built here (SURVEY §2 row 12); `--env synthetic` (default) is the host-side stand-in with the same shapes,
// `--env mock` is the reference's EnvMock, `--env bandit` a Discrete(4) contextual bandit for the categorical head.  New flags: --env, --seed (commented out in the reference,
// ppo2.cpp:130-131), --hidden H1,H2 (graph-less orthogonal init when no --graph is given).
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <limits>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "env_bandit.hpp"
#include "env_mock.hpp"
#include "env_normalize.hpp"
#include "env_synthetic.hpp"
#include "ppo2.hpp"
#include "vec_env.hpp"

namespace {
struct Args {
    std::map<std::string, std::string> values;
    std::map<std::string, bool> flags;
};
// alias -> canonical name; value flags and boolean flags exactly as args.hxx declares them in the reference
const std::map<std::string, std::string> kValueFlags = {
    {"-d", "dir"}, {"--dir", "dir"}, {"-g", "graph"}, {"--graph", "graph"}, {"--graph_path", "graph"}, {"-p", "path"}, {"--path", "path"},
    {"--id", "id"}, {"-s", "steps"}, {"--steps", "steps"}, {"-l", "lr"}, {"--lr", "lr"}, {"--learning_rate", "lr"}, {"--learningrate", "lr"},
    {"-e", "ent"}, {"--ent", "ent"}, {"--entropy", "ent"}, {"-c", "cr"}, {"--cr", "cr"}, {"--clip_range", "cr"}, {"--cliprange", "cr"},
    {"--saves", "saves"}, {"--n_saves", "saves"}, {"--num_saves", "saves"}, {"--epochs", "epochs"}, {"--n_epochs", "epochs"},
    {"--num_epochs", "epochs"}, {"--batch_steps", "batch_steps"}, {"--n_steps", "batch_steps"}, {"--num_steps", "batch_steps"},
    {"--reset_noise_scale", "rns"}, {"--reset_noise", "rns"}, {"--rns", "rns"}, {"--rn", "rns"}, {"--duration", "duration"}, {"--du", "duration"},
    {"-j", "threads"}, {"--jobs", "threads"}, {"--threads", "threads"}, {"--n_threads", "threads"}, {"--num_threads", "threads"}, {"--nt", "threads"},
    {"-f", "fps"}, {"--framerate", "fps"}, {"--fps", "fps"}, {"--env", "env"}, {"--seed", "seed"}, {"--hidden", "hidden"},
    {"--cliprange_vf", "cliprange_vf"}, {"--clip_range_vf", "cliprange_vf"}, {"--activation", "activation"}};
const std::map<std::string, std::string> kBoolFlags = {
    {"--closed_loop", "cl"}, {"--closed-loop", "cl"}, {"--cl", "cl"}, {"-v", "verbose"}, {"--verbose", "verbose"}, {"-r", "resume"},
    {"--resume", "resume"}, {"--bullet", "bullet"}, {"--use_bullet", "bullet"}, {"--bullet_solver", "bullet"}, {"-h", "help"}, {"--help", "help"}};

bool parse(int argc, char** argv, Args& a) {
    for (int i = 1; i < argc; ++i) {
        std::string tok = argv[i], val;
        const size_t eq = tok.find('=');
        if (eq != std::string::npos) {
            val = tok.substr(eq + 1);
            tok = tok.substr(0, eq);
        }
        auto b = kBoolFlags.find(tok);
        if (b != kBoolFlags.end()) {
            a.flags[b->second] = true;
            continue;
        }
        auto v = kValueFlags.find(tok);
        if (v == kValueFlags.end()) {
            std::cerr << "Flag could not be matched: " << tok << std::endl;
            return false;
        }
        if (eq == std::string::npos) {
            if (i + 1 >= argc) {
                std::cerr << "Flag " << tok << " needs a value" << std::endl;
                return false;
            }
            val = argv[++i];
        }
        a.values[v->second] = val;
    }
    return true;
}
std::string get(const Args& a, const char* k, const char* dflt) {
    auto it = a.values.find(k);
    return it == a.values.end() ? std::string(dflt) : it->second;
}
void mkdir_p(const std::string& path) {
    const std::string cmd = "mkdir -p " + path;
    if (system(cmd.c_str()) != 0) std::cerr << "Error creating directory!" << std::endl;
}
}  // namespace

int main(int argc, char** argv) {
    Args a;
    if (!parse(argc, argv, a)) return 1;
    if (a.flags["help"]) {
        std::cout << "This is a gait learner/viewer program using PPO algorithm (B200 core)\n"
                     "  -d --dir, -g --graph --graph_path, -p --path, --id, -s --steps, -l --lr, -e --ent, -c --cr,\n"
                     "  --saves, --epochs --num_epochs, --batch_steps --n_steps, --rns, --cl, -v, -r --resume, --bullet,\n"
                     "  --duration, -j --threads, -f --fps   (as in the reference's ppo2.cpp:93-128)\n"
                     "  --env synthetic|mock|bandit (bandit: a Discrete(4) contextual bandit), --seed N, --hidden H1,H2,\n"
                     "  --cliprange_vf (-1: the graph's value loss decides; >= 0 for a graph with loss/clip_range_vf_ph),\n"
                     "  --activation tanh|relu (graph-less runs; with a graph it must name the graph's own activation)\n";
        return 0;
    }
    const std::string save_path = get(a, "dir", "./exp/ppo_cpp"), graph_path = get(a, "graph", "");
    const bool has_load = a.values.count("path") > 0;
    const float steps = std::stof(get(a, "steps", "2e7")), lr = std::stof(get(a, "lr", "1e-3")), ent = std::stof(get(a, "ent", "0"));
    const float cr = std::stof(get(a, "cr", "0.2"));
    const float cr_vf = std::stof(get(a, "cliprange_vf", "-1"));  // the value ppo2.cpp:215-217 hard-wires
    const int epochs = std::stoi(get(a, "epochs", "10")), batch_steps = std::stoi(get(a, "batch_steps", "2048"));
    const int threads = std::stoi(get(a, "threads", "1"));
    const double duration = std::stod(get(a, "duration", "5."));
    const std::string env_kind = get(a, "env", "synthetic");
    const std::string act_name = get(a, "activation", "");
    if (!act_name.empty() && act_name != "tanh" && act_name != "relu") {
        std::cerr << "--activation must be tanh or relu, not " << act_name << std::endl;
        return 1;
    }
    const int act = act_name == "relu" ? PPO_ACT_RELU : PPO_ACT_TANH;
    if (!act_name.empty() && !graph_path.empty()) {
        const int graph_act = ppo_meta_activation(graph_path.c_str());
        if (graph_act >= 0 && graph_act != act) {
            std::cerr << "--activation " << act_name << " contradicts the graph " << graph_path << ", whose hidden layers are "
                      << (graph_act == PPO_ACT_RELU ? "relu" : "tanh") << std::endl;
            return 1;
        }
    }

    unsigned seed_val;
    if (a.values.count("seed")) {
        seed_val = static_cast<unsigned>(std::stoul(a.values["seed"]));
    } else {  // the reference's clock seed (ppo2.cpp:159-162)
        auto nanos = std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::high_resolution_clock::now().time_since_epoch()).count();
        seed_val = static_cast<unsigned>(nanos % std::numeric_limits<int>::max());
    }
    const std::string run_id = a.values.count("id") ? a.values["id"] : ("ppo_" + std::to_string(time(nullptr)));
    const std::string tb_path = save_path + "/tensorboard/" + run_id + "/";
    const bool training = !has_load || a.flags["resume"];

    std::unique_ptr<Env> wrapped_env;
    std::vector<std::shared_ptr<Env>> envs;
    auto make_env = [&](int i) -> std::shared_ptr<Env> {
        if (env_kind == "mock") return std::make_shared<EnvMock>(1.0);
        if (env_kind == "bandit") return std::make_shared<BanditEnv>(static_cast<uint64_t>(seed_val) ^ 0x1234ull, static_cast<uint32_t>(i));
        return std::make_shared<SyntheticEnv>(static_cast<uint64_t>(seed_val) ^ 0x1234ull, static_cast<uint32_t>(i));
    };
    if (threads > 1) {
        for (int i = 0; i < threads; ++i) envs.push_back(make_env(i));
        wrapped_env = std::make_unique<VecEnv>(envs);
    } else if (env_kind == "mock") {
        wrapped_env = std::make_unique<EnvMock>(1.0);
    } else if (env_kind == "bandit") {
        wrapped_env = std::make_unique<BanditEnv>(static_cast<uint64_t>(seed_val) ^ 0x1234ull, 0);
    } else {
        wrapped_env = std::make_unique<SyntheticEnv>(static_cast<uint64_t>(seed_val) ^ 0x1234ull, 0);
    }
    EnvNormalize env{std::move(wrapped_env), training};

    std::cout << "lr: " << lr << std::endl;
    std::cout << "ent: " << ent << std::endl;
    std::cout << "cr: " << cr << std::endl;

    // gamma .99, vf_coef .5, max_grad_norm .5, lam .95, nminibatches 32 as hard-wired in ppo2.cpp:215-217
    PPO2 algorithm{graph_path, env, .99f, batch_steps, ent, lr, .5f, .5f, .95f, 32, epochs, cr, cr_vf, tb_path};
    algorithm.set_seed(seed_val, seed_val);
    if (graph_path.empty() && !has_load) {
        int h1 = 64, h2 = 64;
        if (a.values.count("hidden")) sscanf(a.values["hidden"].c_str(), "%d,%d", &h1, &h2);
        algorithm.reset_without_graph(h1, h2, seed_val, act);
    }
    if (has_load) {
        algorithm.load(a.values["path"]);
        if (!act_name.empty() && algorithm.activation() != act) {
            std::cerr << "--activation " << act_name << " contradicts the checkpoint " << a.values["path"] << std::endl;
            return 1;
        }
    }

    if (training) {
        mkdir_p(tb_path);
        const std::string checkpoint_dir = save_path + "/checkpoints/" + run_id + "/";
        mkdir_p(checkpoint_dir);
        const std::string checkpoint_path = checkpoint_dir + "/" + run_id + ".pkl";
        const int int_steps = static_cast<int>(steps);
        const int total_saves = a.values.count("saves") ? std::stoi(a.values["saves"]) : (int_steps > 1e6 ? static_cast<int>(int_steps / 1e6) : 1);
        std::cout << "steps: " << int_steps << std::endl;
        std::cout << "num_saves: " << total_saves << std::endl;
        algorithm.learn(int_steps, total_saves, checkpoint_path);
    } else {  // playback (ppo2.cpp:40-77) without rendering
        const int playback_steps = static_cast<int>(duration / 0.015);
        Mat obs = env.reset();
        float episode_reward = 0.f;
        for (int i = 0; i < playback_steps; ++i) {
            const auto out = env.step(algorithm.eval(obs));
            obs = out[0];
            episode_reward += env.get_original_rew()(0, 0);
            if (out[2](0, 0) > .5f) break;
        }
        std::cout << "episode_reward: " << episode_reward << std::endl;
    }
    return 0;
}
