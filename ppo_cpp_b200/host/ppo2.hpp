// PPO2 with the reference's constructor, learn(), eval(), save(), load() (ppo2/ppo2.hpp:31-519) on top of the
// B200 core.  No TensorFlow session: reset() reads the .meta.txt graph (shapes, initial weights, baked constants)
// through the C ABI and creates the device core.
#ifndef PPO_B200_PPO2_HPP
#define PPO_B200_PPO2_HPP

#include <chrono>
#include <cmath>
#include <fstream>
#include <functional>
#include <iostream>
#include <memory>
#include <sstream>
#include <stdexcept>
#include <string>
#include <vector>

#include "tensorboard.hpp"
#include "env.hpp"
#include "env_normalize.hpp"
#include "policies.hpp"
#include "runner.hpp"

// ppo2/base_class.hpp:9-44
class BaseRLModel {
public:
    explicit BaseRLModel(Env& env)
        : env{env}, action_space{env.get_action_space()}, observation_space{env.get_observation_space()},
          n_envs{env.get_num_envs()}, num_timesteps{0} {}

protected:
    bool _init_num_timesteps(bool reset_num_timesteps = true) {
        if (reset_num_timesteps) num_timesteps = 0;
        return num_timesteps == 0;
    }
    Env& env;
    std::string action_space;
    std::string observation_space;
    int n_envs;
    int num_timesteps;
};
class ActorCriticRLModel : public BaseRLModel {
public:
    explicit ActorCriticRLModel(Env& env) : BaseRLModel(env) {}
};

class PPO2 : public ActorCriticRLModel {
public:
    PPO2(std::string model_filename, Env& env, float gamma = 0.99, int n_steps = 128, float ent_coef = 0.01,
         float learning_rate = 2.5e-4, float vf_coef = 0.5f, float max_grad_norm = 0.5, float lam = 0.95, int nminibatches = 4,
         int noptepochs = 4, float cliprange = 0.2, float cliprange_vf = -1., std::string tensorboard_log = "")
        : ActorCriticRLModel(env), model_filename{std::move(model_filename)}, gamma{gamma}, n_steps{n_steps}, ent_coef{ent_coef},
          learning_rate{learning_rate}, vf_coef{vf_coef}, max_grad_norm{max_grad_norm}, lam{lam}, nminibatches{nminibatches},
          noptepochs{noptepochs}, cliprange{cliprange}, cliprange_vf{cliprange_vf}, tensorboard_log{std::move(tensorboard_log)} {
        if (this->model_filename.empty()) {
            std::cout << "PPO unitialized " << std::endl;
        } else {
            reset();
        }
    }

    // additions over the reference: the reference seeds from the clock (ppo2.cpp:159-162) and has no device choice
    void set_seed(unsigned shuffle_seed, uint64_t noise_seed) {
        shuffle_seed_ = shuffle_seed;
        noise_seed_ = noise_seed;
        if (core_) reset();
    }
    // Stable-Baselines' schedules (an addition over the reference, whose PPO2 takes constants): each is evaluated once per
    // update at frac = 1 - (update - 1) / n_updates, as ppo2.py does; the constructor's floats are the constant schedules.
    // An empty function keeps that constant.
    void set_schedules(std::function<float(float)> lr, std::function<float(float)> cr, std::function<float(float)> cr_vf) {
        lr_schedule_ = std::move(lr);
        cr_schedule_ = std::move(cr);
        cr_vf_schedule_ = std::move(cr_vf);
    }
    // graph-less construction for sizes the reference ships no graph for (orthogonal init as Stable-Baselines);
    // activation is a ppo_activation (a graph-built model follows its graph's)
    void reset_without_graph(int hidden1, int hidden2, uint64_t init_seed, int activation = PPO_ACT_TANH) {
        hidden_override_[0] = hidden1;
        hidden_override_[1] = hidden2;
        init_seed_ = init_seed;
        activation_ = activation;
        reset();
    }
    int activation() const { return activation_; }

    void reset() {
        n_batch = n_envs * n_steps;
        std::cout << "ppo2 " << std::endl;
        ppo_core_desc d;
        ppo_core_desc_default(&d);
        d.obs_dim = env.get_observation_space_size();
        d.act_dim = env.get_action_space_size();
        d.n_envs = n_envs; d.n_steps = n_steps; d.nminibatches = nminibatches; d.noptepochs = noptepochs;
        d.gamma = gamma; d.lam = lam;
        d.ent_coef = ent_coef; d.vf_coef = vf_coef; d.max_grad_norm = max_grad_norm;
        d.seed = noise_seed_;
        auto* normalize = dynamic_cast<EnvNormalize*>(&env);
        if (normalize) {
            normalize->fill_desc(d);
        } else {
            d.norm_obs = 0; d.norm_reward = 0; d.training = 0;
        }
        // a Discrete env gets a categorical head over its get_action_space_size() choices, a MultiDiscrete env one categorical per
        // column of its nvec, a MultiBinary env a Bernoulli per action bit; action_space (and nvec) are the env's, or the sidecar's
        // after load()
        const std::string spaces[4] = {Env::SPACE_CONTINOUS(), Env::SPACE_DISCRETE(), Env::SPACE_MULTI_DISCRETE(), Env::SPACE_MULTI_BINARY()};
        int space = -1;  // ppo_action_space: the index into spaces
        for (int i = 0; i < 4; ++i)
            if (action_space == spaces[i]) space = i;
        if (space < 0) throw std::runtime_error("PPO2: unsupported action space " + action_space);
        if (action_space != env.get_action_space())
            throw std::runtime_error("PPO2: the model's action space " + action_space + " is not the env's " + env.get_action_space());
        if (!loaded_nvec_.empty() && loaded_nvec_ != env.get_action_space_nvec())
            throw std::runtime_error("PPO2: the model's MultiDiscrete nvec is not the env's");
        const std::vector<int> nvec = env.get_action_space_nvec();
        const bool from_graph = hidden_override_[0] == 0;
        if (from_graph) {
            ppo_meta_info info;
            ppo_check(ppo_meta_parse(model_filename.c_str(), &info, nullptr, 0), "graph load");
            const int graph_space = ppo_meta_action_space(model_filename.c_str());
            ppo_check(graph_space < 0 ? graph_space : PPO_OK, "graph load");
            if (graph_space != space) {
                std::cout << "the graph's policy head does not match the env's " << action_space << " action space" << std::endl;
                throw std::runtime_error("PPO2: graph " + model_filename + " has a " + (graph_space >= 0 && graph_space < 4 ? spaces[graph_space] : std::string("unknown")) +
                                         " policy head, the env a " + action_space + " action space");
            }
            if (space == PPO_ACTION_MULTI_DISCRETE) {
                std::vector<int> g(64);
                const int k = ppo_meta_action_nvec(model_filename.c_str(), g.data(), static_cast<int>(g.size()));
                ppo_check(k < 0 ? k : PPO_OK, "graph load");
                g.resize(k);
                if (g != nvec) throw std::runtime_error("PPO2: graph " + model_filename + " splits its logits by another nvec than the env's");
            }
            if (info.obs_dim != d.obs_dim || info.act_dim != d.act_dim) {
                std::cout << "graph input/output widths do not match the environment" << std::endl;
                assert(false);
            }
            d.hidden1 = info.hidden1; d.hidden2 = info.hidden2;
        } else {
            d.hidden1 = hidden_override_[0]; d.hidden2 = hidden_override_[1];
        }
        core_ = make_core(d, space, nvec);
        if (from_graph) {
            // the graph's baked ent_coef / vf_coef / clip norm / Adam constants win over the constructor's (SURVEY §3.5)
            ppo_check(ppo_core_load_meta_txt(core_.get(), model_filename.c_str()), "graph load");
            activation_ = ppo_core_activation(core_.get());
        } else {
            ppo_check(ppo_core_init_orthogonal(core_.get(), init_seed_), "orthogonal init");
            ppo_check(ppo_core_set_activation(core_.get(), activation_), "activation");
        }
        ppo_check(ppo_shuffle_seed(core_.get(), shuffle_seed_), "shuffle seed");
        if (env.has_action_mask()) ppo_check(ppo_core_set_action_masking(core_.get(), 1), "action masks");
        if (normalize) normalize->attach_core(core_);
        act_model = std::make_unique<MlpPolicy>(core_, action_width(env));
    }

    void save(std::string save_path, int save_id = -1) {
        if (save_id >= 0) save_path += "." + std::to_string(save_id);
        // weights: TF Saver V2 bundle (<path>.data-00000-of-00001: 15 model tensors, sorted names, raw fp32; <path>.index: its table)
        ppo_check(ppo_core_save_checkpoint_data(core_.get(), save_path.c_str()), "Error saving checkpoint");
        std::cout << "Success save weights !! " << "\n";
        nlohmann::json json{};
        env.serialize(json);
        json["gamma"] = gamma; json["n_steps"] = n_steps; json["vf_coef"] = vf_coef; json["ent_coef"] = ent_coef;
        json["max_grad_norm"] = max_grad_norm; json["learning_rate"] = learning_rate; json["lam"] = lam;
        json["nminibatches"] = nminibatches; json["noptepochs"] = noptepochs; json["cliprange"] = cliprange;
        json["cliprange_vf"] = cliprange_vf; json["observation_space"] = observation_space; json["action_space"] = action_space;
        json["n_envs"] = n_envs; json["model_filename"] = model_filename;
        if (action_space == Env::SPACE_MULTI_DISCRETE()) json["nvec"] = env.get_action_space_nvec();
        // addition over the reference: a graph-less model (reset_without_graph) has no file to recover its shape from
        if (hidden_override_[0] > 0) {
            json["hidden1"] = hidden_override_[0];
            json["hidden2"] = hidden_override_[1];
            if (activation_ == PPO_ACT_RELU) json["activation"] = "relu";  // absent: tanh
        }
        std::ofstream myfile(save_path + ".json");
        if (myfile.is_open()) {
            myfile << json.dump();
            myfile.close();
        } else {
            std::cout << "Unable to open file for saving";
            assert(false);
        }
    }

    // like the reference: restores weights and normaliser statistics, Adam restarts from zero (ppo2.hpp:169-223)
    void load(std::string save_path) {
        std::ifstream in(save_path + ".json");
        if (!in.is_open()) {
            std::cout << "Unable to open file for loading" << std::endl;
            assert(false);
            throw std::runtime_error("Unable to open " + save_path + ".json");
        }
        std::stringstream sstr;
        sstr << in.rdbuf();
        nlohmann::json json = nlohmann::json::parse(sstr.str());
        gamma = json["gamma"].get<float>(); n_steps = json["n_steps"].get<int>(); vf_coef = json["vf_coef"].get<float>();
        ent_coef = json["ent_coef"].get<float>(); max_grad_norm = json["max_grad_norm"].get<float>();
        learning_rate = json["learning_rate"].get<float>(); lam = json["lam"].get<float>();
        nminibatches = json["nminibatches"].get<int>(); noptepochs = json["noptepochs"].get<int>();
        cliprange = json["cliprange"].get<float>(); cliprange_vf = json["cliprange_vf"].get<float>();
        observation_space = json["observation_space"].get<std::string>(); action_space = json["action_space"].get<std::string>();
        n_envs = json["n_envs"].get<int>();
        loaded_nvec_ = json.contains("nvec") ? json["nvec"].get<std::vector<int>>() : std::vector<int>{};
        if (n_envs != env.get_num_envs()) {
            // the reference only stores this number; here the device buffers are sized by it, so the live env wins
            std::cout << "checkpoint was written with n_envs " << n_envs << ", environment has " << env.get_num_envs() << std::endl;
            n_envs = env.get_num_envs();
        }
        if (model_filename.empty()) model_filename = json["model_filename"].get<std::string>();
        else std::cout << "filename passed through CLI overrides deserialized one" << std::endl;
        if (model_filename.empty() && hidden_override_[0] == 0) {  // written by a graph-less run: the sidecar holds the shape
            if (!json.contains("hidden1") || !json.contains("hidden2")) {
                std::cout << "checkpoint names no graph file and no hidden sizes" << std::endl;
                assert(false);
                throw std::runtime_error("checkpoint " + save_path + ".json names neither a graph file nor hidden sizes");
            }
            hidden_override_[0] = json["hidden1"].get<int>();
            hidden_override_[1] = json["hidden2"].get<int>();
            const std::string act = json.contains("activation") ? json["activation"].get<std::string>() : std::string("tanh");
            if (act != "tanh" && act != "relu") throw std::runtime_error("checkpoint " + save_path + ".json: unknown activation " + act);
            activation_ = act == "relu" ? PPO_ACT_RELU : PPO_ACT_TANH;
        }
        reset();
        env.deserialize(json);  // after reset(): the statistics live in the (new) core
        ppo_check(ppo_core_load_checkpoint_data(core_.get(), save_path.c_str()), "Error loading checkpoint");
        std::cout << "Success load weights !! " << std::endl;
    }

    // obs is the env's current observation: an env with action masks hands in its current mask with it
    Mat eval(const Mat& obs) const {
        const Mat mask = env.has_action_mask() ? env.get_action_mask() : Mat();
        Mat actions = act_model->get_deterministic_action(obs, env.has_action_mask() ? &mask : nullptr);
        assert(actions.rows() == obs.rows() && actions.cols() == action_width(env));
        return actions;
    }

    void learn(int total_timesteps, int num_saves = 0, const std::string& save_path = "", const std::string& tb_log_name = "PPO2") {
        if (!core_) {
            std::cout << "Session unitialized, learning aborted.";
            assert(false);
            return;
        }
        // the value loss is fixed by the graph (SURVEY 3.5): only a graph with loss/clip_range_vf_ph takes cliprange_vf
        const bool separate = ppo_core_vf_clip(core_.get()) == PPO_VF_CLIP_SEPARATE;
        if (separate && !cr_vf_schedule_ && cliprange_vf < 0.f) {
            std::cerr << "the graph clips the value with its own range (loss/clip_range_vf_ph): cliprange_vf must be >= 0, got " << cliprange_vf << std::endl;
            throw std::runtime_error("PPO2::learn: the graph needs cliprange_vf >= 0");
        }
        if (!separate && cliprange_vf >= 0.f) {
            std::cout << (ppo_core_vf_clip(core_.get()) == PPO_VF_CLIP_NONE ? "cliprange_vf is ignored: the graph does not clip the value"
                                                                            : "cliprange_vf is ignored: the graph clips the value with cliprange (SURVEY 3.5)")
                      << std::endl;
        }
        _init_num_timesteps();
        Runner runner{env, *act_model, n_steps, gamma, lam};
        std::vector<float> episode_reward(n_envs, 0.f);
        std::unique_ptr<TensorboardWriter> writer;  // TensorboardWriter writer{tensorboard_log, tb_log_name, new_tb_log} (ppo2.hpp:248)
        if (!tb_log_name.empty() && !tensorboard_log.empty()) writer = std::make_unique<TensorboardWriter>(tensorboard_log, tb_log_name);
        const int n_updates = total_timesteps / n_batch;
        int save_interval = -1;
        if (num_saves > 0) save_interval = static_cast<int>(std::ceil(static_cast<float>(n_updates) / static_cast<float>(num_saves)));
        for (int update = 1; update <= n_updates; ++update) {
            assert((n_batch % nminibatches) == 0);
            auto t_start = std::chrono::system_clock::now();
            runner.run(false);
            num_timesteps += n_batch;
            float loss_vals[5];
            const float frac = 1.0f - (static_cast<float>(update) - 1.0f) / static_cast<float>(n_updates);
            const float lr_now = lr_schedule_ ? lr_schedule_(frac) : learning_rate;
            const float cr_now = cr_schedule_ ? cr_schedule_(frac) : cliprange;
            const float cr_vf_now = cr_vf_schedule_ ? cr_vf_schedule_(frac) : cliprange_vf;
            if (separate) ppo_check(ppo_train_update_vf(core_.get(), lr_now, cr_now, cr_vf_now, loss_vals), "train");
            else ppo_check(ppo_train_update(core_.get(), lr_now, cr_now, loss_vals), "train");
            auto t_now = std::chrono::system_clock::now();
            auto duration = std::chrono::duration_cast<std::chrono::microseconds>(t_now - t_start).count();
            last_fps = static_cast<long>(static_cast<double>(n_batch) * 1e6 / static_cast<double>(duration > 0 ? duration : 1));
            std::cout << last_fps << ",";  // fps,pg_loss,vf_loss,entropy,approxkl,clipfrac,  (ppo2.hpp:343-349)
            for (int i = 0; i < 5; ++i) {
                std::cout << loss_vals[i] << ",";
                last_losses[i] = loss_vals[i];
            }
            std::cout << std::endl;
            if (writer) log_episode_rewards(runner, episode_reward, *writer, num_timesteps - n_batch);
            if (save_interval > 0 && num_saves > 0 && update % save_interval == 0) {
                assert(!save_path.empty());
                save(save_path, update / save_interval - 1);
            }
        }
        if (num_saves > 0) {
            assert(!save_path.empty());
            if (save_interval > 0 && ((n_updates % save_interval) != 0)) save(save_path, n_updates / save_interval);
            else if (save_interval == 0) save(save_path);
        }
    }

    const CorePtr& core() const { return core_; }
    long last_fps = 0;
    float last_losses[5] = {0, 0, 0, 0, 0};

private:
    // Utils::total_episode_reward_logger (ppo2/utils.hpp:75-114): the reward summed over each finished episode as the
    // TensorBoard scalar "episode_reward" at global step total_steps + t (ppo2.hpp:358); the same pairs also go to
    // <tensorboard_log>/episode_reward.csv ("step,episode_reward")
    void log_episode_rewards(Runner& runner, std::vector<float>& acc, TensorboardWriter& writer, int total_steps) {
        auto rew = runner.fetch("unnormalized_rewards", 1);
        auto dn = runner.fetch("dones", 1);
        std::ofstream out(tensorboard_log + "/episode_reward.csv", std::ios::app);
        for (int e = 0; e < n_envs; ++e) {
            for (int t = 0; t < n_steps; ++t) {
                if ((*dn)(e * n_steps + t, 0) > .5f) {
                    writer.write_scalar(total_steps + t, "episode_reward", acc[e]);
                    out << (total_steps + t) << "," << acc[e] << "\n";
                    acc[e] = 0.f;
                }
                acc[e] += (*rew)(e * n_steps + t, 0);
            }
        }
    }

    std::string model_filename;
    float gamma;
    int n_steps;
    float ent_coef;
    float learning_rate;
    float vf_coef;
    float max_grad_norm;
    float lam;
    int nminibatches;
    int noptepochs;
    float cliprange;
    float cliprange_vf;
    std::function<float(float)> lr_schedule_, cr_schedule_, cr_vf_schedule_;
    std::string tensorboard_log;
    int n_batch = 0;
    unsigned shuffle_seed_ = 1;
    uint64_t noise_seed_ = 0;
    int hidden_override_[2] = {0, 0};
    uint64_t init_seed_ = 0;
    int activation_ = PPO_ACT_TANH;  // ppo_activation of the core (graph-less: chosen; otherwise the graph's)
    std::vector<int> loaded_nvec_;   // the MultiDiscrete nvec of the sidecar read by load() (empty: none)
    CorePtr core_;
    std::unique_ptr<MlpPolicy> act_model;
};

#endif
