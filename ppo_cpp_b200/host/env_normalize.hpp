// EnvNormalize — VecNormalize wrapper with the reference's constructor and Env interface
// (env/env_normalize.hpp:18-162).  The running statistics and all arithmetic live on the device:
//   * stand-alone use (playback, tests): step()/reset() call ppo_vecnorm_step/reset on a private core;
//   * under PPO2::learn the Runner drives the INNER env directly and lets the core normalise inside
//     ppo_runner_observe (no extra host round trip) — PPO2 attaches its core with attach_core(), which moves the
//     statistics over.
#ifndef PPO_B200_ENV_NORMALIZE_HPP
#define PPO_B200_ENV_NORMALIZE_HPP

#include <memory>

#include "core_handle.hpp"
#include "env.hpp"

class EnvNormalize : public Env {
public:
    EnvNormalize(std::unique_ptr<Env> env, bool training, bool norm_obs = true, bool norm_reward = true, float clip_reward = 10,
                 float clip_obs = 10, float gamma = 0.99, float epsilon = 1e-8)
        : env{std::move(env)}, training{training}, norm_obs{norm_obs}, norm_reward{norm_reward}, clip_reward{clip_reward},
          clip_obs{clip_obs}, gamma{gamma}, epsilon{epsilon} {}

    std::string get_action_space() override { return env->get_action_space(); }
    std::string get_observation_space() override { return env->get_observation_space(); }
    int get_action_space_size() override { return env->get_action_space_size(); }
    std::vector<int> get_action_space_nvec() override { return env->get_action_space_nvec(); }
    bool has_action_mask() override { return env->has_action_mask(); }
    Mat get_action_mask() override { return env->get_action_mask(); }
    int get_observation_space_size() override { return env->get_observation_space_size(); }
    int get_num_envs() override { return env->get_num_envs(); }

    std::vector<Mat> step(const Mat& actions) override {
        const std::vector<Mat>& results = env->step(actions);
        Mat obs(results[0].rows(), results[0].cols()), rews(results[1].rows(), 1);
        ppo_check(ppo_vecnorm_step(core().get(), results[0].data(), results[1].data(), results[2].data(), obs.data(), rews.data(), PPO_HOST),
                  "EnvNormalize::step");
        return {std::move(obs), std::move(rews), results[2]};
    }
    Mat reset() override {
        const Mat& raw = env->reset();
        Mat obs(raw.rows(), raw.cols());
        ppo_check(ppo_vecnorm_reset(core().get(), raw.data(), obs.data(), PPO_HOST), "EnvNormalize::reset");
        return obs;
    }
    void render() override { env->render(); }
    float get_time() override { return env->get_time(); }
    Mat get_original_obs() override { return env->get_original_obs(); }
    Mat get_original_rew() override { return env->get_original_rew(); }

    void serialize(nlohmann::json& json) override {
        const int O = get_observation_space_size();
        std::vector<float> om(O), ov(O), rm(1), rv(1);
        double oc = 0, rc = 0;
        ppo_check(ppo_vecnorm_get_stats(core().get(), om.data(), ov.data(), &oc, rm.data(), rv.data(), &rc), "EnvNormalize::serialize");
        json["obs_rms"]["var"] = ov; json["obs_rms"]["mean"] = om; json["obs_rms"]["count"] = oc;
        json["ret_rms"]["var"] = rv; json["ret_rms"]["mean"] = rm; json["ret_rms"]["count"] = rc;
        env->serialize(json);
    }
    void deserialize(nlohmann::json& json) override {
        auto om = json["obs_rms"]["mean"].get<std::vector<float>>();
        auto ov = json["obs_rms"]["var"].get<std::vector<float>>();
        auto rm = json["ret_rms"]["mean"].get<std::vector<float>>();
        auto rv = json["ret_rms"]["var"].get<std::vector<float>>();
        assert(static_cast<int>(om.size()) == get_observation_space_size());
        ppo_check(ppo_vecnorm_set_stats(core().get(), om.data(), ov.data(), json["obs_rms"]["count"].get<double>(), rm.data(), rv.data(),
                                        json["ret_rms"]["count"].get<double>()),
                  "EnvNormalize::deserialize");
        env->deserialize(json);
    }

    // ---- additions over the reference's interface (used by Runner / PPO2 only)
    Env& inner() { return *env; }
    bool is_training() const { return training; }
    void fill_desc(ppo_core_desc& d) const {
        d.norm_obs = norm_obs; d.norm_reward = norm_reward; d.training = training;
        d.clip_obs = clip_obs; d.clip_reward = clip_reward; d.norm_gamma = gamma; d.norm_epsilon = epsilon;
    }
    // share PPO2's core; statistics gathered so far move over
    void attach_core(const CorePtr& shared) {
        if (core_ && core_ != shared) {
            const int O = get_observation_space_size();
            std::vector<float> om(O), ov(O), rm(1), rv(1);
            double oc = 0, rc = 0;
            ppo_check(ppo_vecnorm_get_stats(core_.get(), om.data(), ov.data(), &oc, rm.data(), rv.data(), &rc), "EnvNormalize::attach_core");
            ppo_check(ppo_vecnorm_set_stats(shared.get(), om.data(), ov.data(), oc, rm.data(), rv.data(), rc), "EnvNormalize::attach_core");
        }
        core_ = shared;
    }

private:
    const CorePtr& core() {
        if (!core_) {  // private core: only VecNormalize state is used
            ppo_core_desc d;
            ppo_core_desc_default(&d);
            d.obs_dim = get_observation_space_size();
            d.act_dim = get_action_space_size();
            d.n_envs = get_num_envs();
            d.n_steps = 1; d.nminibatches = 1; d.noptepochs = 0;
            fill_desc(d);
            core_ = make_core(d);
        }
        return core_;
    }

    std::unique_ptr<Env> env;
    bool training, norm_obs, norm_reward;
    float clip_reward, clip_obs, gamma, epsilon;
    CorePtr core_;
};

#endif
