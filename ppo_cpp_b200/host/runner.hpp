// Runner / MiniBatch with the reference's interface (ppo2/runner.hpp:21-202).
// run() keeps the reference's loop — per step: policy step, env.step on the host, store — but every store and
// all arithmetic (VecNormalize, GAE) happen on the device: the host only moves the env's raw observation, reward
// and done flags in (ppo_runner_observe) and the actions out (ppo_runner_act).
#ifndef PPO_B200_RUNNER_HPP
#define PPO_B200_RUNNER_HPP

#include <memory>
#include <vector>

#include "env.hpp"
#include "env_normalize.hpp"
#include "policies.hpp"

struct MiniBatch {
    std::shared_ptr<Mat> obs, returns, dones, actions, values, neglogpacs, true_rewards, unnormalized_rewards;
    std::vector<std::shared_ptr<Mat>> get_train_input() const { return {obs, returns, dones, actions, values, neglogpacs}; }
    std::vector<std::shared_ptr<Mat>> get_1_dims() const { return {returns, dones, values, neglogpacs, true_rewards, unnormalized_rewards}; }
};

class Runner {
public:
    Runner(Env& env, MlpPolicy& model, int n_steps, float gamma, float lam)
        : env{env}, model{model}, n_steps{n_steps}, gamma{gamma}, lam{lam}, num_envs{env.get_num_envs()},
          normalize{dynamic_cast<EnvNormalize*>(&env)} {
        // obs{env.reset()} (runner.hpp:48): the raw reset observation goes to the core, which applies
        // EnvNormalize::reset (statistics update + normalise + clip) on the device.
        const Mat raw = normalize ? normalize->inner().reset() : env.reset();
        ppo_check(ppo_runner_reset(model.core().get(), raw.data(), PPO_HOST), "Runner::Runner");
    }

    // fetch_all = false skips the device->host export of the eight rollout buffers (PPO2::learn trains on the
    // device and only fetches what its logging needs).
    MiniBatch run(bool fetch_all = true) {
        ppo_core* core = model.core().get();
        Env& stepper = normalize ? normalize->inner() : env;
        Mat actions(num_envs, action_width(env));
        for (int step = 0; step < n_steps; ++step) {
            ppo_check(ppo_runner_act(core, step, actions.data(), PPO_HOST), "Runner::run act");
            const std::vector<Mat>& r = stepper.step(actions);  // env handles action clipping (runner.hpp:112)
            assert(r[0].rows() == num_envs && r[0].cols() == env.get_observation_space_size());
            assert(r[1].rows() == num_envs && r[1].cols() == 1 && r[2].rows() == num_envs && r[2].cols() == 1);
            ppo_check(ppo_runner_observe(core, step, r[0].data(), r[1].data(), r[2].data(), PPO_HOST), "Runner::run observe");
        }
        ppo_check(ppo_runner_finish(core), "Runner::run finish");  // set_returns (runner.hpp:159-191)
        MiniBatch mb{};
        if (fetch_all) {
            mb.obs = fetch("obs", env.get_observation_space_size());
            mb.actions = fetch("actions", action_width(env));
            mb.returns = fetch("returns", 1);
            mb.dones = fetch("dones", 1);
            mb.values = fetch("values", 1);
            mb.neglogpacs = fetch("neglogpacs", 1);
            mb.true_rewards = fetch("true_rewards", 1);
            mb.unnormalized_rewards = fetch("unnormalized_rewards", 1);
        }
        return mb;
    }

    // flat layout of the reference: row = env*n_steps + t (runner.hpp:136-152)
    std::shared_ptr<Mat> fetch(const char* name, int width) const {
        auto m = std::make_shared<Mat>(num_envs * n_steps, width);
        ppo_check(ppo_rollout_get(model.core().get(), name, m->data(), m->size()), "Runner::fetch");
        return m;
    }

private:
    Env& env;
    MlpPolicy& model;
    int n_steps;
    float gamma;
    float lam;
    int num_envs;
    EnvNormalize* normalize;
};

#endif
