// Host-side contextual bandit with a Discrete(n) action space: a small seeded env for the categorical policy head.
// The observation is the one-hot code of a context c in 0 .. n-1; the action is an index (one fp32 column); the reward is 1
// when the action is (c + 1) mod n and 0 otherwise.  A new context is drawn (splitmix64 of seed, env id and step) after every
// step; episodes last 16 steps.  A uniform policy earns 1/n per step, the learned one up to 1, so learning is visible in the
// mean reward.
#ifndef PPO_B200_ENV_BANDIT_HPP
#define PPO_B200_ENV_BANDIT_HPP

#include <cstdint>

#include "env.hpp"

class BanditEnv : public Env {
public:
    explicit BanditEnv(uint64_t seed = 0x1234, uint32_t env_id = 0, int n = 4) : seed{seed}, env_id{env_id}, n{n}, obs(1, n) { reset(); }
    std::string get_action_space() override { return Env::SPACE_DISCRETE(); }
    std::string get_observation_space() override { return Env::SPACE_CONTINOUS(); }
    int get_action_space_size() override { return n; }
    int get_observation_space_size() override { return n; }
    Mat reset() override {
        t_env = 0;
        draw();
        return obs;
    }
    std::vector<Mat> step(const Mat& actions) override {
        last_rew = static_cast<int>(actions(0, 0)) == (ctx + 1) % n ? 1.f : 0.f;
        ++t_env;
        Mat done = Mat::Zero(1, 1);
        if (t_env % 16u == 0u) done(0, 0) = 1.f;
        draw();
        Mat rew(1, 1);
        rew(0, 0) = last_rew;
        return {obs, rew, done};
    }
    Mat get_original_obs() override { return obs; }
    Mat get_original_rew() override {
        Mat r(1, 1);
        r(0, 0) = last_rew;
        return r;
    }
    void serialize(nlohmann::json&) override {}
    void deserialize(nlohmann::json&) override {}
    void render() override {}
    float get_time() override { return static_cast<float>(t_env); }

private:
    void draw() {
        uint64_t z = seed + 0x9E3779B97F4A7C15ull * (((uint64_t)env_id << 32) + (++draws));
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        z ^= z >> 31;
        ctx = static_cast<int>(z % static_cast<uint64_t>(n));
        for (int k = 0; k < n; ++k) obs(0, k) = k == ctx ? 1.f : 0.f;
    }
    uint64_t seed;
    uint32_t env_id;
    int n;
    Mat obs;
    int ctx = 0;
    uint32_t t_env = 0;
    uint64_t draws = 0;
    float last_rew = 0.f;
};

#endif
