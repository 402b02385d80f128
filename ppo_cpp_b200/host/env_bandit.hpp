// Host-side contextual bandit, a small seeded env for the policy heads without logstd, in three modes:
//   DISCRETE        Discrete(n): the observation is the one-hot code of a context c in 0 .. n-1; the action is an index (one fp32
//                   column); the reward is 1 when the action is (c + 1) mod n and 0 otherwise.  A uniform policy earns 1/n.
//   MULTI_DISCRETE  MultiDiscrete([4, 3]) on the one-hot context c in 0 .. 3: two index columns; the reward is
//                   1/2 [a0 == (c + 1) mod 4] + 1/2 [a1 == c mod 3].  A uniform policy earns 1/2 (1/4 + 1/3).
//   MULTI_BINARY    MultiBinary(4): the observation is the bit pattern of a context c in 0 .. 15; the action is 4 columns of 0 / 1;
//                   the reward is the fraction of action bits equal to c's bits.  A uniform policy earns 1/2.
//   MASKED          Discrete(4) on the one-hot context c in 0 .. 3 with invalid-action masks: c forbids one or two actions, never the
//                   rewarded one (c + 1) mod 4; the reward is 1 for that action and 0 otherwise.  A uniform policy over the allowed
//                   actions earns 1/2 or 1/3.  The env counts the forbidden actions it receives (illegal_actions()).
// A new context is drawn (splitmix64 of seed, env id and step) after every step; episodes last 16 steps.  The learned policy
// earns up to 1 per step, so learning is visible in the mean reward.
#ifndef PPO_B200_ENV_BANDIT_HPP
#define PPO_B200_ENV_BANDIT_HPP

#include <cstdint>

#include "env.hpp"

class BanditEnv : public Env {
public:
    enum Mode { DISCRETE, MULTI_DISCRETE, MULTI_BINARY, MASKED };
    explicit BanditEnv(uint64_t seed = 0x1234, uint32_t env_id = 0, int n = 4, Mode mode = DISCRETE)
        : seed{seed}, env_id{env_id}, n{mode == DISCRETE ? n : 4}, mode{mode}, obs(1, this->n) { reset(); }
    std::string get_action_space() override {
        return mode == DISCRETE || mode == MASKED ? Env::SPACE_DISCRETE() : mode == MULTI_DISCRETE ? Env::SPACE_MULTI_DISCRETE() : Env::SPACE_MULTI_BINARY();
    }
    bool has_action_mask() override { return mode == MASKED; }
    Mat get_action_mask() override {
        Mat m(1, n);
        for (int k = 0; k < n; ++k) m(0, k) = allowed(k) ? 1.f : 0.f;
        return m;
    }
    long illegal_actions() const { return illegal; }
    std::string get_observation_space() override { return Env::SPACE_CONTINOUS(); }
    int get_action_space_size() override { return mode == MULTI_DISCRETE ? 4 + 3 : n; }
    std::vector<int> get_action_space_nvec() override { return mode == MULTI_DISCRETE ? std::vector<int>{4, 3} : std::vector<int>{}; }
    int get_observation_space_size() override { return n; }
    Mat reset() override {
        t_env = 0;
        draw();
        return obs;
    }
    std::vector<Mat> step(const Mat& actions) override {
        if (mode == DISCRETE || mode == MASKED) {
            const int a = static_cast<int>(actions(0, 0));
            if (mode == MASKED && !allowed(a)) ++illegal;
            last_rew = a == (ctx + 1) % n ? 1.f : 0.f;
        } else if (mode == MULTI_DISCRETE) {
            last_rew = 0.5f * (static_cast<int>(actions(0, 0)) == (ctx + 1) % 4 ? 1.f : 0.f) + 0.5f * (static_cast<int>(actions(0, 1)) == ctx % 3 ? 1.f : 0.f);
        } else {
            int same = 0;
            for (int k = 0; k < n; ++k) same += (actions(0, k) > 0.5f) == (((ctx >> k) & 1) != 0);
            last_rew = static_cast<float>(same) / static_cast<float>(n);
        }
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
    // MASKED: context c forbids c itself, and (c + 2) mod 4 as well in odd contexts; (c + 1) mod 4, the rewarded action, stays allowed
    bool allowed(int a) const { return a != ctx && !((ctx & 1) && a == (ctx + 2) % n); }
    void draw() {
        uint64_t z = seed + 0x9E3779B97F4A7C15ull * (((uint64_t)env_id << 32) + (++draws));
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        z ^= z >> 31;
        ctx = static_cast<int>(z % static_cast<uint64_t>(mode == MULTI_BINARY ? 1 << n : n));
        for (int k = 0; k < n; ++k) obs(0, k) = (mode == MULTI_BINARY ? ((ctx >> k) & 1) != 0 : k == ctx) ? 1.f : 0.f;
    }
    uint64_t seed;
    uint32_t env_id;
    int n;
    Mode mode;
    Mat obs;
    int ctx = 0;
    uint32_t t_env = 0;
    uint64_t draws = 0;
    float last_rew = 0.f;
    long illegal = 0;
};

#endif
