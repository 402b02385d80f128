// MlpPolicy with the reference's three calls (ppo2/policies.hpp:25-82); tensorflow::Tensor is replaced by Mat
// (SURVEY §8b: "that type must be replaced").  Each call is one C-ABI call instead of one Session::Run.
#ifndef PPO_B200_POLICIES_HPP
#define PPO_B200_POLICIES_HPP

#include <cstdint>
#include <vector>

#include "core_handle.hpp"
#include "mat.hpp"

// an action mask of 0 / 1 floats (Env::get_action_mask) as the bytes the C ABI takes
inline std::vector<uint8_t> action_mask_bytes(const Mat& m) {
    std::vector<uint8_t> b(static_cast<size_t>(m.size()));
    for (size_t i = 0; i < b.size(); ++i) b[i] = m.data()[i] > 0.5f ? 1 : 0;
    return b;
}

class MlpPolicy {
public:
    explicit MlpPolicy(CorePtr core, int act_dim) : core_{std::move(core)}, act_dim_{act_dim} {}

    // {action [n,A], value [n,1], neglogp [n,1]}  (fetch order of policies.hpp:37)
    std::vector<Mat> step(const Mat& obs) {
        Mat action(obs.rows(), act_dim_), value(obs.rows(), 1), neglogp(obs.rows(), 1);
        ppo_check(ppo_policy_step(core_.get(), obs.data(), obs.rows(), nullptr, action.data(), value.data(), neglogp.data(), PPO_HOST), "step");
        return {std::move(action), std::move(value), std::move(neglogp)};
    }
    // mask (optional, [n, logits] of 0 / 1): the argmax over the allowed actions of a masking core
    Mat get_deterministic_action(const Mat& obs, const Mat* mask = nullptr) {
        Mat action(obs.rows(), act_dim_);
        if (mask)
            ppo_check(ppo_policy_mean_masked(core_.get(), obs.data(), obs.rows(), action_mask_bytes(*mask).data(), action.data(), PPO_HOST),
                      "get_action(): evaluation step");
        else
            ppo_check(ppo_policy_mean(core_.get(), obs.data(), obs.rows(), action.data(), PPO_HOST), "get_action(): evaluation step");
        return action;
    }
    Mat value(const Mat& obs) {
        Mat v(obs.rows(), 1);
        ppo_check(ppo_policy_value(core_.get(), obs.data(), obs.rows(), v.data(), PPO_HOST), "value()");
        return v;
    }
    const CorePtr& core() const { return core_; }

private:
    CorePtr core_;
    int act_dim_;
};

#endif
