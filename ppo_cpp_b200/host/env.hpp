// Env abstract class — same interface as the reference's env/env.hpp:16-59 (quasi OpenAI-gym).
#ifndef PPO_B200_ENV_HPP
#define PPO_B200_ENV_HPP

#include <string>
#include <vector>

#include "json_min.hpp"
#include "mat.hpp"

// common/serializable.hpp:11-15
class ISerializable {
public:
    virtual ~ISerializable() {}
    virtual void serialize(nlohmann::json& json) = 0;
    virtual void deserialize(nlohmann::json& json) = 0;
};

class Env : public virtual ISerializable {
public:
    virtual ~Env() {}
    virtual std::string get_action_space() = 0;
    virtual std::string get_observation_space() = 0;
    virtual int get_action_space_size() = 0;
    virtual int get_observation_space_size() = 0;
    // a MultiDiscrete env's choices per action column (Stable-Baselines' nvec); empty for the other spaces
    virtual std::vector<int> get_action_space_nvec() { return {}; }
    virtual int get_num_envs() { return 1; }
    // invalid-action masks (sb3-contrib's action_masks()), Discrete and MultiDiscrete envs only: whether the env has them, and the
    // mask of its current observation, [n_envs, get_action_space_size()] of 0 / 1 (1 allowed) in logit order (for MultiDiscrete the
    // nvec slices side by side); every categorical must allow an action.  PPO2 then trains a masking core (ppo_core_set_action_masking).
    virtual bool has_action_mask() { return false; }
    virtual Mat get_action_mask() { return Mat(); }
    virtual Mat reset() = 0;
    // returns {obs [n,O], rewards [n,1], dones [n,1]}
    virtual std::vector<Mat> step(const Mat& actions) = 0;
    virtual void render() = 0;
    virtual float get_time() = 0;
    virtual Mat get_original_obs() = 0;
    virtual Mat get_original_rew() = 0;

    // the reference's spelling (env/env.hpp:58-59) is part of the checkpoint JSON format
    static const std::string& SPACE_CONTINOUS() {
        static const std::string s = "continous";
        return s;
    }
    static const std::string& SPACE_DISCRETE() {
        static const std::string s = "discrete";
        return s;
    }
    static const std::string& SPACE_MULTI_DISCRETE() {
        static const std::string s = "multi_discrete";
        return s;
    }
    static const std::string& SPACE_MULTI_BINARY() {
        static const std::string s = "multi_binary";
        return s;
    }
};

// columns of an action matrix: get_action_space_size() for a continuous env; one (the index, as a float) for a discrete env,
// whose get_action_space_size() is the number of choices (Stable-Baselines' Discrete(n)); one index per column of
// get_action_space_nvec() for a MultiDiscrete env, whose get_action_space_size() is sum(nvec) (the logits of the policy head);
// get_action_space_size() bits (0 / 1 as floats) for a MultiBinary env
inline int action_width(Env& env) {
    const std::string s = env.get_action_space();
    if (s == Env::SPACE_DISCRETE()) return 1;
    if (s == Env::SPACE_MULTI_DISCRETE()) return static_cast<int>(env.get_action_space_nvec().size());
    return env.get_action_space_size();
}

#endif
