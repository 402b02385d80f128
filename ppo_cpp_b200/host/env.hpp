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
    virtual int get_num_envs() { return 1; }
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
};

// columns of an action matrix: get_action_space_size() for a continuous env; one (the index, as a float) for a discrete env,
// whose get_action_space_size() is the number of choices (Stable-Baselines' Discrete(n))
inline int action_width(Env& env) { return env.get_action_space() == Env::SPACE_DISCRETE() ? 1 : env.get_action_space_size(); }

#endif
