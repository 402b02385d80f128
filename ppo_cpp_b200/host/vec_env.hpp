// VecEnv — thread-per-env vectoriser with the reference's interface and observable behaviour
// (env/vec_env.hpp:16-281): constructor takes (and keeps a reference to) the caller's vector of envs, spawns
// one thread per env which resets its env once, step() runs all envs in lock-step and returns
// {observations, rewards, dones}; reset() does NOT reset the sub-envs, it returns their cached original
// observations; get_original_obs/render/get_time are "not implemented" as in the reference.
// The synchronisation is a generation-counter barrier (one mutex, two condition variables) instead of the
// reference's per-slot mutex/condvar scheme.  get_observation_space_size() returns the OBSERVATION size
// (the reference returns the action size, vec_env.hpp:90-92 — a harmless bug at 18/18, not reproduced).
#ifndef PPO_B200_VEC_ENV_HPP
#define PPO_B200_VEC_ENV_HPP

#include <cassert>
#include <condition_variable>
#include <iostream>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

#include "env.hpp"

class VecEnv : public virtual Env {
public:
    explicit VecEnv(const std::vector<std::shared_ptr<Env>>& envs)
        : envs{envs},
          cached_actions{Mat::Zero(static_cast<int>(envs.size()), envs.empty() ? 0 : envs[0]->get_action_space_size())},
          observations{Mat::Zero(static_cast<int>(envs.size()), envs.empty() ? 0 : envs[0]->get_observation_space_size())},
          rewards{Mat::Zero(static_cast<int>(envs.size()), 1)},
          dones{Mat::Zero(static_cast<int>(envs.size()), 1)},
          original_rewards{Mat::Zero(static_cast<int>(envs.size()), 1)} {
        assert(!envs.empty());
        pending = static_cast<int>(envs.size());
        for (size_t i = 0; i < envs.size(); ++i) threads.emplace_back(&VecEnv::worker, this, static_cast<int>(i));
        std::unique_lock<std::mutex> l(m);
        all_done.wait(l, [this] { return pending == 0; });  // every sub-env has been reset once
    }
    VecEnv(const VecEnv&) = delete;
    VecEnv& operator=(const VecEnv&) = delete;
    ~VecEnv() override {
        {
            std::lock_guard<std::mutex> l(m);
            terminate = true;
            ++generation;
        }
        go.notify_all();
        for (auto& t : threads) t.join();
    }

    std::string get_action_space() override { return envs[0]->get_action_space(); }
    std::string get_observation_space() override { return envs[0]->get_observation_space(); }
    int get_action_space_size() override { return envs[0]->get_action_space_size(); }
    std::vector<int> get_action_space_nvec() override { return envs[0]->get_action_space_nvec(); }
    bool has_action_mask() override { return envs[0]->has_action_mask(); }
    // row i: sub-env i's mask (read between steps, when no worker touches the envs)
    Mat get_action_mask() override {
        Mat result = Mat::Zero(get_num_envs(), get_action_space_size());
        for (size_t i = 0; i < envs.size(); ++i) result.set_row(static_cast<int>(i), envs[i]->get_action_mask());
        return result;
    }
    int get_observation_space_size() override { return envs[0]->get_observation_space_size(); }
    int get_num_envs() override { return static_cast<int>(envs.size()); }

    Mat reset() override {
        Mat result = Mat::Zero(get_num_envs(), get_observation_space_size());
        for (size_t i = 0; i < envs.size(); ++i) result.set_row(static_cast<int>(i), envs[i]->get_original_obs());
        return result;
    }

    std::vector<Mat> step(const Mat& actions) override {
        assert(actions.rows() == get_num_envs());
        {
            std::lock_guard<std::mutex> l(m);
            cached_actions = actions;
            pending = get_num_envs();
            ++generation;
        }
        go.notify_all();
        std::unique_lock<std::mutex> l(m);
        all_done.wait(l, [this] { return pending == 0; });
        return {observations, rewards, dones};
    }

    Mat get_original_obs() override {
        std::cout << "VecEnv::get_original_obs() not implemented\n";
        assert(false);
        return Mat::Zero(get_num_envs(), get_observation_space_size());
    }
    Mat get_original_rew() override { return original_rewards; }
    void serialize(nlohmann::json&) override {}
    void deserialize(nlohmann::json&) override {}
    void render() override {
        std::cout << "VecEnv::render() not implemented\n";
        assert(false);
    }
    float get_time() override {
        std::cout << "VecEnv::get_time() not implemented\n";
        assert(false);
        return -1;
    }

private:
    const std::vector<std::shared_ptr<Env>>& envs;
    std::vector<std::thread> threads;
    std::mutex m;
    std::condition_variable go, all_done;
    unsigned long generation = 0;
    int pending = 0;
    bool terminate = false;
    Mat cached_actions, observations, rewards, dones, original_rewards;

    void finish_one() {
        bool last;
        {
            std::lock_guard<std::mutex> l(m);
            last = (--pending == 0);
        }
        if (last) all_done.notify_one();
    }

    void worker(int id) {
        envs[id]->reset();
        unsigned long seen = 0;
        finish_one();
        for (;;) {
            Mat action;
            {
                std::unique_lock<std::mutex> l(m);
                go.wait(l, [&] { return generation != seen; });
                seen = generation;
                if (terminate) return;
                action = cached_actions.row(id);
            }
            auto res = envs[id]->step(action);  // each worker touches only envs[id] and row id of the outputs
            observations.set_row(id, res[0]);
            rewards.set_row(id, res[1]);
            dones.set_row(id, res[2]);
            original_rewards.set_row(id, envs[id]->get_original_rew());
            finish_one();
        }
    }
};

#endif
