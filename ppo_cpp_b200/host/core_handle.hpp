// RAII handle around the C ABI (include/ppo_core.h).  The host classes in this directory call ONLY the
// C ABI through this handle.  Errors follow the reference's convention: print, then assert(false)
// (ppo2/ppo2.hpp:99-102, policies.hpp:39-43) — plus a std::runtime_error so that NDEBUG builds do not run on.
#ifndef PPO_B200_CORE_HANDLE_HPP
#define PPO_B200_CORE_HANDLE_HPP

#include <cassert>
#include <iostream>
#include <memory>
#include <stdexcept>
#include <string>

#include "../../include/ppo_core.h"

inline void ppo_check(int status, const char* what) {
    if (status != PPO_OK) {
        std::cout << what << " error" << std::endl;
        std::cout << ppo_last_error() << std::endl;
        assert(false);
        throw std::runtime_error(std::string(what) + ": " + ppo_last_error());
    }
}

struct CoreDeleter {
    void operator()(ppo_core* c) const { ppo_core_destroy(c); }
};
using CorePtr = std::shared_ptr<ppo_core>;

inline CorePtr make_core(const ppo_core_desc& desc, int action_space = PPO_ACTION_BOX) {
    ppo_core* raw = nullptr;
    ppo_check(ppo_core_create_ex(&desc, action_space, &raw), "ppo_core_create");
    return CorePtr(raw, CoreDeleter());
}

#endif
