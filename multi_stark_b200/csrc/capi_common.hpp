// Shared by the translation units that define extern "C" entry points.
#pragma once
#include "../../include/msgpu.h"
#include "internal.hpp"

struct msgpu_ctx {
    msg::Ctx c;
};

namespace msg {
void set_last_error(const std::string& s);

template <class F>
static int guard(F&& f) {
    try {
        f();
        return MSGPU_OK;
    } catch (const Error& e) {
        set_last_error(e.what());
        return e.code;
    } catch (const std::exception& e) {
        set_last_error(e.what());
        return MSGPU_ERR_INTERNAL;
    } catch (...) {
        set_last_error("unknown error");
        return MSGPU_ERR_INTERNAL;
    }
}
}  // namespace msg
