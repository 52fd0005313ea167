// rt_error.hpp — the error boundary of the C-ABI, shared by every translation unit that implements rt_status entries.
// No CUDA header: rt_host.cpp is compiled by the host compiler alone.  CUDA_TRY and make_current are in rt_internal.hpp.
#pragma once

#include <exception>
#include <new>

#include "../../include/rt_api.h"

namespace rtd {
// rt_api.cu: the message rt_last_error() returns on this thread
void set_error(const char* fmt, ...) __attribute__((format(printf, 1, 2)));
void set_error_message(const char* msg);
// every parameter of a camera finite (scene descriptions, frame sequences, rt_orbit_cameras)
bool camera_finite(const rt_camera& c);
} // namespace rtd

#define ARG_CHECK(cond, msg)                             \
    do {                                                 \
        if (!(cond)) {                                   \
            rtd::set_error("invalid argument: %s", msg); \
            return RT_ERR_INVALID_ARG;                   \
        }                                                \
    } while (0)

// Every rt_status entry point that can throw is a function-try-block closed by this: nothing propagates through the C ABI
// (SURVEY.md 8b "no exceptions across the boundary"); host containers that cannot grow are RT_ERR_OOM.
#define RT_API_CATCH                                          \
    catch (const std::bad_alloc&) {                           \
        rtd::set_error("out of host memory");                 \
        return RT_ERR_OOM;                                    \
    }                                                         \
    catch (const std::exception& e) {                         \
        rtd::set_error("unexpected exception: %s", e.what()); \
        return RT_ERR_INVALID_ARG;                            \
    }
