// The handle behind mrb_env (private to the library; callers only see the opaque pointer).
#pragma once
#include <string>

#include "common.cuh"

constexpr int kPipeStreams = 16;

struct mrb_env {
    mrb::Params p;
    int device;
    bool bound;
    int32_t *actions_dev;       // staging for mrb_step_host
    // mrb_step_masked scratch, allocated by mrb_create: [B] active env ids, then the compaction's 3 work words.  Env
    // ids fit int32: the state rows of 2^31 envs would not fit a device.
    int32_t *step_list;
    cudaStream_t pipe[kPipeStreams];   // internal streams of the chunked host path (one per chunk)
    cudaEvent_t ev_in, ev_out[kPipeStreams];
    bool pipe_ready;
    std::string err;
};

namespace mrb {
void count_launch();
int fail(mrb_env *e, int code, const std::string &msg);          // e == nullptr: records the create error
int cuda_fail(mrb_env *e, cudaError_t st, const char *what);
}  // namespace mrb
