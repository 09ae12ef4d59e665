// Host interface of the run-time compiled user-model kernels (user_model.cu).
#pragma once
#include <cstdint>
#include <string>

#include <cuda_runtime.h>

#include "../../include/glabc.h"
#include "dist_device.cuh"

namespace glabc {

// compile (or fetch from the process-wide cache) the step kernels specialised for `um` and the glabc_dist_kind of the
// Local (lp_kind) and Global / Importance (gp_kind) proposals; *fn is a CUfunction
// kind: 0 = GlobalMCMC step, 1 = GLMCMC (iSIR) step, 2 = GLMALA step
int user_model_compile(int device, int cc, const glabc_user_model_t& um, int lp_kind, int gp_kind, int kind, void** fn, std::string& err);
// compile only (needs NVRTC, no driver / GPU): validates a model's source; err receives the NVRTC log
int user_model_check(int cc, const glabc_user_model_t& um, int lp_kind, int gp_kind, std::string& err);
int user_model_launch(void* fn, const UserRun& R, int block, cudaStream_t st, std::string& err);
// glabc_k_eval_user of `um`, from any module already loaded for the model whatever its proposal kinds, else from the
// (DiagGaussian, DiagGaussian) module, compiled here
int user_model_eval_fn(int device, int cc, const glabc_user_model_t& um, void** fn, std::string& err);
int user_model_eval_launch(void* fn, const UserEval& E, int sm_count, cudaStream_t st, std::string& err);

}  // namespace glabc
