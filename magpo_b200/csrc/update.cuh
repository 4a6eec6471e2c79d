// Pieces of the update step (rec_magpo.py:214-499) shared between loss.cu and update.cu.
#pragma once
#include "kernels.cuh"

namespace magpo {

// Per-slot mean / population std of the un-normalised advantages of one minibatch (rec_magpo.py:283,356).
int adv_stats(cudaStream_t s, int T, int B, int A, const float* adv, const int32_t* env_index, int n_env, int U,
              double* acc, float* stats);

int magpo_losses(cudaStream_t s, int64_t R, int N, int A, int a, const MagpoSysCfg* sys, float inv_tokens,
                 const float* lg, const float* ll, const uint8_t* mask, const int32_t* action, const float* logp_old,
                 const float* adv, const float* value, const float* value_old, const float* targets,
                 const int32_t* env_slot, const float* stats, float* dlg, float* dll, float* dvalue, float* loss_sums);

// env_index / hs_index / env_slot of every minibatch of an epoch, laid out [M][U][E/M] (rec_magpo.py:439-451)
int epoch_index(cudaStream_t s, int E, int U, int M, const int32_t* batch_perm, int32_t* hs_perm, int first_epoch, int32_t* hs_perm_new,
                int32_t* env_index, int32_t* hs_index, int32_t* env_slot);
// The per-token rows of n_env envs of the trajectory, time-major [T, n_env, A, ...]; agent_perm NULL: agents in order.
int pack_rows(cudaStream_t s, const MagpoNetCfg* net, const MagpoSysCfg* sys, const MagpoTrajectory& traj, const float* advantages,
              const float* targets, const int32_t* env_index, const int32_t* agent_perm, int n_env, const MagpoMinibatch& out);

// guider / learner work may run on forked streams (magpo_debug_set_overlap)
bool nets_overlap_enabled();

}  // namespace magpo
