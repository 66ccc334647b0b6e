// Host interface of the Shack-Hartmann frame (wfs_frame.cu): which kernel serves a frame, the tables the staged kernels
// derive from the uploaded ones and when those go stale, and the launch of every kernel family.
#pragma once
#include <cuda_runtime.h>
#include "wfs_params.cuh"

struct WfsFrame;

// The sensor-frame state of a context of configuration c whose screen layers are screens[l] ([E][N][N], allocated for
// the context's life); err is the device error word that the bounded waits of the staged kernels raise.
// Null: out of host memory.
WfsFrame* wfs_frame_create(const aom_config& c, float* const* screens, int* err, int num_sms);
void wfs_frame_destroy(WfsFrame* s);

// Takes note of an uploaded table (aom_set_table): the staged kernels keep host copies of the tables their own derive
// from, and rebuild theirs on the next frame.  False: out of host memory.
bool wfs_frame_set_table(WfsFrame* s, int table, const void* host, size_t nbytes);

// Routes the frame p (fill_wfs_params) on sensor path `path` (aom_wfs_path), noisy when any environment draws noise in
// it, and launches its kernel on st; start, when not null, is recorded on st right before the launch.  Prepares the
// tables of a staged kernel on first use.  Returns AOM_OK, or an error code with its message in err.
int wfs_frame_launch(WfsFrame* s, const WfsParams& p, int path, bool noisy, cudaEvent_t start, cudaStream_t st,
                     char (&err)[512]);

// Name of the kernel that serves a noise-free frame without kept image on path (aom_wfs_kernel).  When the round-1
// register kernel serves it because the staged kernels refused, err says why; "" when preparing them failed (err).
const char* wfs_frame_kernel_name(WfsFrame* s, int path, char (&err)[512]);
