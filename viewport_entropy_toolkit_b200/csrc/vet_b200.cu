// libvet_b200.so -- C ABI (include/vet_b200.h) over the sm_100a kernels.
// Host side: configuration validation, table construction (lattice, per-axis
// direction tables, cell->tile LUTs, FOV weight columns), scratch management and
// kernel launches.  No CPU compute path: every stage runs on the device.
// One translation unit, written as fragments under host/ (included below in dependency order):
// the kernels live in the *.cuh headers, the host logic of each stage in its own .inl file.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "vet_b200.h"
#include "vet_common.cuh"
#include "vet_stream.cuh"
#include "vet_stream_tma.cuh"
#include "vet_tables.cuh"
#include "vet_transition.cuh"
#include "vet_transition2.cuh"
#include "vet_transition3.cuh"
#include "vet_transition4.cuh"
#include "vet_vectors.cuh"
#include "vet_whist.cuh"
#include "vet_whist_i8.cuh"
#include "vet_naive.cuh"
#include "vet_users.cuh"
#include "vet_transition_counts.cuh"
#include "vet_user_transitions.cuh"

#include "host/vet_host_core.inl"
#include "host/vet_host_tables.inl"
#include "host/vet_host_spatial.inl"
#include "host/vet_api_core.inl"
#include "host/vet_api_vectors.inl"
#include "host/vet_host_transition.inl"
#include "host/vet_api_misc.inl"
#include "host/vet_api_host.inl"
#include "host/vet_host_users.inl"
#include "host/vet_host_transition_counts.inl"
#include "host/vet_host_user_transitions.inl"
