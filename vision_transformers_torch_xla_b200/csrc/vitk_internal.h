// vitk_internal.h — glue between the public C ABI (include/vitk.h) and the kernels.
#pragma once
#include "../../include/vitk.h"

constexpr int EPI_BF16 = VITK_EPI_BF16;
constexpr int EPI_GELU = VITK_EPI_GELU;
constexpr int EPI_RESID = VITK_EPI_RESID;
constexpr int EPI_F32 = VITK_EPI_F32;
constexpr int EPI_DGELU = VITK_EPI_DGELU;
constexpr int EPI_ATOMIC = VITK_EPI_ATOMIC;
constexpr int EPI_PATCH = VITK_EPI_PATCH;
