/*
 * rv_internal.h -- the few things other translation units of librv_b200.so (rv_fog.cu, rv_u16.cu) need from the context that rv_b200.cu
 * owns.  Not part of the C ABI (include/rv_b200.h).
 */
#pragma once
#include "../../include/rv_b200.h"

int rv_internal_device(const rv_ctx *ctx);
void *rv_internal_stream(rv_ctx *ctx);                                  /* the context's main cudaStream_t */
int rv_internal_fail(rv_ctx *ctx, int code, const char *fmt, ...);      /* records the message, returns code */
void rv_internal_count_launches(rv_ctx *ctx, long n);
void *rv_internal_get_fog(rv_ctx *ctx);
void rv_internal_set_fog(rv_ctx *ctx, void *state, void (*destroy)(void *));
void *rv_internal_get_u16(rv_ctx *ctx);
void rv_internal_set_u16(rv_ctx *ctx, void *state, void (*destroy)(void *));
