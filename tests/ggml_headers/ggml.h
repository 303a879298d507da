/* The part of upstream T-MAC's ggml.h (3rdparty/llama.cpp/ggml/include/ggml.h) that t-mac_b200/ggml/ggml-tmac.cpp and
 * tests/test_ggml_shim.py use, restated so that the shim can be compiled and linked in a checkout without the upstream tree:
 * the type ids (ggml.h:359,391-396) and the struct ggml_tensor fields the shim reads.  Not the whole upstream header: the
 * struct has fewer fields, so nothing built against this file may be mixed with upstream ggml objects. */
#pragma once

#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

#define GGML_API
#define GGML_MAX_DIMS 4
#define GGML_MAX_NAME 64

enum ggml_type {
    GGML_TYPE_F32 = 0,
    GGML_TYPE_F16 = 1,
    GGML_TYPE_Q4_0 = 2,
    GGML_TYPE_TQ1_0 = 34,
    GGML_TYPE_TQ2_0 = 35,
    GGML_TYPE_I1 = 36,
    GGML_TYPE_I2 = 37,
    GGML_TYPE_I3 = 38,
    GGML_TYPE_I4 = 39,
};

struct ggml_tensor {
    enum ggml_type type;
    int64_t ne[GGML_MAX_DIMS];
    size_t nb[GGML_MAX_DIMS];
    void * data;
    char name[GGML_MAX_NAME];
    void * extra;
};
