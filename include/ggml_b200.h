/* ggml_b200.h -- C ABI of the B200-native compute library (libggml_b200_kernels.so).
 *
 * This is the drop-in boundary for cortex.llamacpp's hot path: everything ggml's backend
 * vtables (reference: llama.cpp/ggml/src/ggml-backend-impl.h:17-207) need from a device is
 * expressed here with plain pointers and sizes.  The C++ ggml backend in
 * cortex.llamacpp_b200/backend/ggml-b200.cpp is a thin translation of
 * ggml_backend_{reg,device,buffer_type,buffer}_i / ggml_backend_i onto these calls;
 * tests and bench.py bind the same symbols through ctypes.
 *
 * Conventions
 *   - every function returns B200_OK (0) or a negative b200_status unless it returns a handle;
 *     no exceptions cross this boundary (ggml convention: alloc -> NULL, compute -> status).
 *   - tensors are described exactly like ggml_tensor (ggml/include/ggml.h:578-610):
 *     type id, ne[4] elements, nb[4] BYTE strides, device pointer.
 *   - type ids are ggml's own enum values (ggml.h:350-390) so descriptors can be copied 1:1.
 *   - op ids are OUR enum (ggml's op enum shifts between versions); op_params carry the same
 *     int32/float words as ggml_tensor::op_params for that op (SURVEY.md appendix C).
 */
#ifndef GGML_B200_H
#define GGML_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_API __attribute__((visibility("default")))
#define B200_ABI_VERSION 1

typedef enum b200_status {
    B200_OK             = 0,
    B200_ERR_ALLOC      = -1,   /* -> GGML_STATUS_ALLOC_FAILED */
    B200_ERR_FAILED     = -2,   /* -> GGML_STATUS_FAILED       */
    B200_ERR_UNSUPPORTED= -3,   /* op/shape not implemented: caller must have asked b200_supports_op first */
    B200_ERR_NO_DEVICE  = -4,
} b200_status;

/* ggml_type values (ggml.h:350-390) */
typedef enum b200_type {
    B200_TYPE_F32 = 0, B200_TYPE_F16 = 1, B200_TYPE_Q4_0 = 2, B200_TYPE_Q8_0 = 8,
    B200_TYPE_Q4_K = 12, B200_TYPE_Q5_K = 13, B200_TYPE_Q6_K = 14, B200_TYPE_Q8_K = 15,
    B200_TYPE_I32 = 26, B200_TYPE_BF16 = 30,
} b200_type;

/* ops on the hot path (SURVEY.md 8b "minimum op set"); replaces the op switch of
 * ggml_cuda_compute_forward (ggml-cuda.cu:2100-2332) */
typedef enum b200_op_id {
    B200_OP_NONE = 0,
    B200_OP_MUL_MAT,         /* src0 W [K,N,..] any type, src1 f32 [K,M,..] -> f32 [N,M,..]          (mmvq.cu / mmq.cuh) */
    B200_OP_MUL_MAT_ID,      /* src0 as [K,N,E], src1 b f32 [K,nu|1,T], src2 ids i32 [nu,T]           (ggml-cuda.cu:1962)  */
    B200_OP_FLASH_ATTN_EXT,  /* src0 q f32, src1 k, src2 v, src3 mask f16 (optional)                   (fattn*.cu*)         */
    B200_OP_RMS_NORM,        /* params[0] = eps (f32 bits)                                             (norm.cu:107)        */
    B200_OP_ROPE,            /* src1 pos i32, src2 freq factors (optional); params as ggml             (rope.cu)            */
    B200_OP_CPY,             /* src0 -> dst layout/type (f32->f32/f16/q8_0/q4_0, f16->f16/f32, q->f32) (cpy.cu)             */
    B200_OP_CONT,            /* same-type strided -> contiguous                                        (cpy.cu)             */
    B200_OP_ADD, B200_OP_SUB, B200_OP_MUL, B200_OP_DIV,   /* broadcasting src1 over src0               (binbcast.cu)        */
    B200_OP_SILU, B200_OP_GELU, B200_OP_RELU, B200_OP_TANH, B200_OP_SIGMOID, /* unary                  (unary.cu)           */
    B200_OP_GET_ROWS,        /* src0 rows (f32/f16/q*), src1 i32 idx -> f32                            (getrows.cu)         */
    B200_OP_SOFT_MAX,        /* params[0]=scale params[1]=max_bias; src1 mask f16/f32 optional         (softmax.cu)         */
    B200_OP_ARGSORT,         /* params[0] order (0 asc, 1 desc) -> i32                                 (argsort.cu)         */
    B200_OP_SUM_ROWS,        /*                                                                        (sumrows.cu)         */
    B200_OP_SCALE,           /* params[0] = scale                                                      (scale.cu)           */
    B200_OP_SWIGLU_FUSED,    /* dst = silu(src0) * src1 (fusion of UNARY(SILU)+MUL emitted by the backend's matcher)        */
    B200_OP_RMS_NORM_MUL,    /* dst = rms_norm(src0) * src1  (fusion of RMS_NORM+MUL)                                       */
    B200_OP_ALLREDUCE,       /* dst = sum over tensor-parallel ranks of src0 (+ src1 residual, optional); f32, contiguous:   */
                             /* the exchange that replaces ggml_cuda_op_mul_mat's row gather (ggml-cuda.cu:1363-1671)        */
    B200_OP_ARGMAX,          /* src0 f32 [n, rows] -> i32 [rows]: index of the LAST maximum of each row      (argmax.cu; ggml-cpu.c:2393) */
    B200_OP_COUNT
} b200_op_id;

#define B200_MAX_SRC 4
#define B200_TENSOR_FLAG_WEIGHT 1u   /* tensor lives in a weights buffer: constant across graph launches */
/* src0 of a MUL_MAT is a row-split weight (ggml_backend_split_buffer_type, ggml-cuda.cu:723-1050): `data` points to a b200_split in
 * host memory owned by the caller; device d holds rows [row_low[d], row_low[d+1]) of the GGUF matrix as a dense shard.  The matmul runs
 * on every shard's GPU at once and the row ranges of dst land in the main device's memory through NVLink peer stores. */
#define B200_TENSOR_FLAG_SPLIT 2u
#define B200_MAX_SPLIT 16
typedef struct b200_split {
    int32_t n_dev;
    int32_t device[B200_MAX_SPLIT];
    void *  shard[B200_MAX_SPLIT];
    int64_t row_low[B200_MAX_SPLIT + 1];
} b200_split;

typedef struct b200_tensor {
    void *   data;           /* device pointer (already offset to the tensor/view start) */
    int32_t  type;           /* b200_type */
    uint32_t flags;
    int64_t  ne[4];
    uint64_t nb[4];          /* byte strides */
} b200_tensor;

typedef struct b200_op {
    int32_t     op;                    /* b200_op_id */
    int32_t     n_src;
    int32_t     params[16];            /* ggml op_params words */
    b200_tensor dst;
    b200_tensor src[B200_MAX_SRC];
} b200_op;

typedef struct b200_ctx b200_ctx;      /* one per (device, stream): mirrors ggml_backend_cuda_context (common.cuh:730-801) */
typedef struct b200_event b200_event;

/* ---- library / device discovery (ggml_backend_reg_i / ggml_backend_device_i) ---------------- */
B200_API int         b200_abi_version(void);
B200_API int         b200_device_count(void);                         /* 0 if no sm_100 device: ggml_backend_score -> 0 */
B200_API int         b200_device_info(int device, char *name, size_t name_len, size_t *free_bytes, size_t *total_bytes,
                                      int *sm_count, int *cc_major, int *cc_minor);
B200_API const char *b200_last_error(void);                           /* thread-local message of the last failure */

/* ---- context = device + stream (ggml_backend_i: init/free/synchronize) ---------------------- */
B200_API b200_ctx *  b200_ctx_create(int device);
B200_API void        b200_ctx_destroy(b200_ctx *ctx);
B200_API int         b200_ctx_device(const b200_ctx *ctx);
B200_API void *      b200_ctx_stream(const b200_ctx *ctx);            /* cudaStream_t, for callers that time with events */
B200_API int         b200_synchronize(b200_ctx *ctx);

/* ---- memory (ggml_backend_buffer_type_i::alloc_buffer, ggml_backend_buffer_i::set/get/cpy/clear) */
B200_API void *      b200_malloc(int device, size_t size);            /* NULL on OOM (caller handles, ggml-cuda.cu:654-660) */
B200_API void        b200_free(int device, void *ptr);
B200_API void *      b200_host_malloc(size_t size);                   /* pinned; NULL on failure */
B200_API void        b200_host_free(void *ptr);
B200_API int         b200_memset(int device, void *dst, int value, size_t size);                    /* synchronous */
B200_API int         b200_memcpy_h2d(int device, void *dst, const void *src, size_t size);          /* synchronous */
B200_API int         b200_memcpy_d2h(int device, void *dst, const void *src, size_t size);          /* synchronous */
B200_API int         b200_memcpy_d2d(int dst_device, void *dst, int src_device, const void *src, size_t size); /* synchronous, peer ok */
B200_API int         b200_memcpy_h2d_async(b200_ctx *ctx, void *dst, const void *src, size_t size);
B200_API int         b200_memcpy_d2h_async(b200_ctx *ctx, void *dst, const void *src, size_t size);
B200_API int         b200_memcpy_d2d_async(b200_ctx *ctx, void *dst, int src_device, const void *src, size_t size);
/* GGUF -> device load path (replaces the staging loop of llama_model_loader::load_all_data, llama-model-loader.cpp:895-1071): `src` is
 * pageable (mmap'd) host memory; the bytes are gathered into a ring of pinned chunks by a few host threads while the copy engine drains
 * the previous chunks.  b200_upload_slice packs rows [row0, row0 + n_rows) x bytes [col_off, col_off + col_bytes) of a row-major host
 * matrix (rows `src_row_stride` bytes apart) into a dense device buffer: the shard of a row-split / K-split weight, read once from the file. */
B200_API int         b200_upload(b200_ctx *ctx, void *dst, const void *src, size_t size);
B200_API int         b200_upload_slice(b200_ctx *ctx, void *dst, const void *src, size_t src_row_stride, int64_t row0, int64_t n_rows,
                                       size_t col_off, size_t col_bytes);
B200_API size_t      b200_alloc_size(int32_t type, const int64_t ne[4], size_t nbytes); /* padded size a tensor needs (get_alloc_size) */

/* ---- events (ggml_backend_device_i::event_*, ggml_backend_i::event_record/wait) -------------- */
B200_API b200_event *b200_event_create(int device);
B200_API void        b200_event_destroy(b200_event *ev);
B200_API int         b200_event_record(b200_ctx *ctx, b200_event *ev);
B200_API int         b200_event_wait(b200_ctx *ctx, b200_event *ev);  /* stream waits */
B200_API int         b200_event_synchronize(b200_event *ev);          /* host waits */
B200_API float       b200_event_elapsed_ms(b200_event *start, b200_event *stop);

/* ---- compute (ggml_backend_device_i::supports_op, ggml_backend_i::graph_compute) ------------- */
B200_API int         b200_supports_op(int device, const b200_op *op); /* 1 / 0 */
/* Runs ops in order on ctx's stream (asynchronous).  The library may fuse adjacent ops and
 * replay a captured CUDA graph when the same op list (pointers included) is submitted again. */
B200_API int         b200_graph_compute(b200_ctx *ctx, const b200_op *ops, int n_ops);
B200_API int         b200_op_compute(b200_ctx *ctx, const b200_op *op);   /* single op, no fusion */
B200_API int64_t     b200_kernel_launches(const b200_ctx *ctx);       /* kernels launched by this ctx so far (bench: gpu_launches) */
/* keys: "cuda_graphs", "fusion" (0 off, 1 two-op, 2 + llama layer fusions), "pdl", "cpu_exact" (parity mode: the reference CPU
 * backend's summation order; "fa_exact" is an alias), "l2_prefetch" (0 off / 1 / 2), "ffn_pair" (gate|up GEMV writes
 * silu(gate)*up; default 1), "debug_skip" (timing experiments only).  Changing one drops the captured CUDA graphs.
 * Any other key returns B200_ERR_UNSUPPORTED. */
B200_API int         b200_set_option(b200_ctx *ctx, const char *key, int value);

/* ---- tensor parallelism: one process (and one b200_ctx) per GPU ------------------------------
 * Replaces the split-buffer matmul driver ggml_cuda_op_mul_mat + ggml_backend_cuda_split_buffer_type
 * (ggml-cuda.cu:725-1050, 1363-1671) and ggml_cuda_set_peer_access (:1285-1341): weights are sharded
 * Megatron-style by the host (wq/wk/wv/gate/up by rows, wo/down by K at block boundaries) and the only
 * exchange is B200_OP_ALLREDUCE after wo and after down.  The host transports two opaque blobs between
 * its ranks (any way it likes: torch.distributed, MPI, a socket): the 128-byte communicator id of rank 0
 * and the 64-byte peer-memory handle of every rank. */
#define B200_COMM_ID_BYTES     128
#define B200_COMM_HANDLE_BYTES 64
B200_API int         b200_comm_unique_id(void *id128);                                   /* rank 0 */
B200_API int         b200_comm_init(b200_ctx *ctx, const void *id128, int rank, int world); /* collective */
B200_API int         b200_comm_peer_handle(b200_ctx *ctx, void *handle64);               /* this rank's exchange buffer */
B200_API int         b200_comm_peer_attach(b200_ctx *ctx, const void *handles);          /* world x 64 bytes, rank order */
B200_API int         b200_comm_rank(const b200_ctx *ctx);
B200_API int         b200_comm_world(const b200_ctx *ctx);
B200_API int         b200_comm_destroy(b200_ctx *ctx);

/* ---- test hooks: expose the integer stage of the quantised dot so parity can be bit-exact ---- */
/* x f32 [rows, K] (row stride K) -> act blocks in the reference's block_q8_0 / block_q8_K byte layout */
B200_API int         b200_quantize_act(b200_ctx *ctx, int32_t act_type, const float *x, void *blocks, int64_t K, int64_t rows);
/* per weight block b of every row: exact int32 P (and M for q4_K/q5_K) against ONE activation column x f32 [K] */
B200_API int         b200_block_sums(b200_ctx *ctx, int32_t type, const void *W, const float *x, int64_t N, int64_t K,
                                     int32_t *P, int32_t *M);

/* debug: device buffer of [sm_count][16] u64 receiving %globaltimer stamps from the GEMV kernel (NULL = off) */
B200_API int         b200_debug_set_prof(b200_ctx *ctx, void *device_buf);

#ifdef __cplusplus
}
#endif
#endif /* GGML_B200_H */
