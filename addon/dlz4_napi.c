/* dlz4_napi.c -- Node-API addon over the C ABI of include/dlz4_b200.h: the binding a maintainer of divortio-lz4 adds so that
 * the files under src/block and src/buffer, src/xxhash32/xxhash32.js and the worker client call the GPU (INTEGRATION.md 1-3).
 *
 * Status: type-checked only (`make -C addon syntax`, against node_api_stub.h) -- node and <node_api.h> do not exist in the
 * build image, so this file has never been loaded by a JS engine.  Real build: `make -C addon addon NODE_INC=<node>/include/node`.
 *
 * Exports (argument order = the reference's):
 *   compressBlock(src, output, srcStart, srcLen, hashTable, outputOffset) -> bytes          blockCompress.js:31
 *   decompressBlock(input, inputOffset, inputSize, output, outputOffset, dictionary) -> n   blockDecompress.js:30
 *   frameCompress(input, dict, maxBlockSize, blockIndependence, contentChecksum, addContentSize, output, blockChecksum) -> n
 *                                                                                           bufferCompress.js:100
 *   frameDecompress(input, dict, flags) -> Uint8Array                                       bufferDecompress.js:51
 *   xxHash32(input, seed) -> u32                                                            xxhash32.js:21
 *   frameCompressAsync / frameDecompressAsync(...) -> Promise                               workerClient.js:114-152 (LZ4Worker)
 *   allocPinned(bytes) -> Uint8Array over page-locked memory                                (outputBuffer at the full PCIe rate)
 *   compressBatch(src, srcOff, srcLen, dict, maxBlockSize, blockIndependence, contentChecksum, addContentSize, output,
 *                 blockChecksum, frameOff) -> total bytes        frameCompress once per message, one GPU pass (many messages)
 *   decompressBatch(src, frameOff, frameLen, dict, flags, output, dstOff, dstCap, outLen, status) -> first non-zero status
 *                                                              frameDecompress once per frame; per-frame statuses in `status`
 *   (offsets / lengths / capacities of the batch calls are BigUint64Array, srcLen a Uint32Array, status a Uint8Array)
 */
#ifdef DLZ4_NAPI_SYNTAX_ONLY
#include "node_api_stub.h"
#else
#include <node_api.h>
#endif
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "dlz4_b200.h"

static dlz4_ctx *g_ctx;        /* sync calls; one context per process -- the reference is non-re-entrant too (GLOBAL_HASH_TABLE,
                                  bufferCompress.js:55) */
static dlz4_ctx *g_worker_ctx; /* async calls run on libuv pool threads with their own streams and scratch (workerClient.js:28-35:
                                  one worker); serialised by the queue below */

static void message_for(char *msg, size_t cap, dlz4_ctx *ctx, int st, int version) {
    if (st == DLZ4_E_BAD_VERSION) snprintf(msg, cap, "%s %d", dlz4_strerror(st), version);        /* bufferDecompress.js:67 */
    else snprintf(msg, cap, "%s", st == DLZ4_E_CUDA ? dlz4_last_error(ctx) : dlz4_strerror(st));
}

static napi_value fail(napi_env env, int st, int version) {
    char msg[600];
    message_for(msg, sizeof msg, g_ctx, st, version);
    napi_throw_error(env, NULL, msg);
    return NULL;
}

/* Uint8Array / Buffer -> pointer, no copy; null / undefined -> (NULL, 0) */
static int u8(napi_env env, napi_value v, uint8_t **p, size_t *n) {
    napi_valuetype vt;
    bool is_ta = false;
    *p = NULL;
    *n = 0;
    if (napi_typeof(env, v, &vt) != napi_ok) return 0;
    if (vt == napi_undefined || vt == napi_null) return 1;
    if (napi_is_typedarray(env, v, &is_ta) != napi_ok || !is_ta) return 0;
    napi_typedarray_type t;
    napi_value ab;
    size_t off;
    return napi_get_typedarray_info(env, v, &t, n, (void **)p, &ab, &off) == napi_ok;
}

#define ARGS(N)                                                       \
    napi_value a[N];                                                  \
    size_t argc = N;                                                  \
    if (napi_get_cb_info(env, info, &argc, a, NULL, NULL) != napi_ok) return NULL
#define BAD_ARG() (napi_throw_error(env, NULL, "dlz4: invalid argument"), (napi_value)NULL)

static napi_value CompressBlock(napi_env env, napi_callback_info info) {
    ARGS(6);
    uint8_t *src, *out;
    size_t nsrc, nout, nt, boff;
    int32_t start = 0, len = 0, ooff = 0, written = 0;
    int32_t *table = NULL;
    napi_typedarray_type tt;
    napi_value ab;
    if (argc < 5 || !u8(env, a[0], &src, &nsrc) || !u8(env, a[1], &out, &nout)) return BAD_ARG();
    napi_get_value_int32(env, a[2], &start);
    napi_get_value_int32(env, a[3], &len);
    if (napi_get_typedarray_info(env, a[4], &tt, &nt, (void **)&table, &ab, &boff) != napi_ok || tt != napi_int32_array || nt < 16384)
        return BAD_ARG();                                                       /* Int32Array(16384), in/out (bufferCompress.js:55) */
    if (argc > 5) napi_get_value_int32(env, a[5], &ooff);
    int st = dlz4_compress_block(g_ctx, src, nsrc, start, len, table, out, nout, ooff, &written);
    if (st) return fail(env, st, 0);
    napi_value r;
    napi_create_int32(env, written, &r);
    return r;
}

static napi_value DecompressBlock(napi_env env, napi_callback_info info) {
    ARGS(6);
    uint8_t *in, *out, *dict = NULL;
    size_t nin, nout, nd = 0;
    int64_t ioff = 0, isz = 0, ooff = 0, written = 0;
    if (argc < 5 || !u8(env, a[0], &in, &nin) || !u8(env, a[3], &out, &nout)) return BAD_ARG();
    napi_get_value_int64(env, a[1], &ioff);
    napi_get_value_int64(env, a[2], &isz);
    napi_get_value_int64(env, a[4], &ooff);
    if (argc > 5 && !u8(env, a[5], &dict, &nd)) return BAD_ARG();
    int st = dlz4_decompress_block(g_ctx, in, nin, ioff, isz, out, nout, ooff, dict, nd, &written);
    if (st) return fail(env, st, 0);
    napi_value r;
    napi_create_int64(env, written, &r);
    return r;
}

static int frame_opts(napi_env env, napi_value *a, size_t argc, dlz4_frame_opts *o) {
    bool b = false;
    uint32_t mbs = 4194304;
    memset(o, 0, sizeof *o);
    napi_get_value_uint32(env, a[2], &mbs);
    o->max_block_size = mbs;
    napi_get_value_bool(env, a[3], &b);
    o->block_independence = b;
    napi_get_value_bool(env, a[4], &b);
    o->content_checksum = b;
    napi_get_value_bool(env, a[5], &b);
    o->add_content_size = b;
    b = false;
    if (argc > 7) napi_get_value_bool(env, a[7], &b);
    o->block_checksum = b;
    return 1;
}

/* input is already a Uint8Array (ensureBuffer stays in JS, src/shared/lz4Util.js:13-33); returns the frame length.  An
 * undersized output truncates silently like the reference's typed-array stores; JS returns output.subarray(0, min(n, length)). */
static napi_value FrameCompress(napi_env env, napi_callback_info info) {
    ARGS(8);
    uint8_t *in, *dict = NULL, *out;
    size_t nin, nd = 0, nout;
    uint64_t n = 0;
    dlz4_frame_opts o;
    if (argc < 7 || !u8(env, a[0], &in, &nin) || !u8(env, a[1], &dict, &nd) || !u8(env, a[6], &out, &nout)) return BAD_ARG();
    frame_opts(env, a, argc, &o);
    int st = dlz4_frame_compress(g_ctx, in, nin, dict, nd, &o, out, nout, &n);
    if (st) return fail(env, st, 0);
    napi_value r;
    napi_create_double(env, (double)n, &r);
    return r;
}

static napi_value FrameDecompress(napi_env env, napi_callback_info info) {
    ARGS(3);
    uint8_t *in, *dict = NULL;
    size_t nin, nd = 0;
    uint32_t flags = 1;
    dlz4_frame_info_t fi;
    uint64_t n = 0;
    if (argc < 1 || !u8(env, a[0], &in, &nin)) return BAD_ARG();
    if (argc > 1 && !u8(env, a[1], &dict, &nd)) return BAD_ARG();
    if (argc > 2) napi_get_value_uint32(env, a[2], &flags);
    memset(&fi, 0, sizeof fi);
    int st = dlz4_frame_info(in, nin, &fi);
    if (st) return fail(env, st, (int)fi.version);
    void *data;
    napi_value ab, view;
    if (napi_create_arraybuffer(env, fi.max_decoded ? (size_t)fi.max_decoded : 1, &data, &ab) != napi_ok) return NULL;
    st = dlz4_frame_decompress(g_ctx, in, nin, dict, nd, flags, (uint8_t *)data, fi.max_decoded, &n);
    if (st) return fail(env, st, (int)fi.version);
    napi_create_typedarray(env, napi_uint8_array, (size_t)n, ab, 0, &view);      /* result.subarray(0, n), bufferDecompress.js:219 */
    return view;
}

/* typed array of type `want` with at least `count` elements -> pointer */
static int typed(napi_env env, napi_value v, napi_typedarray_type want, size_t count, void **p) {
    napi_typedarray_type t;
    napi_value ab;
    size_t n = 0, off = 0;
    bool is_ta = false;
    if (napi_is_typedarray(env, v, &is_ta) != napi_ok || !is_ta) return 0;
    if (napi_get_typedarray_info(env, v, &t, &n, p, &ab, &off) != napi_ok) return 0;
    return t == want && n >= count;
}

/* frameCompress over many messages (dlz4_frames_compress_batch): message i = src[srcOff[i] .. +srcLen[i]); its frame is
 * output[frameOff[i] .. frameOff[i+1]) (frameOff has n + 1 entries; output needs the sum of the messages' frame bounds). */
static napi_value CompressBatch(napi_env env, napi_callback_info info) {
    ARGS(11);
    uint8_t *src, *dict = NULL, *out;
    size_t nsrc, nd = 0, nout, n = 0;
    void *off, *len, *foff;
    napi_typedarray_type t;
    napi_value ab;
    size_t boff;
    dlz4_frame_opts o;
    if (argc < 11 || !u8(env, a[0], &src, &nsrc) || !u8(env, a[3], &dict, &nd) || !u8(env, a[8], &out, &nout)) return BAD_ARG();
    if (napi_get_typedarray_info(env, a[2], &t, &n, &len, &ab, &boff) != napi_ok || t != napi_uint32_array) return BAD_ARG();
    if (!typed(env, a[1], napi_biguint64_array, n, &off) || !typed(env, a[10], napi_biguint64_array, n + 1, &foff)) return BAD_ARG();
    frame_opts(env, a + 2, argc - 2, &o);
    int st = dlz4_frames_compress_batch(g_ctx, src, nsrc, (const uint64_t *)off, (const uint32_t *)len, (uint32_t)n, dict, (uint32_t)nd, &o,
                                        out, nout, (uint64_t *)foff);
    if (st) return fail(env, st, 0);
    napi_value r;
    napi_create_double(env, (double)((uint64_t *)foff)[n], &r);
    return r;
}

/* frameDecompress over many frames (dlz4_frames_decompress_batch): frame i = src[frameOff[i] .. +frameLen[i]) decodes to
 * output[dstOff[i] .. +dstCap[i]); outLen[i] / status[i] as frameDecompress would end (status 0 or a DLZ4_E_* code; the JS
 * side throws per frame).  Throws only for an invalid call or a CUDA failure. */
static napi_value DecompressBatch(napi_env env, napi_callback_info info) {
    ARGS(10);
    uint8_t *src, *dict = NULL, *out, *status;
    size_t nsrc, nd = 0, nout, n = 0, nst = 0;
    void *foff, *flen, *doff, *dcap, *olen;
    uint32_t flags = 1;
    if (argc < 10 || !u8(env, a[0], &src, &nsrc) || !u8(env, a[3], &dict, &nd) || !u8(env, a[5], &out, &nout) ||
        !u8(env, a[9], &status, &nst)) return BAD_ARG();
    n = nst;
    napi_get_value_uint32(env, a[4], &flags);
    if (!typed(env, a[1], napi_biguint64_array, n, &foff) || !typed(env, a[2], napi_biguint64_array, n, &flen) ||
        !typed(env, a[6], napi_biguint64_array, n, &doff) || !typed(env, a[7], napi_biguint64_array, n, &dcap) ||
        !typed(env, a[8], napi_biguint64_array, n, &olen)) return BAD_ARG();
    int st = dlz4_frames_decompress_batch(g_ctx, src, nsrc, (const uint64_t *)foff, (const uint64_t *)flen, (uint32_t)n, dict, (uint32_t)nd,
                                          flags, out, nout, (const uint64_t *)doff, (const uint64_t *)dcap, (uint64_t *)olen, status);
    if (st >= DLZ4_E_INVALID_ARG) return fail(env, st, 0);
    napi_value r;
    napi_create_double(env, (double)st, &r);
    return r;
}

static napi_value XxHash32(napi_env env, napi_callback_info info) {
    ARGS(2);
    uint8_t *in;
    size_t n;
    uint32_t seed = 0, h = 0;
    if (argc < 1 || !u8(env, a[0], &in, &n)) return BAD_ARG();
    if (argc > 1) napi_get_value_uint32(env, a[1], &seed);
    int st = dlz4_xxh32(g_ctx, in, n, seed, &h);
    if (st) return fail(env, st, 0);
    napi_value r;
    napi_create_uint32(env, h, &r);
    return r;
}

/* ---- LZ4Worker.compress / decompress (workerClient.js:114-152): a Promise per task, the work on a libuv pool thread ---- */
typedef struct {
    napi_async_work work;
    napi_deferred deferred;
    napi_ref keep[3];               /* input, dictionary, output stay alive while the task runs */
    int decompress, status, version;
    uint8_t *in, *dict, *out;
    size_t nin, nd, nout;
    uint32_t flags;
    dlz4_frame_opts opts;
    uint64_t n;
    uint8_t *result;                /* decompress: pinned buffer handed to JS as an external ArrayBuffer */
    char msg[600];
} task_t;

static void free_pinned(napi_env env, void *data, void *hint) {
    (void)env;
    (void)hint;
    dlz4_pinned_free(data);
}

static void task_execute(napi_env env, void *data) {            /* pool thread: no JS calls here */
    task_t *t = (task_t *)data;
    (void)env;
    if (!t->decompress) {
        t->status = dlz4_frame_compress(g_worker_ctx, t->in, t->nin, t->dict, t->nd, &t->opts, t->out, t->nout, &t->n);
    } else {
        dlz4_frame_info_t fi;
        memset(&fi, 0, sizeof fi);
        t->status = dlz4_frame_info(t->in, t->nin, &fi);
        t->version = (int)fi.version;
        if (!t->status) {
            t->nout = fi.max_decoded ? (size_t)fi.max_decoded : 1;
            t->result = (uint8_t *)dlz4_pinned_alloc(t->nout);
            t->status = t->result ? dlz4_frame_decompress(g_worker_ctx, t->in, t->nin, t->dict, t->nd, t->flags, t->result, fi.max_decoded, &t->n)
                                  : DLZ4_E_CUDA;
        }
    }
    if (t->status) message_for(t->msg, sizeof t->msg, g_worker_ctx, t->status, t->version);
}

static void task_complete(napi_env env, napi_status status, void *data) {
    task_t *t = (task_t *)data;
    napi_value v, msg;
    if (status != napi_ok || t->status) {
        napi_create_string_utf8(env, t->status ? t->msg : "dlz4: task cancelled", (size_t)-1, &msg);
        napi_create_error(env, NULL, msg, &v);
        if (t->result) dlz4_pinned_free(t->result);
        napi_reject_deferred(env, t->deferred, v);
    } else if (!t->decompress) {
        napi_create_double(env, (double)t->n, &v);               /* JS: output.subarray(0, min(n, output.length)) */
        napi_resolve_deferred(env, t->deferred, v);
    } else {
        napi_value ab;
        napi_create_external_arraybuffer(env, t->result, t->nout, free_pinned, NULL, &ab);
        napi_create_typedarray(env, napi_uint8_array, (size_t)t->n, ab, 0, &v);
        napi_resolve_deferred(env, t->deferred, v);
    }
    for (int i = 0; i < 3; ++i)
        if (t->keep[i]) napi_delete_reference(env, t->keep[i]);
    napi_delete_async_work(env, t->work);
    free(t);
}

static napi_value queue_task(napi_env env, task_t *t, const char *name) {
    napi_value promise, rname;
    if (napi_create_promise(env, &t->deferred, &promise) != napi_ok) { free(t); return NULL; }
    napi_create_string_utf8(env, name, (size_t)-1, &rname);
    napi_create_async_work(env, NULL, rname, task_execute, task_complete, t, &t->work);
    napi_queue_async_work(env, t->work);
    return promise;
}

static napi_value FrameCompressAsync(napi_env env, napi_callback_info info) {
    ARGS(8);
    task_t *t = (task_t *)calloc(1, sizeof *t);
    if (!t) return NULL;
    if (argc < 7 || !u8(env, a[0], &t->in, &t->nin) || !u8(env, a[1], &t->dict, &t->nd) || !u8(env, a[6], &t->out, &t->nout)) {
        free(t);
        return BAD_ARG();
    }
    frame_opts(env, a, argc, &t->opts);
    napi_create_reference(env, a[0], 1, &t->keep[0]);
    if (t->dict) napi_create_reference(env, a[1], 1, &t->keep[1]);
    napi_create_reference(env, a[6], 1, &t->keep[2]);
    return queue_task(env, t, "dlz4.compress");
}

static napi_value FrameDecompressAsync(napi_env env, napi_callback_info info) {
    ARGS(3);
    task_t *t = (task_t *)calloc(1, sizeof *t);
    if (!t) return NULL;
    t->decompress = 1;
    t->flags = 1;
    if (argc < 1 || !u8(env, a[0], &t->in, &t->nin) || (argc > 1 && !u8(env, a[1], &t->dict, &t->nd))) {
        free(t);
        return BAD_ARG();
    }
    if (argc > 2) napi_get_value_uint32(env, a[2], &t->flags);
    napi_create_reference(env, a[0], 1, &t->keep[0]);
    if (t->dict) napi_create_reference(env, a[1], 1, &t->keep[1]);
    return queue_task(env, t, "dlz4.decompress");
}

static napi_value AllocPinned(napi_env env, napi_callback_info info) {
    ARGS(1);
    int64_t n = 0;
    if (argc < 1 || napi_get_value_int64(env, a[0], &n) != napi_ok || n < 0) return BAD_ARG();
    void *p = dlz4_pinned_alloc((uint64_t)n);
    if (!p) return fail(env, DLZ4_E_CUDA, 0);
    napi_value ab, view;
    napi_create_external_arraybuffer(env, p, (size_t)n, free_pinned, NULL, &ab);
    napi_create_typedarray(env, napi_uint8_array, (size_t)n, ab, 0, &view);
    return view;
}

NAPI_MODULE_INIT() {
    /* no CPU fallback: without a CUDA device the module fails to load */
    if (dlz4_init(0, &g_ctx) != DLZ4_OK || dlz4_init(0, &g_worker_ctx) != DLZ4_OK) {
        napi_throw_error(env, NULL, dlz4_last_error(g_ctx));
        return NULL;
    }
    napi_property_descriptor d[] = {
        {"compressBlock", 0, CompressBlock, 0, 0, 0, napi_default, 0},
        {"decompressBlock", 0, DecompressBlock, 0, 0, 0, napi_default, 0},
        {"frameCompress", 0, FrameCompress, 0, 0, 0, napi_default, 0},
        {"frameDecompress", 0, FrameDecompress, 0, 0, 0, napi_default, 0},
        {"xxHash32", 0, XxHash32, 0, 0, 0, napi_default, 0},
        {"frameCompressAsync", 0, FrameCompressAsync, 0, 0, 0, napi_default, 0},
        {"frameDecompressAsync", 0, FrameDecompressAsync, 0, 0, 0, napi_default, 0},
        {"allocPinned", 0, AllocPinned, 0, 0, 0, napi_default, 0},
        {"compressBatch", 0, CompressBatch, 0, 0, 0, napi_default, 0},
        {"decompressBatch", 0, DecompressBatch, 0, 0, 0, napi_default, 0},
    };
    napi_define_properties(env, exports, sizeof d / sizeof d[0], d);
    return exports;
}
