/* swb_jni.c -- JNI shim between the reference's JVM (Java 1.8, Spark 1.5.2 -- pom.xml:17-32) and libswb200.
 *
 * One native method per C-ABI entry a Java host needs (include/swb200.h); the Java side is java/sw/NativeSW.java
 * (`static native` methods of class sw.NativeSW, `System.loadLibrary("swbjni")`).  Handles cross as jlong, sequences
 * as Latin-1 byte[] + long[] offsets (n + 1 entries), results come back as primitive arrays.  A non-zero status
 * becomes an unchecked java.lang.RuntimeException carrying swb_last_error(): Function3.call declares no checked
 * exception (reference SmithWaterman.java:62).
 *
 * Build (on a host with a JDK):
 *   gcc -shared -fPIC -O2 -I$JAVA_HOME/include -I$JAVA_HOME/include/linux -Iinclude jni/swb_jni.c \
 *       -Lsparksmithwaterman_b200/_lib -lswb200 -Wl,-rpath,'$ORIGIN' -o libswbjni.so
 * Without a JDK the file is still compiled and link-checked against tests/jni_stub/jni.h (-DSWB_JNI_USE_STUB
 * -Itests/jni_stub): symbol names and argument lists are verified against NativeSW.java by
 * tests/test_abi_and_host.py.  That object is not loadable into a JVM. */
#include <jni.h>
#include <stdlib.h>
#include <string.h>

#include "swb200.h"

#define H(type, x) ((type *)(intptr_t)(x))

static void throw_last(JNIEnv *e, const char *fallback)
{
    const char *m = swb_last_error();
    (*e)->ThrowNew(e, (*e)->FindClass(e, "java/lang/RuntimeException"), (m && *m) ? m : fallback);
}

static jintArray ints(JNIEnv *e, const int32_t *p, int64_t n)
{
    if (n < 0 || n > 0x7fffffff) { (*e)->ThrowNew(e, (*e)->FindClass(e, "java/lang/RuntimeException"), "result array exceeds a Java array"); return 0; }
    jintArray a = (*e)->NewIntArray(e, (jsize)n);
    if (a && n && p) (*e)->SetIntArrayRegion(e, a, 0, (jsize)n, (const jint *)p);
    return a;
}

static jlongArray longs(JNIEnv *e, const int64_t *p, int64_t n)
{
    if (n < 0 || n > 0x7fffffff) { (*e)->ThrowNew(e, (*e)->FindClass(e, "java/lang/RuntimeException"), "result array exceeds a Java array"); return 0; }
    jlongArray a = (*e)->NewLongArray(e, (jsize)n);
    if (a && n && p) (*e)->SetLongArrayRegion(e, a, 0, (jsize)n, (const jlong *)p);
    return a;
}

/* ---- context ------------------------------------------------------------------------------------ */
JNIEXPORT jstring JNICALL Java_sw_NativeSW_lastError(JNIEnv *e, jclass c) { (void)c; return (*e)->NewStringUTF(e, swb_last_error()); }
JNIEXPORT jint JNICALL Java_sw_NativeSW_deviceCount(JNIEnv *e, jclass c) { (void)e; (void)c; return swb_device_count(); }

JNIEXPORT jlong JNICALL Java_sw_NativeSW_create(JNIEnv *e, jclass c, jint device, jlong workspaceBytes)
{
    (void)c;
    swb_ctx *ctx = 0;
    if (swb_create(device, workspaceBytes, &ctx)) { throw_last(e, "swb_create"); return 0; }
    return (jlong)(intptr_t)ctx;
}
JNIEXPORT void JNICALL Java_sw_NativeSW_destroy(JNIEnv *e, jclass c, jlong ctx) { (void)e; (void)c; swb_destroy(H(swb_ctx, ctx)); }

/* ---- reference set: InOutOps.GetRefSeqs' ref[1] strings (InOutOps.java:100-169) ---------------------- */
JNIEXPORT jlong JNICALL Java_sw_NativeSW_refsetLoad(JNIEnv *e, jclass c, jlong ctx, jbyteArray bytes, jlongArray offsets)
{
    (void)c;
    const jsize n = (*e)->GetArrayLength(e, offsets) - 1;
    jlong *o = (jlong *)(*e)->GetPrimitiveArrayCritical(e, offsets, 0);
    jbyte *b = (jbyte *)(*e)->GetPrimitiveArrayCritical(e, bytes, 0);
    swb_refset *rs = 0;
    const int rc = swb_refset_load(H(swb_ctx, ctx), n, (const char *)b, (const int64_t *)o, &rs);
    (*e)->ReleasePrimitiveArrayCritical(e, bytes, b, JNI_ABORT);
    (*e)->ReleasePrimitiveArrayCritical(e, offsets, o, JNI_ABORT);
    if (rc) { throw_last(e, "swb_refset_load"); return 0; }
    return (jlong)(intptr_t)rs;
}
JNIEXPORT void JNICALL Java_sw_NativeSW_refsetFree(JNIEnv *e, jclass c, jlong rs) { (void)e; (void)c; swb_refset_free(H(swb_refset, rs)); }

/* ---- align: the loop body of Distribution.MapRef.call (Distribution.java:419-426) for all refs x reads --- */
JNIEXPORT jlong JNICALL Java_sw_NativeSW_align(JNIEnv *e, jclass c, jlong ctx, jlong refset, jbyteArray readBytes,
                                               jlongArray readOffsets, jint match, jint mismatch, jint gap, jint flags)
{
    (void)c;
    const jsize n = (*e)->GetArrayLength(e, readOffsets) - 1;
    jlong *o = (jlong *)(*e)->GetPrimitiveArrayCritical(e, readOffsets, 0);
    jbyte *b = (jbyte *)(*e)->GetPrimitiveArrayCritical(e, readBytes, 0);
    swb_result *res = 0;
    const int rc = swb_align(H(swb_ctx, ctx), H(swb_refset, refset), n, (const char *)b, (const int64_t *)o, match, mismatch,
                             gap, (uint32_t)flags, &res);
    (*e)->ReleasePrimitiveArrayCritical(e, readBytes, b, JNI_ABORT);
    (*e)->ReleasePrimitiveArrayCritical(e, readOffsets, o, JNI_ABORT);
    if (rc) { throw_last(e, "swb_align"); return 0; }
    return (jlong)(intptr_t)res;
}
/* ---- hits mode: every pair scored, only each read's topK best pairs (score >= minScore) traced (swb_align_hits) ---- */
JNIEXPORT jlong JNICALL Java_sw_NativeSW_alignHits(JNIEnv *e, jclass c, jlong ctx, jlong refset, jbyteArray readBytes,
                                                   jlongArray readOffsets, jint match, jint mismatch, jint gap, jint flags,
                                                   jint topK, jint minScore)
{
    (void)c;
    const jsize n = (*e)->GetArrayLength(e, readOffsets) - 1;
    jlong *o = (jlong *)(*e)->GetPrimitiveArrayCritical(e, readOffsets, 0);
    jbyte *b = (jbyte *)(*e)->GetPrimitiveArrayCritical(e, readBytes, 0);
    swb_result *res = 0;
    const int rc = swb_align_hits(H(swb_ctx, ctx), H(swb_refset, refset), n, (const char *)b, (const int64_t *)o, match, mismatch,
                                  gap, (uint32_t)flags, topK, minScore, &res);
    (*e)->ReleasePrimitiveArrayCritical(e, readBytes, b, JNI_ABORT);
    (*e)->ReleasePrimitiveArrayCritical(e, readOffsets, o, JNI_ABORT);
    if (rc) { throw_last(e, "swb_align_hits"); return 0; }
    return (jlong)(intptr_t)res;
}
/* {score, ref, i, j} x k per read of a hits-mode result; empty for a plain one */
JNIEXPORT jintArray JNICALL Java_sw_NativeSW_resultHits(JNIEnv *e, jclass c, jlong res)
{
    (void)c;
    const swb_result *r = H(swb_result, res);
    int32_t k = 0;
    const int32_t *h = swb_result_hits(r, &k);
    return ints(e, h, h ? swb_result_n_reads(r) * k * 4 : 0);
}
/* ---- all-hits mode: every pair within `margin` of the read's best score (and >= minScore) traced (swb_align_all_hits) ---- */
JNIEXPORT jlong JNICALL Java_sw_NativeSW_alignAllHits(JNIEnv *e, jclass c, jlong ctx, jlong refset, jbyteArray readBytes,
                                                      jlongArray readOffsets, jint match, jint mismatch, jint gap, jint flags,
                                                      jint minScore, jint margin)
{
    (void)c;
    const jsize n = (*e)->GetArrayLength(e, readOffsets) - 1;
    jlong *o = (jlong *)(*e)->GetPrimitiveArrayCritical(e, readOffsets, 0);
    jbyte *b = (jbyte *)(*e)->GetPrimitiveArrayCritical(e, readBytes, 0);
    swb_result *res = 0;
    const int rc = swb_align_all_hits(H(swb_ctx, ctx), H(swb_refset, refset), n, (const char *)b, (const int64_t *)o, match,
                                      mismatch, gap, (uint32_t)flags, minScore, margin, &res);
    (*e)->ReleasePrimitiveArrayCritical(e, readBytes, b, JNI_ABORT);
    (*e)->ReleasePrimitiveArrayCritical(e, readOffsets, o, JNI_ABORT);
    if (rc) { throw_last(e, "swb_align_all_hits"); return 0; }
    return (jlong)(intptr_t)res;
}
/* n_reads + 1 offsets into resultHitList of an all-hits result; empty for any other */
JNIEXPORT jlongArray JNICALL Java_sw_NativeSW_resultHitOffsets(JNIEnv *e, jclass c, jlong res)
{
    (void)c;
    const swb_result *r = H(swb_result, res);
    int64_t n = 0;
    const int64_t *off = swb_result_hit_offsets(r, &n);
    return longs(e, off, off ? swb_result_n_reads(r) + 1 : 0);
}
/* {score, ref, i, j} per listed pair of an all-hits result, read by read; empty for any other */
JNIEXPORT jintArray JNICALL Java_sw_NativeSW_resultHitList(JNIEnv *e, jclass c, jlong res)
{
    (void)c;
    const swb_result *r = H(swb_result, res);
    int64_t n = 0;
    const int64_t *off = swb_result_hit_offsets(r, &n);
    return ints(e, swb_result_hit_list(r), off ? n * 4 : 0);
}

/* ---- one pair through the submission queue: the unchanged driver's per-pair OptAlignments.call (Distribution.java:419-426).
 * The call may wait for other threads' requests, so the bytes are copied out instead of held critical. */
JNIEXPORT jlong JNICALL Java_sw_NativeSW_alignPair(JNIEnv *e, jclass c, jlong ctx, jbyteArray ref, jbyteArray read, jint match,
                                                   jint mismatch, jint gap, jint flags)
{
    (void)c;
    const jsize n = (*e)->GetArrayLength(e, ref), m = (*e)->GetArrayLength(e, read);
    jbyte *buf = (jbyte *)malloc((size_t)n + (size_t)m + 1);
    if (!buf) { (*e)->ThrowNew(e, (*e)->FindClass(e, "java/lang/RuntimeException"), "swb_align_pair: out of memory"); return 0; }
    (*e)->GetByteArrayRegion(e, ref, 0, n, buf);
    (*e)->GetByteArrayRegion(e, read, 0, m, buf + n);
    swb_result *res = 0;
    const int rc = swb_align_pair(H(swb_ctx, ctx), (const char *)buf, n, (const char *)buf + n, m, match, mismatch, gap,
                                  (uint32_t)flags, &res);
    free(buf);
    if (rc) { throw_last(e, "swb_align_pair"); return 0; }
    return (jlong)(intptr_t)res;
}
JNIEXPORT void JNICALL Java_sw_NativeSW_resultFree(JNIEnv *e, jclass c, jlong res) { (void)e; (void)c; swb_result_free(H(swb_result, res)); }

/* ---- result arrays ------------------------------------------------------------------------------- */
JNIEXPORT jintArray JNICALL Java_sw_NativeSW_scores(JNIEnv *e, jclass c, jlong res)
{
    (void)c;
    const swb_result *r = H(swb_result, res);
    return ints(e, swb_result_scores(r), swb_result_n_refs(r) * swb_result_n_reads(r));
}
JNIEXPORT jintArray JNICALL Java_sw_NativeSW_refTotals(JNIEnv *e, jclass c, jlong res)
{
    (void)c;
    const swb_result *r = H(swb_result, res);
    return ints(e, swb_result_ref_totals(r), swb_result_n_refs(r));
}
JNIEXPORT jintArray JNICALL Java_sw_NativeSW_bestHits(JNIEnv *e, jclass c, jlong res)
{
    (void)c;
    const swb_result *r = H(swb_result, res);
    return ints(e, swb_result_best_hits(r), swb_result_n_reads(r) * 4);
}
JNIEXPORT jlongArray JNICALL Java_sw_NativeSW_cellOffsets(JNIEnv *e, jclass c, jlong res)
{
    (void)c;
    const swb_result *r = H(swb_result, res);
    return longs(e, swb_result_cell_offsets(r), swb_result_n_refs(r) * swb_result_n_reads(r) + 1);
}
JNIEXPORT jintArray JNICALL Java_sw_NativeSW_cells(JNIEnv *e, jclass c, jlong res)
{
    (void)c;
    const swb_result *r = H(swb_result, res);
    return ints(e, swb_result_cells(r), swb_result_total_cells(r) * 2);
}
JNIEXPORT jintArray JNICALL Java_sw_NativeSW_beginnings(JNIEnv *e, jclass c, jlong res)
{
    (void)c;
    const swb_result *r = H(swb_result, res);
    return ints(e, swb_result_beginnings(r), swb_result_total_cells(r));
}
JNIEXPORT jintArray JNICALL Java_sw_NativeSW_opLens(JNIEnv *e, jclass c, jlong res)
{
    (void)c;
    const swb_result *r = H(swb_result, res);
    return ints(e, swb_result_op_lens(r), swb_result_total_cells(r));
}
JNIEXPORT jlong JNICALL Java_sw_NativeSW_pairCellCount(JNIEnv *e, jclass c, jlong res, jlong pair)
{
    (void)e; (void)c;
    return swb_result_pair_cell_count(H(swb_result, res), pair);
}
/* {i, j, beginning, opLen} of the k-th max cell of pair p, in the reference's list order (SmithWaterman.java:157-185) */
JNIEXPORT jintArray JNICALL Java_sw_NativeSW_pairCell(JNIEnv *e, jclass c, jlong res, jlong pair, jlong k)
{
    (void)c;
    int32_t v[4] = {0, 0, 0, 0};
    if (swb_result_pair_cell(H(swb_result, res), pair, k, &v[0], &v[1], &v[2], &v[3])) { throw_last(e, "swb_result_pair_cell"); return 0; }
    return ints(e, v, 4);
}
/* {refAln, readAln} of materialised cell `cell`: what GetAlignment.call returns (SmithWaterman.java:418-435) */
JNIEXPORT jobjectArray JNICALL Java_sw_NativeSW_materialize(JNIEnv *e, jclass c, jlong res, jlong cell, jint opLen,
                                                            jbyteArray ref, jbyteArray read)
{
    (void)c;
    const jsize nref = (*e)->GetArrayLength(e, ref), nread = (*e)->GetArrayLength(e, read);
    char *ra = (char *)malloc((size_t)opLen + 1), *qa = (char *)malloc((size_t)opLen + 1);
    if (!ra || !qa) { free(ra); free(qa); (*e)->ThrowNew(e, (*e)->FindClass(e, "java/lang/OutOfMemoryError"), "swb_jni"); return 0; }
    jbyte *rb = (jbyte *)(*e)->GetPrimitiveArrayCritical(e, ref, 0);
    jbyte *qb = (jbyte *)(*e)->GetPrimitiveArrayCritical(e, read, 0);
    const int rc = swb_result_materialize(H(swb_result, res), cell, (const char *)rb, nref, (const char *)qb, nread, ra, qa,
                                          (int64_t)opLen + 1);
    (*e)->ReleasePrimitiveArrayCritical(e, read, qb, JNI_ABORT);
    (*e)->ReleasePrimitiveArrayCritical(e, ref, rb, JNI_ABORT);
    jobjectArray out = 0;
    if (rc) throw_last(e, "swb_result_materialize");
    else {
        out = (*e)->NewObjectArray(e, 2, (*e)->FindClass(e, "[B"), 0);
        jbyteArray a = (*e)->NewByteArray(e, opLen), b = (*e)->NewByteArray(e, opLen);
        if (out && a && b) {
            (*e)->SetByteArrayRegion(e, a, 0, opLen, (const jbyte *)ra);
            (*e)->SetByteArrayRegion(e, b, 0, opLen, (const jbyte *)qa);
            (*e)->SetObjectArrayElement(e, out, 0, a);
            (*e)->SetObjectArrayElement(e, out, 1, b);
        }
    }
    free(ra); free(qa);
    return out;
}

/* ---- multi-GPU: the reference's partition point sc.parallelize(refs) (Distribution.java:337-338) ---------- */
JNIEXPORT jlong JNICALL Java_sw_NativeSW_multiCreate(JNIEnv *e, jclass c, jintArray devices, jlong workspaceBytes)
{
    (void)c;
    const jsize n = (*e)->GetArrayLength(e, devices);
    jint *d = (jint *)(*e)->GetPrimitiveArrayCritical(e, devices, 0);
    swb_multi *m = 0;
    const int rc = swb_multi_create((const int32_t *)d, n, workspaceBytes, &m);
    (*e)->ReleasePrimitiveArrayCritical(e, devices, d, JNI_ABORT);
    if (rc) { throw_last(e, "swb_multi_create"); return 0; }
    return (jlong)(intptr_t)m;
}
JNIEXPORT void JNICALL Java_sw_NativeSW_multiDestroy(JNIEnv *e, jclass c, jlong m) { (void)e; (void)c; swb_multi_destroy(H(swb_multi, m)); }
JNIEXPORT void JNICALL Java_sw_NativeSW_multiRefsetLoad(JNIEnv *e, jclass c, jlong m, jbyteArray bytes, jlongArray offsets)
{
    (void)c;
    const jsize n = (*e)->GetArrayLength(e, offsets) - 1;
    jlong *o = (jlong *)(*e)->GetPrimitiveArrayCritical(e, offsets, 0);
    jbyte *b = (jbyte *)(*e)->GetPrimitiveArrayCritical(e, bytes, 0);
    const int rc = swb_multi_refset_load(H(swb_multi, m), n, (const char *)b, (const int64_t *)o);
    (*e)->ReleasePrimitiveArrayCritical(e, bytes, b, JNI_ABORT);
    (*e)->ReleasePrimitiveArrayCritical(e, offsets, o, JNI_ABORT);
    if (rc) throw_last(e, "swb_multi_refset_load");
}
JNIEXPORT jlongArray JNICALL Java_sw_NativeSW_multiShardRefs(JNIEnv *e, jclass c, jlong m, jint shard)
{
    (void)c;
    int64_t n = 0;
    const int64_t *ids = swb_multi_shard_refs(H(swb_multi, m), shard, &n);
    return longs(e, ids, n);
}
JNIEXPORT jlong JNICALL Java_sw_NativeSW_multiAlign(JNIEnv *e, jclass c, jlong m, jbyteArray readBytes, jlongArray readOffsets,
                                                    jint match, jint mismatch, jint gap, jint flags)
{
    (void)c;
    const jsize n = (*e)->GetArrayLength(e, readOffsets) - 1;
    jlong *o = (jlong *)(*e)->GetPrimitiveArrayCritical(e, readOffsets, 0);
    jbyte *b = (jbyte *)(*e)->GetPrimitiveArrayCritical(e, readBytes, 0);
    swb_multi_result *res = 0;
    const int rc = swb_multi_align(H(swb_multi, m), n, (const char *)b, (const int64_t *)o, match, mismatch, gap, (uint32_t)flags, &res);
    (*e)->ReleasePrimitiveArrayCritical(e, readBytes, b, JNI_ABORT);
    (*e)->ReleasePrimitiveArrayCritical(e, readOffsets, o, JNI_ABORT);
    if (rc) { throw_last(e, "swb_multi_align"); return 0; }
    return (jlong)(intptr_t)res;
}
JNIEXPORT jlong JNICALL Java_sw_NativeSW_multiAlignHits(JNIEnv *e, jclass c, jlong m, jbyteArray readBytes, jlongArray readOffsets,
                                                        jint match, jint mismatch, jint gap, jint flags, jint topK, jint minScore)
{
    (void)c;
    const jsize n = (*e)->GetArrayLength(e, readOffsets) - 1;
    jlong *o = (jlong *)(*e)->GetPrimitiveArrayCritical(e, readOffsets, 0);
    jbyte *b = (jbyte *)(*e)->GetPrimitiveArrayCritical(e, readBytes, 0);
    swb_multi_result *res = 0;
    const int rc = swb_multi_align_hits(H(swb_multi, m), n, (const char *)b, (const int64_t *)o, match, mismatch, gap, (uint32_t)flags,
                                        topK, minScore, &res);
    (*e)->ReleasePrimitiveArrayCritical(e, readBytes, b, JNI_ABORT);
    (*e)->ReleasePrimitiveArrayCritical(e, readOffsets, o, JNI_ABORT);
    if (rc) { throw_last(e, "swb_multi_align_hits"); return 0; }
    return (jlong)(intptr_t)res;
}
JNIEXPORT jlong JNICALL Java_sw_NativeSW_multiShard(JNIEnv *e, jclass c, jlong mres, jint shard)
{
    (void)e; (void)c;
    return (jlong)(intptr_t)swb_multi_result_shard(H(swb_multi_result, mres), shard);
}
JNIEXPORT jintArray JNICALL Java_sw_NativeSW_multiBestHits(JNIEnv *e, jclass c, jlong mres, jint nReads)
{
    (void)c;
    return ints(e, swb_multi_result_best_hits(H(swb_multi_result, mres)), (int64_t)nReads * 4);
}
/* merged {score, global ref, i, j} x k per read of a hits-mode multi result; empty for a plain one */
JNIEXPORT jintArray JNICALL Java_sw_NativeSW_multiResultHits(JNIEnv *e, jclass c, jlong mres, jint nReads)
{
    (void)c;
    int32_t k = 0;
    const int32_t *h = swb_multi_result_hits(H(swb_multi_result, mres), &k);
    return ints(e, h, h ? (int64_t)nReads * k * 4 : 0);
}
JNIEXPORT void JNICALL Java_sw_NativeSW_multiResultFree(JNIEnv *e, jclass c, jlong mres) { (void)e; (void)c; swb_multi_result_free(H(swb_multi_result, mres)); }
