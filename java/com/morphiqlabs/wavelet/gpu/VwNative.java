package com.morphiqlabs.wavelet.gpu;

import java.lang.foreign.Arena;
import java.lang.foreign.FunctionDescriptor;
import java.lang.foreign.Linker;
import java.lang.foreign.MemorySegment;
import java.lang.foreign.SymbolLookup;
import java.lang.foreign.ValueLayout;
import java.lang.invoke.MethodHandle;

import static java.lang.foreign.ValueLayout.ADDRESS;
import static java.lang.foreign.ValueLayout.JAVA_DOUBLE;
import static java.lang.foreign.ValueLayout.JAVA_INT;
import static java.lang.foreign.ValueLayout.JAVA_LONG;

/**
 * Panama FFM (java.lang.foreign, final since JDK 22) downcall handles for libvwmodwt.so -- the C ABI declared in
 * include/vw_modwt.h.  This file is the Java twin of vectorwave_b200/_native.py (which the tests exercise through
 * ctypes); it belongs in the extensions tier (JDK 24) next to BatchMODWT.  The build image has no JDK, so it is
 * compiled only where one exists: {@code javac --release 22 java/com/morphiqlabs/wavelet/gpu/*.java}.
 *
 * <p>Signals and results live in page-locked off-heap segments obtained from {@link #allocPinned(long)} (DMA-able,
 * exposed with {@code MemorySegment.reinterpret}); heap {@code double[]} arguments are copied into such a segment
 * once per call (the API-compatible path).</p>
 */
public final class VwNative {
    public static final int VW_OK = 0;
    public static final int FLAG_DEVICE_PTRS = 1, FLAG_CHECK_FINITE = 2, FLAG_BITEXACT = 4, FLAG_NO_FUSE = 8, FLAG_NO_SYNC = 16;
    public static final int ORDER_SPLIT = 0, ORDER_PAIR = 1;

    private static final Linker LINKER = Linker.nativeLinker();
    private static final SymbolLookup LIB = SymbolLookup.libraryLookup(
            System.getProperty("vectorwave.gpu.library", "libvwmodwt.so"), Arena.global());

    private static MethodHandle h(String name, FunctionDescriptor fd) {
        return LINKER.downcallHandle(LIB.find(name).orElseThrow(() -> new UnsatisfiedLinkError(name)), fd);
    }

    public static final MethodHandle vw_init = h("vw_init", FunctionDescriptor.of(JAVA_INT, JAVA_INT, ADDRESS));
    public static final MethodHandle vw_destroy = h("vw_destroy", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    static final MethodHandle vw_last_error = h("vw_last_error", FunctionDescriptor.of(ADDRESS, ADDRESS));
    static final MethodHandle vw_alloc_pinned = h("vw_alloc_pinned", FunctionDescriptor.of(ADDRESS, JAVA_LONG));
    static final MethodHandle vw_free_pinned = h("vw_free_pinned", FunctionDescriptor.ofVoid(ADDRESS));
    static final MethodHandle vw_max_levels = h("vw_max_levels", FunctionDescriptor.of(JAVA_INT, JAVA_LONG, JAVA_INT, JAVA_INT));
    /** int vw_conv_modwt(ctx, x, n, filter, lf, mode, out, flags) */
    static final MethodHandle vw_conv_modwt = h("vw_conv_modwt",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS, JAVA_LONG, JAVA_INT, ADDRESS, JAVA_INT));
    /** int vw_modwt_forward(ctx, x, batch, n, ldx, hs, gs, l, levels, mode, w, ldw, level_stride_w, vj, ldv, flags) */
    public static final MethodHandle vw_modwt_forward = h("vw_modwt_forward",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, JAVA_LONG, JAVA_LONG, ADDRESS, ADDRESS, JAVA_INT,
                    JAVA_INT, JAVA_INT, ADDRESS, JAVA_LONG, JAVA_LONG, ADDRESS, JAVA_LONG, JAVA_INT));
    /** int vw_modwt_inverse(ctx, w, ldw, level_stride_w, vj, ldv, batch, n, hs, gs, l, levels, mode, align, order,
     *  detail_mask, use_approx, xout, ldx, flags) */
    public static final MethodHandle vw_modwt_inverse = h("vw_modwt_inverse",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, JAVA_LONG, ADDRESS, JAVA_LONG, JAVA_LONG, JAVA_LONG,
                    ADDRESS, ADDRESS, JAVA_INT, JAVA_INT, JAVA_INT, ADDRESS, JAVA_INT, JAVA_LONG, JAVA_INT, ADDRESS,
                    JAVA_LONG, JAVA_INT));
    /** int vw_modwt_forward_varlen(ctx, x, const int64_t *offsets (host), batch, hs, gs, l, mode, w, v, flags) -- rows of
     *  different lengths packed back to back (MODWTTransform.forwardBatch with mixed lengths) */
    public static final MethodHandle vw_modwt_forward_varlen = h("vw_modwt_forward_varlen",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS, ADDRESS, JAVA_INT, JAVA_INT, ADDRESS,
                    ADDRESS, JAVA_INT));
    /** int vw_modwt_inverse_varlen(ctx, w, v, const int64_t *offsets (host), batch, hs, gs, l, mode, xout, flags) */
    public static final MethodHandle vw_modwt_inverse_varlen = h("vw_modwt_inverse_varlen",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS, ADDRESS, JAVA_INT, JAVA_INT,
                    ADDRESS, JAVA_INT));
    /** int vw_swt_denoise(ctx, x, batch, n, ldx, hs, gs, l, levels, mode, align, order, threshold, soft, out, ldo,
     *  thresholds_out, flags) */
    public static final MethodHandle vw_swt_denoise = h("vw_swt_denoise",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, JAVA_LONG, JAVA_LONG, ADDRESS, ADDRESS, JAVA_INT,
                    JAVA_INT, JAVA_INT, ADDRESS, JAVA_INT, JAVA_DOUBLE, JAVA_INT, ADDRESS, JAVA_LONG, ADDRESS, JAVA_INT));
    /** int vw_wavelet_denoise(ctx, x, batch, n, ldx, hs, gs, l, levels, mode, align, order, multilevel, method,
     *  fixed_threshold, soft, out, ldo, thresholds_out, flags) -- WaveletDenoiser over a batch, thresholds [level][row] */
    public static final MethodHandle vw_wavelet_denoise = h("vw_wavelet_denoise",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, JAVA_LONG, JAVA_LONG, ADDRESS, ADDRESS, JAVA_INT,
                    JAVA_INT, JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_DOUBLE, JAVA_INT, ADDRESS, JAVA_LONG,
                    ADDRESS, JAVA_INT));
    static final MethodHandle vw_threshold = h("vw_threshold",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, JAVA_LONG, JAVA_LONG, ADDRESS, JAVA_INT, JAVA_INT, JAVA_INT));
    static final MethodHandle vw_universal_threshold = h("vw_universal_threshold",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, JAVA_LONG, JAVA_LONG, ADDRESS, JAVA_INT));

    static final MethodHandle vw_energy = h("vw_energy",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, JAVA_LONG, JAVA_LONG, ADDRESS, JAVA_INT));
    static final MethodHandle vw_median_abs = h("vw_median_abs",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, JAVA_LONG, JAVA_LONG, ADDRESS, JAVA_INT));
    static final MethodHandle vw_mean_variance = h("vw_mean_variance",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, JAVA_LONG, JAVA_LONG, ADDRESS, ADDRESS, JAVA_INT));
    /** BatchSIMDMODWT SoA statics in place: (ctx, soa_x, batch, n, hs, gs, l, levels, double*[levels] soa_w, soa_v, flags) */
    static final MethodHandle vw_modwt_forward_soa = h("vw_modwt_forward_soa",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, JAVA_LONG, ADDRESS, ADDRESS, JAVA_INT, JAVA_INT, ADDRESS, ADDRESS, JAVA_INT));
    /** WaveletDenoiser.calculateSUREThreshold on the device: (ctx, c, batch, n, ld, sigma[batch], thr_out[batch], risk_out|NULL, flags) */
    static final MethodHandle vw_sure_threshold = h("vw_sure_threshold",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, JAVA_LONG, JAVA_LONG, ADDRESS, ADDRESS, ADDRESS, JAVA_INT));
    public static final MethodHandle vw_device_alloc = h("vw_device_alloc", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_LONG, ADDRESS));
    public static final MethodHandle vw_device_free = h("vw_device_free", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    public static final MethodHandle vw_copy_h2d = h("vw_copy_h2d", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG));
    public static final MethodHandle vw_copy_d2h = h("vw_copy_d2h", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG));
    /** int vw_modwt_stream_level(ctx, vin, batch, ldin, hist, n, hs, gs, l, level, w, ldw, v, ldv, flags) -- one level of
     *  BatchStreamingMODWT.process* on device rows of [history | block] (BatchStreamingMODWT.java:55-163) */
    static final MethodHandle vw_modwt_stream_level = h("vw_modwt_stream_level",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, JAVA_LONG, JAVA_LONG, JAVA_LONG, ADDRESS, ADDRESS,
                    JAVA_INT, JAVA_INT, ADDRESS, JAVA_LONG, ADDRESS, JAVA_LONG, JAVA_INT));
    /** int vw_stream_create(ctx, hs, gs, l, levels, mode, vw_stream_state **out) -- BatchStreamingMODWT's histories in HBM
     *  (ZERO_PADDING / SYMMETRIC); vw_stream_process runs a block's whole cascade, vw_stream_flush the tail (:55-276) */
    public static final MethodHandle vw_stream_create = h("vw_stream_create",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_INT, JAVA_INT, JAVA_INT, ADDRESS));
    public static final MethodHandle vw_stream_destroy = h("vw_stream_destroy", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    /** int vw_stream_process(ctx, st, x, batch, n, ldx, w, ldw, level_stride_w, v, ldv, flags) */
    public static final MethodHandle vw_stream_process = h("vw_stream_process",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, JAVA_LONG, JAVA_LONG, ADDRESS, JAVA_LONG,
                    JAVA_LONG, ADDRESS, JAVA_LONG, JAVA_INT));
    /** int vw_stream_flush(ctx, st, tail_length, w, ldw, level_stride_w, v, ldv, flags) -- histories not advanced */
    public static final MethodHandle vw_stream_flush = h("vw_stream_flush",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS, JAVA_LONG, JAVA_LONG, ADDRESS, JAVA_LONG, JAVA_INT));
    public static final MethodHandle vw_stream_reset = h("vw_stream_reset", FunctionDescriptor.of(JAVA_INT, ADDRESS));

    // ---- ABI v2: device-resident results, several GPUs from one thread, graph replay (include/vw_modwt.h) -----------
    /** int vw_modwt_decompose_h(ctx, x, batch, n, ldx, hs, gs, l, levels, mode, vw_result **res, flags) */
    public static final MethodHandle vw_modwt_decompose_h = h("vw_modwt_decompose_h",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, JAVA_LONG, JAVA_LONG, ADDRESS, ADDRESS, JAVA_INT, JAVA_INT,
                    JAVA_INT, ADDRESS, JAVA_INT));
    /** int vw_result_get_level / vw_result_set_level(ctx, res, level, buf, ld, flags) */
    public static final MethodHandle vw_result_get_level = h("vw_result_get_level",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS, JAVA_LONG, JAVA_INT));
    public static final MethodHandle vw_result_set_level = h("vw_result_set_level",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS, JAVA_LONG, JAVA_INT));
    /** int vw_result_threshold(ctx, res, level, thresholds, per_row, soft) */
    public static final MethodHandle vw_result_threshold = h("vw_result_threshold",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT));
    /** int vw_result_universal_threshold(ctx, res, soft, thresholds_out) */
    public static final MethodHandle vw_result_universal_threshold = h("vw_result_universal_threshold",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS));
    /** int vw_result_energy(ctx, res, level, out) */
    public static final MethodHandle vw_result_energy = h("vw_result_energy",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS));
    /** int vw_modwt_reconstruct_h(ctx, res, hs, gs, l, mode, align, order, detail_mask, use_approx, xout, ldx, flags) */
    public static final MethodHandle vw_modwt_reconstruct_h = h("vw_modwt_reconstruct_h",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, JAVA_INT, JAVA_INT, ADDRESS, JAVA_INT, JAVA_LONG,
                    JAVA_INT, ADDRESS, JAVA_LONG, JAVA_INT));
    public static final MethodHandle vw_result_free = h("vw_result_free", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    /** int vw_span_plan_query(l, levels, n_local, world, vw_span_plan *out) -- sizeof(vw_span_plan) = SPAN_PLAN_BYTES */
    public static final long SPAN_PLAN_BYTES = 16 + 8 + 8 + 4 * 16 * 4 + 2 * 16 * 8 + 4 * 8;
    public static final MethodHandle vw_span_plan_query = h("vw_span_plan_query",
            FunctionDescriptor.of(JAVA_INT, JAVA_INT, JAVA_INT, JAVA_LONG, JAVA_INT, ADDRESS));
    /** int vw_init_multi(const int *devices, ndev, vw_multi **out); vw_destroy_multi(m); vw_multi_ctx(m, rank) */
    public static final MethodHandle vw_init_multi = h("vw_init_multi", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, ADDRESS));
    public static final MethodHandle vw_destroy_multi = h("vw_destroy_multi", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    public static final MethodHandle vw_multi_ctx = h("vw_multi_ctx", FunctionDescriptor.of(ADDRESS, ADDRESS, JAVA_INT));
    public static final MethodHandle vw_multi_last_error = h("vw_multi_last_error", FunctionDescriptor.of(ADDRESS, ADDRESS));
    /** int vw_modwt_forward_sharded(m, plan, double*const* xext, hs, gs, mode, double*const* w, row_stride, double*const* v,
     *  float *exchange_ms, flags) */
    public static final MethodHandle vw_modwt_forward_sharded = h("vw_modwt_forward_sharded",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS, JAVA_INT, ADDRESS, JAVA_LONG, ADDRESS, ADDRESS,
                    JAVA_INT));
    /** int vw_modwt_inverse_sharded(m, plan, w, row_stride, v, hs, gs, mode, order, xout, exchange_ms, flags) */
    public static final MethodHandle vw_modwt_inverse_sharded = h("vw_modwt_inverse_sharded",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS, ADDRESS, ADDRESS, JAVA_INT, JAVA_INT, ADDRESS,
                    ADDRESS, JAVA_INT));
    /** int vw_swt_denoise_sharded(m, plan, xext, hs, gs, mode, order, threshold, soft, w, row_stride, v, xout,
     *  double *threshold_out, flags): one long signal denoised across the devices with the exact universal threshold */
    public static final MethodHandle vw_swt_denoise_sharded = h("vw_swt_denoise_sharded",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS, JAVA_INT, JAVA_INT, JAVA_DOUBLE, JAVA_INT,
                    ADDRESS, JAVA_LONG, ADDRESS, ADDRESS, ADDRESS, JAVA_INT));
    /** int vw_modwt_inverse_span_all_thr(ctx, plan, w, row_stride, v, hs, gs, order, const double *thr_dev, soft, xout, flags) */
    public static final MethodHandle vw_modwt_inverse_span_all_thr = h("vw_modwt_inverse_span_all_thr",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS, ADDRESS, ADDRESS, JAVA_INT, ADDRESS, JAVA_INT,
                    ADDRESS, JAVA_INT));
    /** The cross-rank median rounds (one process per GPU): state_bytes(n_local); init(ctx, state, n_total); for round in
     *  0 .. SPAN_MEDIAN_ROUNDS-1: hist(ctx, state, c, n_local, round, uint64 *hist) -> caller's all-reduce (sum) ->
     *  pick(ctx, state, round, const uint64 *hist_sum); value(ctx, state, factor, double *out_dev).  Device pointers. */
    public static final int SPAN_MEDIAN_ROUNDS = 7;
    public static final MethodHandle vw_span_median_bins = h("vw_span_median_bins", FunctionDescriptor.of(JAVA_INT, JAVA_INT));
    public static final MethodHandle vw_span_median_state_bytes = h("vw_span_median_state_bytes", FunctionDescriptor.of(JAVA_LONG, JAVA_LONG));
    public static final MethodHandle vw_span_median_init = h("vw_span_median_init", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG));
    public static final MethodHandle vw_span_median_hist = h("vw_span_median_hist",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, JAVA_INT, ADDRESS));
    public static final MethodHandle vw_span_median_pick = h("vw_span_median_pick",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS));
    public static final MethodHandle vw_span_median_value = h("vw_span_median_value",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_DOUBLE, ADDRESS));
    /** CUDA-graph replay of a fixed call sequence: vw_graph_begin(ctx); ...calls...; vw_graph_end(ctx, &g); vw_graph_launch(ctx, g, flags) */
    public static final MethodHandle vw_graph_begin = h("vw_graph_begin", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    public static final MethodHandle vw_graph_end = h("vw_graph_end", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    public static final MethodHandle vw_graph_launch = h("vw_graph_launch", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT));
    public static final MethodHandle vw_graph_destroy = h("vw_graph_destroy", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));

    private VwNative() {}

    /** Page-locked host memory as a segment of {@code bytes} bytes (freed with {@link #freePinned}). */
    public static MemorySegment allocPinned(long bytes) {
        try {
            MemorySegment p = (MemorySegment) vw_alloc_pinned.invokeExact(bytes);
            if (p.equals(MemorySegment.NULL)) throw new OutOfMemoryError("vw_alloc_pinned(" + bytes + ")");
            return p.reinterpret(bytes);
        } catch (Throwable t) {
            throw rethrow(t);
        }
    }

    public static void freePinned(MemorySegment seg) {
        try {
            vw_free_pinned.invokeExact(seg);
        } catch (Throwable t) {
            throw rethrow(t);
        }
    }

    public static RuntimeException rethrow(Throwable t) {
        if (t instanceof RuntimeException r) return r;
        if (t instanceof Error e) throw e;
        return new RuntimeException(t);
    }

    public static String lastError(MemorySegment ctx) {
        try {
            MemorySegment s = (MemorySegment) vw_last_error.invokeExact(ctx);
            return s.reinterpret(512).getString(0);
        } catch (Throwable t) {
            throw rethrow(t);
        }
    }

    public static void copyIn(MemorySegment dst, double[] src) {
        MemorySegment.copy(src, 0, dst, ValueLayout.JAVA_DOUBLE, 0, src.length);
    }

    public static double[] copyOut(MemorySegment src, long offsetDoubles, int n) {
        double[] out = new double[n];
        MemorySegment.copy(src, ValueLayout.JAVA_DOUBLE, offsetDoubles * 8, out, 0, n);
        return out;
    }
}
