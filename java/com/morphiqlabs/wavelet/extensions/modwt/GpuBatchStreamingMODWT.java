package com.morphiqlabs.wavelet.extensions.modwt;

import com.morphiqlabs.wavelet.api.BoundaryMode;
import com.morphiqlabs.wavelet.api.DiscreteWavelet;
import com.morphiqlabs.wavelet.gpu.PinnedArena;
import com.morphiqlabs.wavelet.gpu.VwNative;

import java.lang.foreign.Arena;
import java.lang.foreign.MemorySegment;
import java.lang.foreign.ValueLayout;

/**
 * {@link BatchStreamingMODWT} (extensions/modwt/BatchStreamingMODWT.java:55-276) on the B200 engine for ZERO_PADDING and
 * SYMMETRIC: every level's history stays in HBM behind one native stream state, and each block -- its whole cascade, the
 * first-block initialisation and the batch-size restart (:306-320) included -- is one {@code vw_stream_process} call.
 * PERIODIC streaming has no state and stays on {@link GpuBatchMODWT}.  The facade keeps its own validation (empty blocks,
 * level checks, {@code tailLength} limits); this class returns the same result records.
 *
 * <pre>
 *   try (GpuBatchStreamingMODWT s = new GpuBatchStreamingMODWT(wavelet, BoundaryMode.SYMMETRIC, levels)) {
 *       BatchMODWT.MultiLevelResult r = s.processMultiLevel(block);   // per block
 *       BatchMODWT.MultiLevelResult tail = s.flushMultiLevel(s.getMinFlushTailLength());
 *   }
 * </pre>
 * Blocks and results are staged through the calling thread's pooled pinned block ({@link PinnedArena}).
 */
public final class GpuBatchStreamingMODWT implements AutoCloseable {
    private final MemorySegment ctx, state;
    private final int levels, filterLength;
    private int batch;   // rows of the running stream, 0 before the first block

    public GpuBatchStreamingMODWT(DiscreteWavelet wavelet, BoundaryMode mode, int levels) {
        if (levels < 1) throw new IllegalArgumentException("levels must be >= 1");
        if (mode != BoundaryMode.ZERO_PADDING && mode != BoundaryMode.SYMMETRIC)
            throw new IllegalArgumentException("the stream state serves ZERO_PADDING and SYMMETRIC (PERIODIC streaming is stateless)");
        double s = 1.0 / Math.sqrt(2.0);
        double[] h = wavelet.lowPassDecomposition(), g = wavelet.highPassDecomposition();
        double[] hs = new double[h.length], gs = new double[g.length];
        for (int i = 0; i < h.length; i++) { hs[i] = h[i] * s; gs[i] = g[i] * s; }
        this.levels = levels;
        this.filterLength = h.length;
        try (Arena a = Arena.ofConfined()) {
            MemorySegment out = a.allocate(ValueLayout.ADDRESS);
            int rc = (int) VwNative.vw_init.invokeExact(Integer.getInteger("vectorwave.gpu.device", -1), out);
            if (rc != VwNative.VW_OK) throw new IllegalStateException("libvwmodwt: no CUDA device (" + rc + ")");
            ctx = out.get(ValueLayout.ADDRESS, 0);
            MemorySegment hseg = a.allocateFrom(ValueLayout.JAVA_DOUBLE, hs), gseg = a.allocateFrom(ValueLayout.JAVA_DOUBLE, gs);
            rc = (int) VwNative.vw_stream_create.invokeExact(ctx, hseg, gseg, hs.length, levels,
                    mode == BoundaryMode.ZERO_PADDING ? 1 : 2, out);
            if (rc != VwNative.VW_OK) {
                String msg = VwNative.lastError(ctx);
                int ignored = (int) VwNative.vw_destroy.invokeExact(ctx);
                throw new IllegalArgumentException(msg);
            }
            state = out.get(ValueLayout.ADDRESS, 0);
        } catch (Throwable t) {
            throw VwNative.rethrow(t);
        }
    }

    private void check(int rc) {
        if (rc == VwNative.VW_OK) return;
        String msg = VwNative.lastError(ctx);
        if (rc == 1) throw new NullPointerException(msg);
        if (rc == 6 || rc == 7 || rc == 104 || rc == 400) throw new IllegalArgumentException(msg);
        throw new IllegalStateException("libvwmodwt: " + rc + ": " + msg);
    }

    /** BatchStreamingMODWT.processSingleLevel (:55-103); levels must be 1. */
    public BatchMODWT.SingleLevelResult processSingleLevel(double[][] block) {
        if (levels != 1) throw new IllegalStateException("This instance is configured for levels=" + levels + ", expected=1");
        BatchMODWT.MultiLevelResult r = processMultiLevel(block);
        return new BatchMODWT.SingleLevelResult(r.finalApprox(), r.detailPerLevel()[0]);
    }

    /** BatchStreamingMODWT.processMultiLevel (:111-163): details [levels][batch][n], final approximation [batch][n]. */
    public BatchMODWT.MultiLevelResult processMultiLevel(double[][] block) {
        int b = block.length, n = block[0].length;
        long bn = (long) b * n;
        PinnedArena pin = PinnedArena.current();
        pin.reset();
        MemorySegment[] seg = pin.takeAll(8L * bn, 8L * bn * levels, 8L * bn);
        for (int i = 0; i < b; i++) MemorySegment.copy(block[i], 0, seg[0], ValueLayout.JAVA_DOUBLE, 8L * i * n, n);
        try {
            check((int) VwNative.vw_stream_process.invokeExact(ctx, state, seg[0], (long) b, (long) n, (long) n, seg[1], (long) n,
                    bn, seg[2], (long) n, 0));
        } catch (Throwable t) {
            throw VwNative.rethrow(t);
        }
        batch = b;
        return result(seg[1], seg[2], b, n);
    }

    /** BatchStreamingMODWT.flushSingleLevel (:183-222). */
    public BatchMODWT.SingleLevelResult flushSingleLevel(int tailLength) {
        if (levels != 1) throw new IllegalStateException("This instance is configured for levels=" + levels + ", expected=1");
        BatchMODWT.MultiLevelResult r = flushMultiLevel(tailLength);
        return new BatchMODWT.SingleLevelResult(r.finalApprox(), r.detailPerLevel()[0]);
    }

    /** BatchStreamingMODWT.flushMultiLevel (:231-276): the tail's cascade; the histories are not advanced. */
    public BatchMODWT.MultiLevelResult flushMultiLevel(int tailLength) {
        if (tailLength <= 0) return new BatchMODWT.MultiLevelResult(new double[levels][0][0], new double[0][0]);
        if (batch == 0) throw new IllegalStateException("No prior blocks processed; cannot flush");
        long bt = (long) batch * tailLength;
        PinnedArena pin = PinnedArena.current();
        pin.reset();
        MemorySegment[] seg = pin.takeAll(8L * bt * levels, 8L * bt);
        try {
            check((int) VwNative.vw_stream_flush.invokeExact(ctx, state, (long) tailLength, seg[0], (long) tailLength, bt, seg[1],
                    (long) tailLength, 0));
        } catch (Throwable t) {
            throw VwNative.rethrow(t);
        }
        return result(seg[0], seg[1], batch, tailLength);
    }

    private BatchMODWT.MultiLevelResult result(MemorySegment w, MemorySegment v, int b, int n) {
        long bn = (long) b * n;
        double[][][] detail = new double[levels][b][];
        double[][] approx = new double[b][];
        for (int j = 0; j < levels; j++)
            for (int i = 0; i < b; i++) detail[j][i] = VwNative.copyOut(w, j * bn + (long) i * n, n);
        for (int i = 0; i < b; i++) approx[i] = VwNative.copyOut(v, (long) i * n, n);
        return new BatchMODWT.MultiLevelResult(detail, approx);
    }

    public int getMinFlushTailLength() { return filterLength - 1; }

    /** Back to "no block seen": the next block starts a new stream. */
    public void reset() {
        try {
            check((int) VwNative.vw_stream_reset.invokeExact(state));
        } catch (Throwable t) {
            throw VwNative.rethrow(t);
        }
        batch = 0;
    }

    @Override
    public void close() {
        try {
            int rc = (int) VwNative.vw_stream_destroy.invokeExact(ctx, state);
            rc = (int) VwNative.vw_destroy.invokeExact(ctx);
        } catch (Throwable t) {
            throw VwNative.rethrow(t);
        }
    }
}
