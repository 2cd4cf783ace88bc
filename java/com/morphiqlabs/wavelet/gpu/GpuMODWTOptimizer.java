package com.morphiqlabs.wavelet.gpu;

import com.morphiqlabs.wavelet.api.BoundaryMode;
import com.morphiqlabs.wavelet.api.Wavelet;
import com.morphiqlabs.wavelet.api.spi.MODWTOptimizer;
import com.morphiqlabs.wavelet.exception.ErrorCode;
import com.morphiqlabs.wavelet.exception.InvalidArgumentException;
import com.morphiqlabs.wavelet.exception.InvalidSignalException;

import java.lang.foreign.Arena;
import java.lang.foreign.MemorySegment;
import java.lang.foreign.ValueLayout;

/**
 * ServiceLoader provider for the reference's (dormant) MODWT SPI --
 * vectorwave-core/src/main/java/com/morphiqlabs/wavelet/api/spi/MODWTOptimizer.java:39,49,59 -- backed by the
 * B200 engine.  Register it with a line {@code com.morphiqlabs.wavelet.gpu.GpuMODWTOptimizer} in
 * {@code META-INF/services/com.morphiqlabs.wavelet.api.spi.MODWTOptimizer} (same pattern as
 * vectorwave-extensions/src/main/resources/META-INF/services/...WaveletTransformOptimizer).
 *
 * <p>Filters are scaled by {@code 1.0 / Math.sqrt(2.0)} here, exactly as MODWTTransform.java:139-150 does, so the
 * table quirks stay the reference's; the native side applies no scaling.</p>
 */
public final class GpuMODWTOptimizer implements MODWTOptimizer, AutoCloseable {
    private final MemorySegment ctx;

    public GpuMODWTOptimizer() {
        try (Arena a = Arena.ofConfined()) {
            MemorySegment out = a.allocate(ValueLayout.ADDRESS);
            int rc = (int) VwNative.vw_init.invokeExact(Integer.getInteger("vectorwave.gpu.device", -1), out);
            if (rc != VwNative.VW_OK) throw new IllegalStateException("vw_init failed: " + rc + " (no CUDA device? there is no CPU fallback)");
            ctx = out.get(ValueLayout.ADDRESS, 0);
        } catch (Throwable t) {
            throw VwNative.rethrow(t);
        }
    }

    static int modeOf(BoundaryMode m) {
        return switch (m) {
            case PERIODIC -> 0;
            case ZERO_PADDING -> 1;
            case SYMMETRIC -> 2;
            default -> 3; // rejected by the engine with CFG_UNSUPPORTED_BOUNDARY_MODE
        };
    }

    static double[] scaled(double[] f) {
        double s = 1.0 / Math.sqrt(2.0);
        double[] out = new double[f.length];
        for (int i = 0; i < f.length; i++) out[i] = f[i] * s;
        return out;
    }

    /** vw_status -> the reference's exceptions (CORE/exception/ErrorCode.java:24-118). */
    void check(int rc) {
        if (rc == VwNative.VW_OK) return;
        String msg = VwNative.lastError(ctx);
        switch (rc) {
            case 1 -> throw new NullPointerException(msg);
            case 3 -> throw new InvalidSignalException(ErrorCode.VAL_NON_FINITE_VALUES, msg);
            case 5 -> throw new InvalidArgumentException(ErrorCode.VAL_TOO_LARGE, msg);
            case 6 -> throw new InvalidSignalException(ErrorCode.VAL_EMPTY, msg);
            case 103 -> throw new InvalidArgumentException(ErrorCode.CFG_UNSUPPORTED_BOUNDARY_MODE, msg);
            case 104 -> throw new InvalidArgumentException(ErrorCode.CFG_INVALID_DECOMPOSITION_LEVEL, msg);
            case 7, 400 -> throw new IllegalArgumentException(msg);
            default -> throw new IllegalStateException("libvwmodwt: " + rc + ": " + msg);
        }
    }

    /** MODWTOptimizer.MODWTOptimizedResult (MODWTOptimizer.java:75-84). */
    private record Result(double[] w, double[] v) implements MODWTOptimizedResult {
        @Override public double[] getWaveletCoefficients() { return w; }
        @Override public double[] getScalingCoefficients() { return v; }
    }

    @Override
    public boolean isSupported() {
        return true;   // the constructor already failed loudly if no CUDA device / library was found
    }

    @Override
    public int getPriority() {
        return 1000;   // above the Vector-API provider
    }

    @Override
    public String getName() {
        return "B200 CUDA MODWT engine (libvwmodwt.so)";
    }

    @Override
    public MODWTOptimizedResult forward(double[] signal, Wavelet wavelet, BoundaryMode mode) {
        return forwardBatch(new double[][]{signal}, wavelet, mode)[0];
    }

    @Override
    public MODWTOptimizedResult[] forwardBatch(double[][] signals, Wavelet wavelet, BoundaryMode mode) {
        int b = signals.length, n = signals[0].length;
        for (double[] s : signals)
            if (s.length != n) return forwardBatchMixed(signals, wavelet, mode);
        double[] hs = scaled(wavelet.lowPassDecomposition()), gs = scaled(wavelet.highPassDecomposition());
        long bytes = (long) b * n * 8;
        PinnedArena pin = PinnedArena.current();      // pooled: cudaMallocHost per call would cost more than the transform
        pin.reset();
        MemorySegment[] seg = pin.takeAll(bytes, bytes, bytes);
        MemorySegment x = seg[0], w = seg[1], v = seg[2];
        try (Arena a = Arena.ofConfined()) {
            for (int i = 0; i < b; i++) MemorySegment.copy(signals[i], 0, x, ValueLayout.JAVA_DOUBLE, (long) i * n * 8, n);
            MemorySegment hseg = a.allocateFrom(ValueLayout.JAVA_DOUBLE, hs), gseg = a.allocateFrom(ValueLayout.JAVA_DOUBLE, gs);
            check((int) VwNative.vw_modwt_forward.invokeExact(ctx, x, (long) b, (long) n, (long) n, hseg, gseg, hs.length, 1,
                    modeOf(mode), w, (long) n, (long) b * n, v, (long) n, VwNative.FLAG_CHECK_FINITE));
            MODWTOptimizedResult[] out = new MODWTOptimizedResult[b];
            for (int i = 0; i < b; i++)
                out[i] = new Result(VwNative.copyOut(w, (long) i * n, n), VwNative.copyOut(v, (long) i * n, n));
            return out;
        } catch (Throwable t) {
            throw VwNative.rethrow(t);
        }
    }

    /** Rows of different lengths, each transformed at its own length: packed back to back and sent as ONE
     *  vw_modwt_forward_varlen call (MODWTTransform.forwardBatch, MODWTTransform.java:486-515, runs forward per row). */
    private MODWTOptimizedResult[] forwardBatchMixed(double[][] signals, Wavelet wavelet, BoundaryMode mode) {
        int b = signals.length;
        long[] off = new long[b + 1];
        for (int i = 0; i < b; i++) off[i + 1] = off[i] + signals[i].length;
        long total = off[b];
        double[] hs = scaled(wavelet.lowPassDecomposition()), gs = scaled(wavelet.highPassDecomposition());
        PinnedArena pin = PinnedArena.current();
        pin.reset();
        MemorySegment[] seg = pin.takeAll(total * 8, total * 8, total * 8);
        MemorySegment x = seg[0], w = seg[1], v = seg[2];
        try (Arena a = Arena.ofConfined()) {
            for (int i = 0; i < b; i++)
                MemorySegment.copy(signals[i], 0, x, ValueLayout.JAVA_DOUBLE, off[i] * 8, signals[i].length);
            MemorySegment offseg = a.allocateFrom(ValueLayout.JAVA_LONG, off);
            MemorySegment hseg = a.allocateFrom(ValueLayout.JAVA_DOUBLE, hs), gseg = a.allocateFrom(ValueLayout.JAVA_DOUBLE, gs);
            int rc = (int) VwNative.vw_modwt_forward_varlen.invokeExact(ctx, x, offseg, (long) b, hseg, gseg, hs.length,
                    modeOf(mode), w, v, VwNative.FLAG_CHECK_FINITE);
            check(rc);
            MODWTOptimizedResult[] out = new MODWTOptimizedResult[b];
            for (int i = 0; i < b; i++) {
                int n = signals[i].length;
                out[i] = new Result(VwNative.copyOut(w, off[i], n), VwNative.copyOut(v, off[i], n));
            }
            return out;
        } catch (Throwable t) {
            throw VwNative.rethrow(t);
        }
    }

    @Override
    public double[] inverse(double[] waveletCoeffs, double[] scalingCoeffs, Wavelet wavelet, BoundaryMode mode) {
        double[] detail = waveletCoeffs, approx = scalingCoeffs;
        int n = approx.length;
        double[] hs = scaled(wavelet.lowPassReconstruction()), gs = scaled(wavelet.highPassReconstruction());
        PinnedArena pin = PinnedArena.current();
        pin.reset();
        MemorySegment[] seg = pin.takeAll(n * 8L, n * 8L, n * 8L);
        MemorySegment w = seg[0], v = seg[1], x = seg[2];
        try (Arena a = Arena.ofConfined()) {
            VwNative.copyIn(w, detail);
            VwNative.copyIn(v, approx);
            MemorySegment hseg = a.allocateFrom(ValueLayout.JAVA_DOUBLE, hs), gseg = a.allocateFrom(ValueLayout.JAVA_DOUBLE, gs);
            // MODWTTransform.inverse: pair-added products; SYMMETRIC uses t-l => sigma = -1, tau = 0 (MODWTTransform.java:277-295)
            MemorySegment align = MemorySegment.NULL;
            if (mode == BoundaryMode.SYMMETRIC) align = a.allocateFrom(ValueLayout.JAVA_INT, -1, 0, -1, 0);
            check((int) VwNative.vw_modwt_inverse.invokeExact(ctx, w, (long) n, (long) n, v, (long) n, 1L, (long) n, hseg, gseg,
                    hs.length, 1, modeOf(mode), align, VwNative.ORDER_PAIR, 1L, 1, x, (long) n, 0));
            return VwNative.copyOut(x, 0, n);
        } catch (Throwable t) {
            throw VwNative.rethrow(t);
        }
    }

    /** BatchSIMDMODWT.batchMultiLevelMODWTSoA (extensions/modwt/BatchSIMDMODWT.java:343-381) on the caller's SoA arrays
     *  ([t * batchSize + b]); levels == 1 with the literal Haar taps is batchMODWTSoA (:64-81).  No AoS round trip. */
    public void batchMultiLevelMODWTSoA(double[] soaSignals, double[][] soaDetailPerLevel, double[] soaApproxOut,
                                        Wavelet wavelet, int batchSize, int signalLength, int levels) {
        if (soaDetailPerLevel.length != levels) throw new IllegalArgumentException("soaDetailPerLevel length must equal levels");
        long tot = (long) batchSize * signalLength;
        double[] hs = scaled(wavelet.lowPassDecomposition()), gs = scaled(wavelet.highPassDecomposition());
        PinnedArena pin = PinnedArena.current();
        pin.reset();
        MemorySegment[] seg = pin.takeAll(tot * 8, tot * 8 * (levels + 1));
        MemorySegment x = seg[0], out = seg[1];
        try (Arena a = Arena.ofConfined()) {
            VwNative.copyIn(x, soaSignals);
            MemorySegment hseg = a.allocateFrom(ValueLayout.JAVA_DOUBLE, hs), gseg = a.allocateFrom(ValueLayout.JAVA_DOUBLE, gs);
            MemorySegment ptrs = a.allocate(ValueLayout.ADDRESS, levels);
            for (int j = 0; j < levels; j++) ptrs.setAtIndex(ValueLayout.ADDRESS, j, out.asSlice((long) j * tot * 8, tot * 8));
            check((int) VwNative.vw_modwt_forward_soa.invokeExact(ctx, x, (long) batchSize, (long) signalLength, hseg, gseg,
                    hs.length, levels, ptrs, out.asSlice((long) levels * tot * 8, tot * 8), 0));
            for (int j = 0; j < levels; j++)
                MemorySegment.copy(out, ValueLayout.JAVA_DOUBLE, (long) j * tot * 8, soaDetailPerLevel[j], 0, (int) tot);
            MemorySegment.copy(out, ValueLayout.JAVA_DOUBLE, (long) levels * tot * 8, soaApproxOut, 0, (int) tot);
        } catch (Throwable t) {
            throw VwNative.rethrow(t);
        }
    }

    @Override
    public void close() {
        try {
            VwNative.vw_destroy.invokeExact(ctx);
        } catch (Throwable t) {
            throw VwNative.rethrow(t);
        }
    }
}
