/*
 * Foreign Function & Memory API (java.lang.foreign, final in JDK 22) binding of libsdrgpu.so -- the C ABI declared in
 * include/sdrgpu.h.  One downcall handle per entry point the shim classes of this package use; status codes map to the
 * exceptions the replaced Java code threw.  Not compiled in the build image (no JDK there): sources for the
 * maintainer, syntactically complete against smyers119/sdrtrunk's packages.
 */
package io.github.dsheirer.gpu;

import io.github.dsheirer.dsp.filter.design.FilterDesignException;

import java.lang.foreign.Arena;
import java.lang.foreign.FunctionDescriptor;
import java.lang.foreign.Linker;
import java.lang.foreign.MemoryLayout;
import java.lang.foreign.MemorySegment;
import java.lang.foreign.StructLayout;
import java.lang.foreign.SymbolLookup;
import java.lang.invoke.MethodHandle;
import java.nio.BufferOverflowException;

import static java.lang.foreign.ValueLayout.ADDRESS;
import static java.lang.foreign.ValueLayout.JAVA_DOUBLE;
import static java.lang.foreign.ValueLayout.JAVA_FLOAT;
import static java.lang.foreign.ValueLayout.JAVA_INT;
import static java.lang.foreign.ValueLayout.JAVA_LONG;

public final class SdrGpu
{
    public static final int HOST = 0, DEVICE = 1;
    public static final int LAYOUT_RESULTS = 0, LAYOUT_CHANNELS = 1;
    public static final int FORMAT_F32 = 0, FORMAT_U8 = 1, FORMAT_S8 = 2, FORMAT_S16LE = 3;
    public static final int PRESET_P25_C4FM = 0, PRESET_P25_LSM = 1, PRESET_P25_HDQPSK = 2, PRESET_NBFM = 3, PRESET_DMR = 4;
    public static final int SYNC_NONE = 0, SYNC_P25_PHASE1 = 1, SYNC_P25_PHASE2 = 2, SYNC_P25_PHASE2_FRAMED = 3;

    private static final Linker LINKER = Linker.nativeLinker();
    private static final SymbolLookup LIB = SymbolLookup.libraryLookup(System.getProperty("sdrgpu.library", "libsdrgpu.so"),
        Arena.global());

    private static MethodHandle h(String name, FunctionDescriptor descriptor)
    {
        return LINKER.downcallHandle(LIB.find(name).orElseThrow(() -> new UnsatisfiedLinkError(name)), descriptor);
    }

    /** struct sdrgpu_output_channel { int bin1; int bin2; long long frequency_offset_hz; double gain; } */
    public static final StructLayout OUTPUT_CHANNEL = MemoryLayout.structLayout(JAVA_INT.withName("bin1"), JAVA_INT.withName("bin2"),
        JAVA_LONG.withName("frequency_offset_hz"), JAVA_DOUBLE.withName("gain"));

    /** struct sdrgpu_bank_output { uint8_t *symbols; int symbol_stride; float *demod; long long demod_stride_floats; int *counts; }:
     * one bank's outputs of sdrgpu_pipeline_process_routed */
    public static final StructLayout BANK_OUTPUT = MemoryLayout.structLayout(
        ADDRESS.withName("symbols"), JAVA_INT.withName("symbol_stride"), MemoryLayout.paddingLayout(4),
        ADDRESS.withName("demod"), JAVA_LONG.withName("demod_stride_floats"), ADDRESS.withName("counts"));

    /** struct sdrgpu_bank_config (include/sdrgpu.h), natural C alignment on x86-64 / aarch64 */
    public static final StructLayout BANK_CONFIG = MemoryLayout.structLayout(
        JAVA_INT.withName("n_channels"), MemoryLayout.paddingLayout(4),
        JAVA_DOUBLE.withName("sample_rate"),
        JAVA_INT.withName("decimation"), MemoryLayout.paddingLayout(4),
        ADDRESS.withName("fir_taps"),
        JAVA_INT.withName("n_fir_taps"), JAVA_FLOAT.withName("fir_gain"),
        JAVA_INT.withName("agc"), JAVA_INT.withName("block_size"),
        JAVA_INT.withName("demod"), MemoryLayout.paddingLayout(4),
        JAVA_DOUBLE.withName("symbol_rate"), JAVA_DOUBLE.withName("pll_bandwidth"),
        JAVA_FLOAT.withName("sample_counter_gain"), JAVA_FLOAT.withName("fm_gain"),
        JAVA_DOUBLE.withName("squelch_alpha"), JAVA_DOUBLE.withName("squelch_threshold_db"),
        JAVA_INT.withName("squelch_ramp"), JAVA_INT.withName("max_samples_per_call"));

    static final MethodHandle INIT = h("sdrgpu_init", FunctionDescriptor.of(JAVA_INT, JAVA_INT));
    static final MethodHandle LAST_ERROR = h("sdrgpu_last_error", FunctionDescriptor.of(ADDRESS));
    static final MethodHandle ALLOC_PINNED = h("sdrgpu_alloc_pinned", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_LONG));
    static final MethodHandle FREE_PINNED = h("sdrgpu_free_pinned", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    static final MethodHandle CHAN_CREATE = h("sdrgpu_chan_create",
        FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, JAVA_INT, JAVA_INT));
    static final MethodHandle CHAN_DESTROY = h("sdrgpu_chan_destroy", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    static final MethodHandle CHAN_SET_SAMPLE_RATE = h("sdrgpu_chan_set_sample_rate", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_DOUBLE));
    static final MethodHandle CHAN_SET_INPUT_FORMAT = h("sdrgpu_chan_set_input_format", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT));
    static final MethodHandle CHAN_SELECT = h("sdrgpu_chan_select",
        FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS, JAVA_INT));
    static final MethodHandle CHAN_PROCESS = h("sdrgpu_chan_process",
        FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, JAVA_INT, ADDRESS, JAVA_LONG, JAVA_INT, JAVA_INT, ADDRESS));
    static final MethodHandle CHAN_BLOCKS_FOR = h("sdrgpu_chan_blocks_for", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT));
    static final MethodHandle BANK_CONFIG_PRESET = h("sdrgpu_bank_config_preset",
        FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT, JAVA_DOUBLE, ADDRESS, JAVA_INT, JAVA_INT));
    static final MethodHandle BANK_CREATE = h("sdrgpu_bank_create", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    static final MethodHandle BANK_DESTROY = h("sdrgpu_bank_destroy", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    static final MethodHandle BANK_PROCESS = h("sdrgpu_bank_process",
        FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, JAVA_INT, JAVA_INT, ADDRESS, JAVA_INT, ADDRESS, JAVA_LONG,
            ADDRESS, JAVA_INT));
    static final MethodHandle BANK_CORRECT_INVERSION = h("sdrgpu_bank_correct_inversion",
        FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, JAVA_DOUBLE));
    static final MethodHandle BANK_SET_SYNC_DETECTOR = h("sdrgpu_bank_set_sync_detector", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT));
    /** (bank, enabled): FM_SQUELCH banks write one squelch status byte per assembler buffer into `symbols`
     *  (state after the buffer in bits 0-1: 0 ATTACK, 1 DECAY, 2 MUTE, 3 UNMUTE; bit 2: the squelch changed during it) */
    static final MethodHandle BANK_SET_SQUELCH_REPORTING = h("sdrgpu_bank_set_squelch_reporting",
        FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT));
    /** (bank, channel | -1 for all, threshold dB): PowerSquelch.setSquelchThreshold per channel, from the next buffer on */
    static final MethodHandle BANK_SET_SQUELCH_THRESHOLD = h("sdrgpu_bank_set_squelch_threshold",
        FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, JAVA_DOUBLE));
    /** the listeners of DQPSKDecisionDirectedDemodulatorInstrumented for one channel of a bank: (bank, channel | -1) */
    static final MethodHandle BANK_SET_SYMBOL_TAP = h("sdrgpu_bank_set_symbol_tap", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT));
    /** (bank, double[6 * capacity] values, capacity, int[1] nSymbols): symbol I, Q, samples per symbol, loop frequency, sampling point, PLL error */
    static final MethodHandle BANK_READ_SYMBOL_TAP = h("sdrgpu_bank_read_symbol_tap",
        FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS));
    static final MethodHandle PIPELINE_CREATE_MULTI = h("sdrgpu_pipeline_create_multi",
        FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS));
    /** (pipeline*, channelizers[], nChans, banks[], nBanks, int[] route): one channelizer pass feeds several banks; route[r] is
     * the bank index of selected channel r in pipeline row order */
    static final MethodHandle PIPELINE_CREATE_ROUTED = h("sdrgpu_pipeline_create_routed",
        FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS, JAVA_INT, ADDRESS));
    /** (pipeline, iq[], nFloats, inMem, BANK_OUTPUT[nBanks], outMem) */
    static final MethodHandle PIPELINE_PROCESS_ROUTED = h("sdrgpu_pipeline_process_routed",
        FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, JAVA_INT, ADDRESS, JAVA_INT));
    static final MethodHandle PIPELINE_DESTROY = h("sdrgpu_pipeline_destroy", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    static final MethodHandle PIPELINE_PROCESS_MULTI = h("sdrgpu_pipeline_process_multi",
        FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, JAVA_INT, ADDRESS, JAVA_INT, ADDRESS, JAVA_LONG, ADDRESS, JAVA_INT));
    /** asynchronous form for a continuous stream: (pipeline, iq[], nFloats, symbols, symbolStride, counts); at most two in flight */
    static final MethodHandle PIPELINE_SUBMIT_MULTI = h("sdrgpu_pipeline_submit_multi",
        FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS, JAVA_INT, ADDRESS));
    /** returns when the OLDEST submitted call has its dibits and counts in the host buffers it was given */
    static final MethodHandle PIPELINE_WAIT = h("sdrgpu_pipeline_wait", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    static final MethodHandle DESIGN_REMEZ_LOW_PASS = h("sdrgpu_design_remez_low_pass",
        FunctionDescriptor.of(JAVA_INT, JAVA_DOUBLE, JAVA_DOUBLE, JAVA_DOUBLE, JAVA_DOUBLE, JAVA_DOUBLE, JAVA_INT, JAVA_INT, JAVA_INT,
            ADDRESS, JAVA_INT, ADDRESS));

    private SdrGpu()
    {
    }

    /** sdrgpu_init(device): once per process and device, before any handle is created */
    public static void init(int device)
    {
        try
        {
            check((int)INIT.invokeExact(device));
        }
        catch(RuntimeException re)
        {
            throw re;
        }
        catch(Throwable t)
        {
            throw new IllegalStateException(t);
        }
    }

    /** pinned host staging buffer (sdrgpu_alloc_pinned), `bytes` long */
    public static MemorySegment allocPinned(long bytes)
    {
        try(Arena arena = Arena.ofConfined())
        {
            MemorySegment out = arena.allocate(ADDRESS);
            check((int)ALLOC_PINNED.invokeExact(out, bytes));
            return out.get(ADDRESS, 0).reinterpret(bytes);
        }
        catch(RuntimeException re)
        {
            throw re;
        }
        catch(Throwable t)
        {
            throw new IllegalStateException(t);
        }
    }

    /** status -> the exception the replaced Java code threw (include/sdrgpu.h: sdrgpu_status) */
    public static void check(int status)
    {
        if(status == 0)
        {
            return;
        }

        String message;

        try
        {
            message = ((MemorySegment)LAST_ERROR.invokeExact()).reinterpret(512).getString(0);
        }
        catch(Throwable t)
        {
            message = "libsdrgpu status " + status;
        }

        switch(status)
        {
            case 1 -> throw new IllegalArgumentException(message);
            case 2 -> throw new IllegalStateException(message);
            case 4 -> throw new BufferOverflowException();      //caller moves the source to its OVERFLOW state
            case 5 -> throw new IllegalStateException(new FilterDesignException(message));
            default -> throw new IllegalStateException("CUDA: " + message);
        }
    }
}
