/*
 * GPU-backed replacement of ComplexPolyphaseChannelizerM2 (J/dsp/filter/channelizer/ComplexPolyphaseChannelizerM2.java:
 * 93-235, 337-428): same constructor arguments, same Listener<ReusableComplexBuffer> input, same base class.  The filter
 * bank, the inverse DFT and -- for the channels whose output processor is a GpuChannelOutputProcessor -- the channel
 * extraction, frequency-correction mix, two-bin synthesis and gain run in one sdrgpu_chan_process call per tuner buffer
 * (channel layout); each registered processor then receives its own contiguous channel stream.
 */
package io.github.dsheirer.gpu;

import io.github.dsheirer.dsp.filter.FilterFactory;
import io.github.dsheirer.dsp.filter.channelizer.AbstractComplexPolyphaseChannelizer;
import io.github.dsheirer.dsp.filter.channelizer.ComplexPolyphaseChannelizerM2;
import io.github.dsheirer.dsp.filter.design.FilterDesignException;
import io.github.dsheirer.sample.buffer.ReusableComplexBuffer;

import java.lang.foreign.Arena;
import java.lang.foreign.MemorySegment;
import java.util.ArrayList;
import java.util.List;
import java.util.concurrent.ConcurrentLinkedQueue;
import java.util.concurrent.CopyOnWriteArrayList;

import static java.lang.foreign.ValueLayout.ADDRESS;
import static java.lang.foreign.ValueLayout.JAVA_FLOAT;
import static java.lang.foreign.ValueLayout.JAVA_INT;
import static java.lang.foreign.ValueLayout.JAVA_LONG;

public class GpuPolyphaseChannelizer extends AbstractComplexPolyphaseChannelizer
{
    private static final double CHANNEL_BANDWIDTH = 25000.0;   //ComplexPolyphaseChannelizerM2.java: 25 kHz channels, 2x oversampled

    private final Arena mArena = Arena.ofShared();
    private final List<GpuChannelOutputProcessor> mProcessors = new CopyOnWriteArrayList<>();
    private MemorySegment mHandle;
    private MemorySegment mPinnedIn;
    private MemorySegment mPinnedOut;
    private MemorySegment mBlockCount;
    private int mMaxInputFloats;
    private int mMaxBlocks;
    private boolean mSelectionChanged = true;
    //the processors as of the last selection (and whether each had two bins then), and the synthesis filter it carried
    private final List<GpuChannelOutputProcessor> mSelected = new ArrayList<>();
    private final List<Boolean> mSelectedTwoBin = new ArrayList<>();
    private float[] mSelectedFilter;
    private final ConcurrentLinkedQueue<GpuChannelOutputProcessor> mOffsetsChanged = new ConcurrentLinkedQueue<>();

    /**
     * @param taps prototype low-pass filter, channelCount * tapsPerChannel long (FilterFactory.getSincM2Channelizer)
     * @param sampleRate of the tuner stream
     * @param channelCount even number of polyphase channels
     * @param maxInputFloats largest tuner buffer (interleaved floats) that receive() will be handed
     */
    public GpuPolyphaseChannelizer(float[] taps, int sampleRate, int channelCount, int maxInputFloats)
    {
        super(sampleRate, channelCount);
        create(taps, sampleRate, channelCount, maxInputFloats);
    }

    /** As ComplexPolyphaseChannelizerM2(double sampleRate, int tapsPerChannel) (:114-126) */
    public GpuPolyphaseChannelizer(double sampleRate, int tapsPerChannel, int maxInputFloats) throws FilterDesignException
    {
        super(sampleRate, ComplexPolyphaseChannelizerM2.getChannelCount(sampleRate));
        float[] taps = FilterFactory.getSincM2Channelizer(CHANNEL_BANDWIDTH, getChannelCount(), tapsPerChannel, false);
        create(taps, (int)sampleRate, getChannelCount(), maxInputFloats);
    }

    private void create(float[] taps, int sampleRate, int channelCount, int maxInputFloats)
    {
        mMaxInputFloats = maxInputFloats;
        mMaxBlocks = maxInputFloats / channelCount + 2;     //one block per channelCount / 2 complex samples
        try
        {
            MemorySegment out = mArena.allocate(ADDRESS);
            MemorySegment nativeTaps = mArena.allocateFrom(JAVA_FLOAT, taps);
            //status 1 -> the IllegalArgumentException of ComplexPolyphaseChannelizerM2.java:97-100 for an odd channel count
            SdrGpu.check((int)SdrGpu.CHAN_CREATE.invokeExact(out, nativeTaps, taps.length, channelCount, maxInputFloats));
            mHandle = out.get(ADDRESS, 0);
            SdrGpu.check((int)SdrGpu.CHAN_SET_SAMPLE_RATE.invokeExact(mHandle, (double)sampleRate));
        }
        catch(RuntimeException re)
        {
            throw re;
        }
        catch(Throwable t)
        {
            throw new IllegalStateException(t);
        }

        mPinnedIn = SdrGpu.allocPinned(4L * maxInputFloats);
        mBlockCount = mArena.allocate(JAVA_INT);
    }

    /** Output processor factory used in place of PolyphaseChannelManager.getOutputProcessor (:198-222) */
    public GpuChannelOutputProcessor getOutputProcessor(List<Integer> indexes, float[] synthesisFilter)
    {
        GpuChannelOutputProcessor processor = new GpuChannelOutputProcessor(this, indexes, synthesisFilter, getChannelCount());
        mProcessors.add(processor);
        mSelectionChanged = true;
        return processor;
    }

    void remove(GpuChannelOutputProcessor processor)
    {
        mProcessors.remove(processor);
        mSelectionChanged = true;
    }

    void selectionChanged()
    {
        mSelectionChanged = true;
    }

    /** a registered processor's offset changed: sent with the others changed since the last buffer (updateOffsets) */
    void frequencyOffsetChanged(GpuChannelOutputProcessor processor)
    {
        mOffsetsChanged.add(processor);
    }

    /**
     * sdrgpu_chan_set_frequency_offsets for the processors whose offset changed since the last buffer: the index of each
     * in the selection (registration order) and its current offset.  Not needed after a re-selection, which carries the
     * offsets itself.
     */
    private void updateOffsets() throws Throwable
    {
        List<GpuChannelOutputProcessor> processors = mProcessors;
        List<Integer> indexes = new ArrayList<>();
        List<Long> offsets = new ArrayList<>();
        GpuChannelOutputProcessor changed;

        while((changed = mOffsetsChanged.poll()) != null)
        {
            int index = processors.indexOf(changed);

            if(index >= 0 && !indexes.contains(index))
            {
                indexes.add(index);
                offsets.add(changed.getFrequencyOffset());
            }
        }

        if(indexes.isEmpty())
        {
            return;
        }

        try(Arena arena = Arena.ofConfined())
        {
            int n = indexes.size();
            MemorySegment nativeIndexes = arena.allocate(JAVA_INT, n);
            MemorySegment nativeOffsets = arena.allocate(JAVA_LONG, n);

            for(int i = 0; i < n; i++)
            {
                nativeIndexes.setAtIndex(JAVA_INT, i, indexes.get(i));
                nativeOffsets.setAtIndex(JAVA_LONG, i, offsets.get(i));
            }

            SdrGpu.check((int)SdrGpu.CHAN_SET_FREQUENCY_OFFSETS.invokeExact(mHandle, nativeIndexes, nativeOffsets, n));
        }
    }

    /**
     * One sdrgpu_output_channel per registered processor, in registration order.  sdrgpu_chan_update_selection with each
     * processor's index in the last selection (-1 for a new one), so that processors carry on across additions, removals
     * and setPolyphaseChannelIndices as in PolyphaseChannelManager; sdrgpu_chan_select only for the first selection and
     * for a new synthesis filter while two-bin processors are kept, which restarts them.
     */
    private void updateSelection() throws Throwable
    {
        List<GpuChannelOutputProcessor> processors = mProcessors;
        int n = processors.size();

        if(n == 0)
        {
            return;
        }

        try(Arena arena = Arena.ofConfined())
        {
            MemorySegment channels = arena.allocate(SdrGpu.OUTPUT_CHANNEL, n);
            MemorySegment previous = arena.allocate(JAVA_INT, n);
            float[] synthesis = null;
            boolean keptTwoBin = false;

            for(int i = 0; i < n; i++)
            {
                GpuChannelOutputProcessor p = processors.get(i);
                MemorySegment c = channels.asSlice(i * SdrGpu.OUTPUT_CHANNEL.byteSize(), SdrGpu.OUTPUT_CHANNEL.byteSize());
                c.set(JAVA_INT, 0, p.getFirstIndex());
                c.set(JAVA_INT, 4, p.getSecondIndex());                //-1 for a one-bin channel
                c.set(java.lang.foreign.ValueLayout.JAVA_LONG, 8, p.getFrequencyOffset());
                c.set(java.lang.foreign.ValueLayout.JAVA_DOUBLE, 16, p.getGain());

                if(p.getSynthesisFilter() != null)
                {
                    synthesis = p.getSynthesisFilter();
                }

                //a processor moved to a different bin count continues as a new channel
                int index = mSelected.indexOf(p);
                boolean twoBin = p.getSecondIndex() >= 0;

                if(index >= 0 && mSelectedTwoBin.get(index) != twoBin)
                {
                    index = -1;
                }

                keptTwoBin |= index >= 0 && twoBin;
                previous.setAtIndex(JAVA_INT, i, index);
            }

            boolean newFilter = synthesis != null && synthesis != mSelectedFilter;
            boolean select = mSelected.isEmpty() || (newFilter && keptTwoBin);
            //sdrgpu_chan_select takes the filter every time, an update only when it changed (NULL keeps the current one)
            boolean passFilter = synthesis != null && (select || newFilter);
            MemorySegment filter = passFilter ? arena.allocateFrom(JAVA_FLOAT, synthesis) : MemorySegment.NULL;
            int filterLength = passFilter ? synthesis.length : 0;

            if(select)
            {
                SdrGpu.check((int)SdrGpu.CHAN_SELECT.invokeExact(mHandle, channels, n, filter, filterLength));
            }
            else
            {
                SdrGpu.check((int)SdrGpu.CHAN_UPDATE_SELECTION.invokeExact(mHandle, channels, previous, n, filter, filterLength));
            }

            mSelected.clear();
            mSelectedTwoBin.clear();

            for(GpuChannelOutputProcessor p : processors)
            {
                mSelected.add(p);
                mSelectedTwoBin.add(p.getSecondIndex() >= 0);
            }

            if(synthesis != null)
            {
                mSelectedFilter = synthesis;
            }
        }

        long outBytes = 8L * mMaxBlocks * n;

        if(mPinnedOut == null || mPinnedOut.byteSize() < outBytes)
        {
            mPinnedOut = SdrGpu.allocPinned(outBytes);
        }

        mSelectionChanged = false;
    }

    /**
     * Primary input: a buffer of interleaved I/Q tuner samples (ComplexPolyphaseChannelizerM2.receive, :190-235).
     */
    @Override
    public void receive(ReusableComplexBuffer reusableComplexBuffer)
    {
        float[] samples = reusableComplexBuffer.getSamples();

        try
        {
            if(mSelectionChanged)
            {
                mOffsetsChanged.clear();   //the selection update carries every processor's current offset
                updateSelection();
            }
            else
            {
                updateOffsets();
            }

            List<GpuChannelOutputProcessor> processors = mProcessors;
            int n = processors.size();

            if(n > 0)
            {
                if(samples.length > mMaxInputFloats)
                {
                    throw new java.nio.BufferOverflowException();
                }

                MemorySegment.copy(samples, 0, mPinnedIn, JAVA_FLOAT, 0, samples.length);
                long stride = 2L * mMaxBlocks;
                SdrGpu.check((int)SdrGpu.CHAN_PROCESS.invokeExact(mHandle, mPinnedIn, samples.length, SdrGpu.HOST, mPinnedOut,
                    stride, SdrGpu.HOST, SdrGpu.LAYOUT_CHANNELS, mBlockCount));
                int blocks = mBlockCount.get(JAVA_INT, 0);

                for(int i = 0; i < n; i++)
                {
                    processors.get(i).deliver(mPinnedOut, 4L * stride * i, 2 * blocks, reusableComplexBuffer.getTimestamp());
                }
            }
        }
        catch(RuntimeException re)
        {
            throw re;
        }
        catch(Throwable t)
        {
            throw new IllegalStateException(t);
        }
        finally
        {
            reusableComplexBuffer.decrementUserCount();
        }
    }

    @Override
    public void setRates(double sampleRate, int channelCount)
    {
        if(channelCount != getChannelCount())
        {
            throw new IllegalArgumentException("a GPU channelizer handle is created for one channel count: create a new one");
        }

        super.setRates(sampleRate, channelCount);

        try
        {
            SdrGpu.check((int)SdrGpu.CHAN_SET_SAMPLE_RATE.invokeExact(mHandle, sampleRate));
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

    public void start()
    {
    }

    public void stop()
    {
    }

    public void dispose()
    {
        try
        {
            SdrGpu.check((int)SdrGpu.CHAN_DESTROY.invokeExact(mHandle));
            SdrGpu.check((int)SdrGpu.FREE_PINNED.invokeExact(mPinnedIn));

            if(mPinnedOut != null)
            {
                SdrGpu.check((int)SdrGpu.FREE_PINNED.invokeExact(mPinnedOut));
            }
        }
        catch(RuntimeException re)
        {
            throw re;
        }
        catch(Throwable t)
        {
            throw new IllegalStateException(t);
        }

        mArena.close();
    }
}
