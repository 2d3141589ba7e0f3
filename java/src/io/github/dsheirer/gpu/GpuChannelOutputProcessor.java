/*
 * IPolyphaseChannelOutputProcessor (J/dsp/filter/channelizer/output/IPolyphaseChannelOutputProcessor.java:27-81) whose
 * work -- ReusableChannelResultsBuffer.getChannel, the frequency-correction Oscillator, the two-bin synthesizer and
 * applyGain (OneChannelOutputProcessor.java:81-106, TwoChannelOutputProcessor.java:98-121) -- has already happened on the
 * GPU inside GpuPolyphaseChannelizer.receive.  The channelizer hands this processor its channel's contiguous I/Q stream;
 * processChannelResults() forwards what has arrived to the channel's ReusableComplexBufferAssembler, on the channel's own
 * thread, exactly where PolyphaseChannelSource.processSamples (J/source/tuner/channel/PolyphaseChannelSource.java:116-157)
 * calls it.
 */
package io.github.dsheirer.gpu;

import io.github.dsheirer.dsp.filter.channelizer.output.IPolyphaseChannelOutputProcessor;
import io.github.dsheirer.sample.buffer.ReusableChannelResultsBuffer;
import io.github.dsheirer.sample.buffer.ReusableComplexBufferAssembler;
import io.github.dsheirer.source.Source;

import java.lang.foreign.MemorySegment;
import java.util.List;
import java.util.concurrent.LinkedTransferQueue;

import static java.lang.foreign.ValueLayout.JAVA_FLOAT;

public class GpuChannelOutputProcessor implements IPolyphaseChannelOutputProcessor
{
    private final GpuPolyphaseChannelizer mChannelizer;
    private final LinkedTransferQueue<float[]> mQueue = new LinkedTransferQueue<>();
    private final double mGain;
    private volatile int mFirstIndex;
    private volatile int mSecondIndex = -1;
    private volatile long mFrequencyOffset;
    private volatile float[] mSynthesisFilter;
    private volatile long mTimestamp;
    private Source mOverflowListener;

    GpuChannelOutputProcessor(GpuPolyphaseChannelizer channelizer, List<Integer> indexes, float[] synthesisFilter, double gain)
    {
        mChannelizer = channelizer;
        mGain = gain;
        mSynthesisFilter = synthesisFilter;
        setPolyphaseChannelIndices(indexes);
    }

    /** called by the channelizer's thread after each sdrgpu_chan_process: row `offsetBytes` of the pinned output */
    void deliver(MemorySegment pinnedOut, long offsetBytes, int floatCount, long timestamp)
    {
        float[] samples = new float[floatCount];
        MemorySegment.copy(pinnedOut, JAVA_FLOAT, offsetBytes, samples, 0, floatCount);
        mTimestamp = timestamp;

        //three seconds of channel samples at most, as ChannelOutputProcessor's OverflowableReusableBufferTransferQueue
        if(mQueue.size() > 600)
        {
            if(mOverflowListener != null)
            {
                mOverflowListener.broadcastOverflowState(true);   //Source.java:104-110
            }

            return;
        }

        mQueue.offer(samples);
    }

    /** not used: the channelizer delivers channel streams, not channel results */
    @Override
    public void receiveChannelResults(ReusableChannelResultsBuffer channelResultsBuffer)
    {
        channelResultsBuffer.decrementUserCount();
    }

    @Override
    public void processChannelResults(ReusableComplexBufferAssembler reusableComplexBufferAssembler)
    {
        float[] samples;

        while((samples = mQueue.poll()) != null)
        {
            reusableComplexBufferAssembler.updateTimestamp(mTimestamp);
            reusableComplexBufferAssembler.receive(samples);
        }
    }

    @Override
    public void setFrequencyOffset(long frequency)
    {
        //only the oscillator's angle changes (ChannelOutputProcessor.java:91-95): applied before the next buffer without
        //re-selecting, so the other channels of the tuner keep their oscillators and synthesizers
        mFrequencyOffset = frequency;
        mChannelizer.frequencyOffsetChanged(this);
    }

    @Override
    public int getInputChannelCount()
    {
        return mSecondIndex >= 0 ? 2 : 1;
    }

    @Override
    public void setPolyphaseChannelIndices(List<Integer> indexes)
    {
        if(indexes.size() != 1 && indexes.size() != 2)
        {
            throw new IllegalArgumentException("Output processor requires one or two channel indexes - provided indexes " + indexes);
        }

        mFirstIndex = indexes.get(0);
        mSecondIndex = indexes.size() == 2 ? indexes.get(1) : -1;
        mChannelizer.selectionChanged();
    }

    @Override
    public int getPolyphaseChannelIndexCount()
    {
        return getInputChannelCount();
    }

    @Override
    public void setSynthesisFilter(float[] filter)
    {
        if(mSecondIndex < 0)
        {
            throw new IllegalArgumentException("The one channel output processor does not support filter updates");
        }

        mSynthesisFilter = filter;
        mChannelizer.selectionChanged();
    }

    @Override
    public void setSourceOverflowListener(Source source)
    {
        mOverflowListener = source;
    }

    @Override
    public void dispose()
    {
        mChannelizer.remove(this);
        mQueue.clear();
    }

    int getFirstIndex()
    {
        return mFirstIndex;
    }

    int getSecondIndex()
    {
        return mSecondIndex;
    }

    long getFrequencyOffset()
    {
        return mFrequencyOffset;
    }

    double getGain()
    {
        return mGain;
    }

    float[] getSynthesisFilter()
    {
        return mSecondIndex >= 0 ? mSynthesisFilter : null;
    }
}
