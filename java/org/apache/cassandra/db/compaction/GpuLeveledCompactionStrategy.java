/*
 * Table option:  ALTER TABLE ks.t WITH compaction = {'class': 'org.apache.cassandra.db.compaction.GpuLeveledCompactionStrategy'};
 * Resolved by reflection (CompactionParams.java:296-299). Levels, candidates and task selection are LeveledCompactionStrategy's; only the
 * task that EXECUTES a chosen candidate changes: every LeveledCompactionTask that is not a major compaction (LeveledCompactionStrategy.java:170,
 * 209, 225) becomes a GpuCompactionTask with the same level and maxSSTableBytes, whose b200c_compact call switches output files as
 * MaxSSTableSizeWriter does and returns Filter.db / Summary.db / Statistics.db per file. A user-defined level-0 task passes Long.MAX_VALUE:
 * one file, through the same multi-file path. Major compactions (MajorLeveledCompactionWriter moves files up a level while it writes),
 * single-sstable uplevels and anything outside the engine's envelope keep the stock task.
 * Not compiled in the build image (no JDK); see B200C.java for the compile line.
 */
package org.apache.cassandra.db.compaction;

import java.lang.reflect.Field;
import java.util.ArrayList;
import java.util.Collection;
import java.util.Map;

import org.apache.cassandra.db.ColumnFamilyStore;
import org.apache.cassandra.db.lifecycle.LifecycleTransaction;
import org.apache.cassandra.io.sstable.format.SSTableReader;

public class GpuLeveledCompactionStrategy extends LeveledCompactionStrategy
{
    // LeveledCompactionTask keeps these private; the task is built by the strategy, so they are read back from it
    private static final Field MAX_SSTABLE_BYTES = field("maxSSTableBytes"), MAJOR = field("majorCompaction");

    private static Field field(String name)
    {
        try
        {
            Field f = LeveledCompactionTask.class.getDeclaredField(name);
            f.setAccessible(true);
            return f;
        }
        catch (NoSuchFieldException e)
        {
            throw new IllegalStateException("LeveledCompactionTask." + name, e);
        }
    }

    public GpuLeveledCompactionStrategy(ColumnFamilyStore cfs, Map<String, String> options)
    {
        super(cfs, options);
    }

    /** a GpuCompactionTask for a non-major LeveledCompactionTask whose table and inputs the engine covers; the stock task otherwise */
    private AbstractCompactionTask gpuOrStock(AbstractCompactionTask stock)
    {
        if (stock == null || stock.getClass() != LeveledCompactionTask.class)
            return stock;                                               // SingleSSTableLCSTask, or a task of another kind
        LeveledCompactionTask t = (LeveledCompactionTask) stock;
        long maxBytes;
        try
        {
            if (MAJOR.getBoolean(t)) return stock;
            maxBytes = MAX_SSTABLE_BYTES.getLong(t);
        }
        catch (IllegalAccessException e)
        {
            return stock;
        }
        LifecycleTransaction txn = t.transaction;
        if (maxBytes <= 0 || !GpuCompactionTask.supports(cfs, txn.originals()))
            return stock;
        GpuCompactionTask gpu = new GpuCompactionTask(cfs, txn, t.gcBefore, t.getLevel(), maxBytes);
        gpu.setCompactionType(t.compactionType);
        return gpu;
    }

    @Override
    public AbstractCompactionTask getNextBackgroundTask(long gcBefore)
    {
        return gpuOrStock(super.getNextBackgroundTask(gcBefore));
    }

    @Override
    public synchronized Collection<AbstractCompactionTask> getMaximalTask(long gcBefore, boolean splitOutput)
    {
        return super.getMaximalTask(gcBefore, splitOutput);            // major: MajorLeveledCompactionWriter, stock task
    }

    @Override
    public AbstractCompactionTask getUserDefinedTask(Collection<SSTableReader> sstables, long gcBefore)
    {
        return gpuOrStock(super.getUserDefinedTask(sstables, gcBefore));
    }

    @Override
    public AbstractCompactionTask getCompactionTask(LifecycleTransaction txn, long gcBefore, long maxSSTableBytes)
    {
        return gpuOrStock(super.getCompactionTask(txn, gcBefore, maxSSTableBytes));
    }
}
