/*
 * GpuCompactionTask — CompactionTask.runMayThrow (S/db/compaction/CompactionTask.java:114-285) with the merge loop
 *     while (ci.hasNext()) writer.append(ci.next());                                   (:213-231)
 * replaced by ONE call of b200c_compact (include/b200c.h). Everything around the loop stays the reference's: the transaction owns the
 * inputs, the controller decides gcBefore / purgeability / fully expired sstables, outputs are tracked by the LifecycleTransaction and
 * opened as SSTableReaders, compaction_history and the metrics are updated by the inherited code paths.
 *
 * Not compiled in the build image (no JDK); see B200C.java for the compile line. What the native side guarantees is exercised through
 * the same C ABI from Python (tests/test_gpu_compaction.py) and this class only moves addresses and lengths.
 */
package org.apache.cassandra.db.compaction;

import java.io.IOException;
import java.nio.ByteBuffer;
import java.nio.ByteOrder;
import java.nio.MappedByteBuffer;
import java.nio.channels.FileChannel;
import java.nio.file.StandardOpenOption;
import java.util.ArrayList;
import java.util.Collection;
import java.util.EnumMap;
import java.util.List;
import java.util.Map;
import java.util.Set;

import org.apache.cassandra.config.DatabaseDescriptor;
import org.apache.cassandra.db.Directories;
import org.apache.cassandra.db.compaction.writers.CompactionAwareWriter;
import org.apache.cassandra.db.compaction.writers.MaxSSTableSizeWriter;
import org.apache.cassandra.db.ColumnFamilyStore;
import org.apache.cassandra.db.SerializationHeader;
import org.apache.cassandra.db.Slice;
import org.apache.cassandra.db.commitlog.CommitLogPosition;
import org.apache.cassandra.db.commitlog.IntervalSet;
import org.apache.cassandra.db.lifecycle.LifecycleTransaction;
import org.apache.cassandra.db.marshal.AbstractType;
import org.apache.cassandra.db.rows.EncodingStats;
import org.apache.cassandra.dht.ByteOrderedPartitioner;
import org.apache.cassandra.dht.Murmur3Partitioner;
import org.apache.cassandra.io.compress.CompressionMetadata;
import org.apache.cassandra.io.sstable.Component;
import org.apache.cassandra.io.sstable.CorruptSSTableException;
import org.apache.cassandra.io.sstable.Descriptor;
import org.apache.cassandra.io.sstable.format.SSTableFormat.Components;
import org.apache.cassandra.io.sstable.format.SSTableReader;
import org.apache.cassandra.io.sstable.format.big.BigFormat;
import org.apache.cassandra.io.sstable.format.big.BigTableReader;
import org.apache.cassandra.io.sstable.indexsummary.IndexSummary;
import org.apache.cassandra.io.sstable.metadata.CompactionMetadata;
import org.apache.cassandra.io.sstable.metadata.MetadataComponent;
import org.apache.cassandra.io.sstable.metadata.MetadataType;
import org.apache.cassandra.io.sstable.metadata.StatsMetadata;
import org.apache.cassandra.io.sstable.metadata.ValidationMetadata;
import org.apache.cassandra.io.util.DataOutputStreamPlus;
import org.apache.cassandra.io.util.File;
import org.apache.cassandra.io.util.FileOutputStreamPlus;
import org.apache.cassandra.schema.ColumnMetadata;
import org.apache.cassandra.schema.CompressionParams;
import org.apache.cassandra.schema.TableMetadata;
import org.apache.cassandra.service.ActiveRepairService;
import org.apache.cassandra.utils.EstimatedHistogram;
import org.apache.cassandra.utils.FBUtilities;
import org.apache.cassandra.utils.streamhist.StreamingTombstoneHistogramBuilder;

import com.clearspring.analytics.stream.cardinality.HyperLogLogPlus;
import com.clearspring.analytics.stream.cardinality.ICardinality;

import static org.apache.cassandra.db.compaction.B200C.Layout.*;

public class GpuCompactionTask extends CompactionTask
{
    private final int level;                 // level of the output sstables (Statistics.db sstableLevel)
    private final long maxSSTableBytes;      // 0: one output (DefaultCompactionWriter); else MaxSSTableSizeWriter's switch limit, Long.MAX_VALUE included

    public GpuCompactionTask(ColumnFamilyStore cfs, LifecycleTransaction txn, long gcBefore)
    {
        this(cfs, txn, gcBefore, 0, 0L);
    }

    /** a leveled task (LeveledCompactionTask without majorCompaction): outputs of at most maxSSTableBytes on disk, written at `level` */
    public GpuCompactionTask(ColumnFamilyStore cfs, LifecycleTransaction txn, long gcBefore, int level, long maxSSTableBytes)
    {
        super(cfs, txn, gcBefore);
        this.level = level;
        this.maxSSTableBytes = maxSSTableBytes;
    }

    @Override
    protected int getLevel()
    {
        return level;
    }

    /** the writer of the stock path (super.runMayThrow() after B200C_EUNSUPPORTED): a leveled task keeps LeveledCompactionTask's
     *  MaxSSTableSizeWriter (LeveledCompactionTask.java:46-54), so the fallback writes files of maxSSTableBytes at the task's level too */
    @Override
    public CompactionAwareWriter getCompactionAwareWriter(ColumnFamilyStore cfs, Directories directories, LifecycleTransaction txn, Set<SSTableReader> nonExpiredSSTables)
    {
        if (maxSSTableBytes > 0)
            return new MaxSSTableSizeWriter(cfs, directories, txn, nonExpiredSSTables, maxSSTableBytes, level, false);
        return super.getCompactionAwareWriter(cfs, directories, txn, nonExpiredSSTables);
    }

    @Override
    protected boolean partialCompactionsAcceptable()
    {
        return maxSSTableBytes > 0 ? level == 0 : super.partialCompactionsAcceptable();     // LeveledCompactionTask.partialCompactionsAcceptable
    }

    // ---- the envelope of include/b200c.h, checked BEFORE a task is built so that unsupported tables keep the stock task -------------------
    public static boolean supports(ColumnFamilyStore cfs, Set<SSTableReader> inputs)
    {
        TableMetadata t = cfs.metadata();
        if (inputs.isEmpty() || inputs.size() > B200C.MAX_INPUTS) return false;
        if (!(t.partitioner instanceof Murmur3Partitioner) && !(t.partitioner instanceof ByteOrderedPartitioner)) return false;
        if (t.isIndex() || t.staticColumns().size() > B200C.MAX_STATIC_COLUMNS) return false;
        for (ColumnMetadata c : t.staticColumns())
            if (c.isComplex() || columnClass(c.type) < 0) return false;                          // (simple static columns, counters included; multi-cell static columns keep the stock task)
        if (t.clusteringColumns().size() > B200C.MAX_CLUSTERING || t.regularColumns().size() >= B200C.MAX_COLUMNS) return false;
        int complex = 0;
        for (ColumnMetadata c : t.regularColumns())
        {
            if (c.isComplex()) { if (columnClass(c.type) < 0 || ++complex > B200C.MAX_COMPLEX_COLUMNS) return false; }
            else if (columnClass(c.type) < 0) return false;
        }
        for (ColumnMetadata c : t.clusteringColumns())
            if (clusteringClass(c.type) < 0) return false;
        if (cfs.getCompactionStrategyManager().getCompactionParams().tombstoneOption() != org.apache.cassandra.schema.CompactionParams.TombstoneOption.NONE) return false;
        if (t.enforceStrictLiveness()) return false;
        for (SSTableReader r : inputs)
        {
            if (!(r instanceof BigTableReader) || !r.descriptor.version.version.equals("oa")) return false;
            if (!r.compression) return false;
            String comp = r.getCompressionMetadata().parameters.getSstableCompressor().getClass().getSimpleName();
            if (compressorId(comp) < 0 || r.getCompressionMetadata().chunkLength() > 65536) return false;
        }
        return B200C.deviceCount() > 0;
    }

    static int compressorId(String simpleName)
    {
        if (simpleName.endsWith("LZ4Compressor")) return B200C.COMP_LZ4;
        if (simpleName.endsWith("SnappyCompressor")) return B200C.COMP_SNAPPY;
        return -1;
    }

    /** comparison / layout class of a value type (b200c.h B200C_TYPE_*): -1 = outside the envelope */
    static int typeClass(AbstractType<?> type)
    {
        String n = type.getClass().getSimpleName();
        switch (n)
        {
            case "LongType": case "TimestampType": case "Int32Type": return B200C.TYPE_FIXED_SIGNED;
            case "DateType": case "DoubleType": case "FloatType": case "BooleanType": case "UUIDType": case "TimeUUIDType": case "LexicalUUIDType": return B200C.TYPE_FIXED_BYTES;
            case "ShortType": case "ByteType": return B200C.TYPE_VAR_SIGNED;
            case "UTF8Type": case "AsciiType": case "BytesType": return B200C.TYPE_BYTES;
            default: return -1;
        }
    }

    /** b200c_column.type / .fixed_len of a regular column: simple columns as typeClass; multi-cell collections (map / set / list) as
     *  B200C_COLUMN_COMPLEX(value class, path class) / B200C_COLUMN_FIXED(value length, path length) — include/b200c.h. The cell path is
     *  CollectionType.nameComparator() (map key, set element, list timeuuid), the cell value CollectionType.valueComparator(). -1: refused
     *  (non-frozen UDTs, element types outside the envelope). Frozen collections are single opaque values. */
    static int columnClass(AbstractType<?> type)
    {
        if (type.isCounter()) return B200C.TYPE_COUNTER;                 // counter context: merged shard by shard (Cells.resolveCounter), variable length
        if (!type.isMultiCell()) return type.isCollection() || type.isUDT() ? B200C.TYPE_BYTES : typeClass(type);
        if (!(type instanceof org.apache.cassandra.db.marshal.CollectionType)) return -1;
        org.apache.cassandra.db.marshal.CollectionType<?> ct = (org.apache.cassandra.db.marshal.CollectionType<?>) type;
        int path = ct.kind == org.apache.cassandra.db.marshal.CollectionType.Kind.LIST ? B200C.TYPE_TIMEUUID : elementClass(ct.nameComparator());
        int value = ct.kind == org.apache.cassandra.db.marshal.CollectionType.Kind.SET ? B200C.TYPE_BYTES : elementClass(ct.valueComparator());
        return path < 0 || value < 0 ? -1 : value | ((path + 1) << 8);
    }
    static int columnFixedLen(AbstractType<?> type)
    {
        if (!type.isMultiCell()) return type.isCollection() || type.isUDT() ? 0 : Math.max(0, type.valueLengthIfFixed());
        org.apache.cassandra.db.marshal.CollectionType<?> ct = (org.apache.cassandra.db.marshal.CollectionType<?>) type;
        int path = ct.kind == org.apache.cassandra.db.marshal.CollectionType.Kind.LIST ? 16 : elementFixedLen(ct.nameComparator());
        int value = ct.kind == org.apache.cassandra.db.marshal.CollectionType.Kind.SET ? 0 : elementFixedLen(ct.valueComparator());
        return value | (path << 16);
    }
    private static int elementClass(AbstractType<?> t) { return t.isCollection() || t.isUDT() ? B200C.TYPE_BYTES : typeClass(t); }       // (frozen inside a collection)
    private static int elementFixedLen(AbstractType<?> t) { return t.isCollection() || t.isUDT() ? 0 : Math.max(0, t.valueLengthIfFixed()); }

    /** clustering columns additionally need a comparison the engine implements: signed integers or unsigned bytes */
    static int clusteringClass(AbstractType<?> type)
    {
        if (type.isReversed()) return -1;
        switch (type.getClass().getSimpleName())
        {
            case "LongType": case "TimestampType": case "Int32Type": case "DateType": case "ShortType": case "ByteType": case "UTF8Type": case "AsciiType": case "BytesType":
                return typeClass(type);
            default: return -1;
        }
    }

    // ---- one input sstable: component files mapped (and pinned once), chunk offsets and summary positions in native order --------------------
    private static final class Input implements AutoCloseable
    {
        final SSTableReader reader;
        final MappedByteBuffer data, index;
        final ByteBuffer chunkOffsets, summaryPositions;
        final long nChunks, nSummary;

        Input(SSTableReader r) throws IOException
        {
            reader = r;
            data = map(r.descriptor.fileFor(Components.DATA));
            index = map(r.descriptor.fileFor(BigFormat.Components.PRIMARY_INDEX));
            // CompressionInfo.db: UTF name | i32 nOpts | (UTF,UTF)* | i32 chunkLength | i32 maxCompressedLength | i64 dataLength | i32 n | i64 offset x n (BE)
            CompressionMetadata cm = r.getCompressionMetadata();
            ByteBuffer info = map(r.descriptor.fileFor(Components.COMPRESSION_INFO)).order(ByteOrder.BIG_ENDIAN);
            int p = 2 + (info.getShort(0) & 0xFFFF);
            int nOpts = info.getInt(p); p += 4;
            for (int i = 0; i < 2 * nOpts; i++) p += 2 + (info.getShort(p) & 0xFFFF);
            p += 4 + 4 + 8;
            int n = info.getInt(p); p += 4;
            nChunks = n;
            chunkOffsets = B200C.struct(8 * Math.max(n, 1));
            for (int i = 0; i < n; i++) chunkOffsets.putLong(8 * i, info.getLong(p + 8 * i));
            assert cm.dataLength >= 0;
            // Summary.db sample positions: already in memory for every open big-format reader (IndexSummary.getPosition :190-193)
            IndexSummary s = ((BigTableReader) r).getIndexSummary();
            nSummary = s.size();
            summaryPositions = B200C.struct(8 * Math.max(s.size(), 1));
            for (int i = 0; i < s.size(); i++) summaryPositions.putLong(8 * i, s.getPosition(i));
            B200C.hostRegister(B200C.address(data), data.capacity());
            B200C.hostRegister(B200C.address(index), index.capacity());
        }

        static MappedByteBuffer map(File f) throws IOException
        {
            try (FileChannel ch = FileChannel.open(f.toPath(), StandardOpenOption.READ))
            {
                return ch.map(FileChannel.MapMode.READ_ONLY, 0, ch.size());
            }
        }

        public void close()
        {
            B200C.hostUnregister(B200C.address(data));
            B200C.hostUnregister(B200C.address(index));
        }
    }

    @Override
    protected void runMayThrow() throws Exception
    {
        if (transaction.originals().isEmpty())
            return;
        final long ctx = B200C.context();
        B200C.cancelReset(ctx);                                   // a new task is bound to this context (b200c.h: sticky cancel)

        try (CompactionController controller = getCompactionController(transaction.originals()))
        {
            Set<SSTableReader> fullyExpired = controller.getFullyExpiredSSTables();
            List<SSTableReader> actuallyCompact = new ArrayList<>(com.google.common.collect.Sets.difference(transaction.originals(), fullyExpired));
            actuallyCompact.sort((a, b) -> a.descriptor.id.toString().compareTo(b.descriptor.id.toString()));
            final long nowInSec = FBUtilities.nowInSeconds();      // :183 — the determinism input of the run
            final TableMetadata table = cfs.metadata();
            final SerializationHeader header = SerializationHeader.make(table, actuallyCompact);       // SerializationHeader.java:77-100
            final EncodingStats outStats = header.stats();
            final List<ColumnMetadata> outColumns = new ArrayList<>();
            header.columns().regulars.forEach(outColumns::add);
            final List<ColumnMetadata> outStatics = new ArrayList<>();
            header.columns().statics.forEach(outStatics::add);

            List<Input> inputs = new ArrayList<>();
            try
            {
                for (SSTableReader r : actuallyCompact) inputs.add(new Input(r));
                // ---- manifest --------------------------------------------------------------------------------------------------------------
                ByteBuffer in = B200C.struct(SIZEOF_INPUT * inputs.size());
                long totalIn = 0, totalIndex = 0, totalCompressed = 0;
                for (int i = 0; i < inputs.size(); i++)
                {
                    Input s = inputs.get(i); int o = i * SIZEOF_INPUT;
                    CompressionMetadata cm = s.reader.getCompressionMetadata();
                    in.putLong(o + IN_DATA, B200C.address(s.data)).putLong(o + IN_DATA_LEN, s.data.capacity());
                    in.putLong(o + IN_INDEX, B200C.address(s.index)).putLong(o + IN_INDEX_LEN, s.index.capacity());
                    in.putLong(o + IN_CHUNK_OFFSETS, B200C.address(s.chunkOffsets)).putLong(o + IN_NCHUNKS, s.nChunks);
                    in.putLong(o + IN_DATA_LENGTH, cm.dataLength);
                    in.putInt(o + IN_COMPRESSOR, compressorId(cm.parameters.getSstableCompressor().getClass().getSimpleName()));
                    in.putInt(o + IN_CHUNK_LEN, cm.chunkLength()).putInt(o + IN_MAX_COMPRESSED_LEN, cm.maxCompressedLength());
                    List<ColumnMetadata> have = new ArrayList<>();
                    s.reader.header.columns().regulars.forEach(have::add);
                    in.putInt(o + IN_NCOLUMNS, have.size());
                    for (int c = 0; c < have.size(); c++) in.putInt(o + IN_COLUMN_MAP + 4 * c, outColumns.indexOf(have.get(c)));
                    List<ColumnMetadata> haveStatic = new ArrayList<>();
                    s.reader.header.columns().statics.forEach(haveStatic::add);
                    in.putInt(o + IN_NSTATIC_COLUMNS, haveStatic.size());
                    for (int c = 0; c < haveStatic.size(); c++) in.putInt(o + IN_STATIC_COLUMN_MAP + 4 * c, outStatics.indexOf(haveStatic.get(c)));
                    EncodingStats hs = s.reader.header.stats();
                    in.putLong(o + IN_HEADER_STATS, hs.minTimestamp).putLong(o + IN_HEADER_STATS + 8, hs.minLocalDeletionTime).putInt(o + IN_HEADER_STATS + 16, hs.minTTL);
                    in.putInt(o + IN_LEVEL, s.reader.getSSTableLevel());
                    in.putLong(o + IN_SUMMARY_POSITIONS, B200C.address(s.summaryPositions)).putLong(o + IN_NSUMMARY, s.nSummary);
                    totalIn += cm.dataLength; totalIndex += s.index.capacity(); totalCompressed += s.data.capacity();
                }
                CompressionParams cp = table.params.compression;
                int outComp = compressorId(cp.getSstableCompressor().getClass().getSimpleName());
                ByteBuffer m = B200C.struct(SIZEOF_MANIFEST);
                m.putInt(M_ABI_VERSION, B200C.ABI_VERSION).putInt(M_NINPUTS, inputs.size()).putLong(M_INPUTS, B200C.address(in));
                m.putInt(M_NCLUSTERING, table.clusteringColumns().size());
                for (int k = 0; k < table.clusteringColumns().size(); k++)
                {
                    AbstractType<?> t = table.clusteringColumns().get(k).type;
                    m.putInt(M_CLUSTERING + 8 * k, clusteringClass(t)).putInt(M_CLUSTERING + 8 * k + 4, Math.max(0, t.valueLengthIfFixed()));
                }
                m.putInt(M_NCOLUMNS, outColumns.size());
                for (int k = 0; k < outColumns.size(); k++)
                    m.putInt(M_COLUMNS + 8 * k, columnClass(outColumns.get(k).type)).putInt(M_COLUMNS + 8 * k + 4, columnFixedLen(outColumns.get(k).type));      // (header order: simple columns, then multi-cell ones)
                m.putInt(M_NSTATIC_COLUMNS, outStatics.size());
                for (int k = 0; k < outStatics.size(); k++)
                    m.putInt(M_STATIC_COLUMNS + 8 * k, columnClass(outStatics.get(k).type)).putInt(M_STATIC_COLUMNS + 8 * k + 4, Math.max(0, outStatics.get(k).type.valueLengthIfFixed()));
                m.putLong(M_OUT_STATS, outStats.minTimestamp).putLong(M_OUT_STATS + 8, outStats.minLocalDeletionTime).putInt(M_OUT_STATS + 16, outStats.minTTL);
                m.putInt(M_OUT_COMPRESSOR, outComp).putInt(M_OUT_CHUNK_LEN, cp.chunkLength()).putInt(M_OUT_MAX_COMPRESSED_LEN, cp.maxCompressedLength());
                m.putInt(M_COLUMN_INDEX_SIZE, DatabaseDescriptor.getColumnIndexSize(BigFormat.getInstance().getDefaultColumnIndexSize()));
                m.putLong(M_NOW_IN_SEC, nowInSec).putLong(M_GC_BEFORE, controller.gcBefore);
                // purge evaluator: min timestamp over the live sstables / memtables that overlap the compaction (CompactionController.java:247-286).
                // One threshold for the whole ring here; a host that wants the per-key precision fills purge_range_* per token range.
                long purgeMax = Long.MAX_VALUE;
                for (SSTableReader o : cfs.getOverlappingLiveSSTables(actuallyCompact)) purgeMax = Math.min(purgeMax, o.getMinTimestamp());
                for (org.apache.cassandra.db.memtable.Memtable mt : cfs.getTracker().getView().getAllMemtables()) purgeMax = Math.min(purgeMax, mt.getMinTimestamp());
                m.putLong(M_PURGE_MAX_TIMESTAMP, controller.compactingRepaired() ? purgeMax : Long.MIN_VALUE);   // only_purge_repaired_tombstones: nothing purgeable
                m.putLong(M_TOKEN_LO, Long.MIN_VALUE).putLong(M_TOKEN_HI, Long.MAX_VALUE);
                m.putLong(M_MAX_SSTABLE_BYTES, maxSSTableBytes);    // 0: DefaultCompactionWriter (STCS); LCS: MaxSSTableSizeWriter, one output per file
                m.putInt(M_PARTITIONER, table.partitioner instanceof Murmur3Partitioner ? B200C.PARTITIONER_MURMUR3 : B200C.PARTITIONER_BYTE_ORDERED);
                // Filter.db geometry as SortedTableWriter would choose it (FilterFactory.getFilter(estimatedKeys, fpChance))
                long estimatedKeys = Math.max(1, SSTableReader.getApproximateKeyCount(actuallyCompact));
                if (maxSSTableBytes > 0)                            // MaxSSTableSizeWriter: every file's filter is sized for keysPerSSTable (CompactionAwareWriter.sstableKeyCount)
                    estimatedKeys = Math.max(1, estimatedKeys / Math.max(1, expectedWriteSize(actuallyCompact, estimatedKeys) / maxSSTableBytes));
                double fp = table.params.bloomFilterFpChance;
                int[] spec = BloomSpec.of(estimatedKeys, fp);
                m.putInt(M_BLOOM_HASH_COUNT, spec[0]).putLong(M_BLOOM_WORDS, fp >= 1.0 ? 0L : ((estimatedKeys * spec[1] + 20 - 1) >>> 6) + 1);
                m.putInt(M_MIN_INDEX_INTERVAL, table.params.minIndexInterval);

                // ---- result + caller-provided output buffers ------------------------------------------------------------------------------------
                // one output slot per file: a single-output task gets buffers for the whole stream; a leveled one starts from the file limit and,
                // on B200C_ETOOSMALL, calls again with the number of files and the sizes the engine reported (required_*_cap, *_len of each slot)
                long dataCap = B200C.compressBound(outComp, totalIn, cp.chunkLength()), indexCap = totalIndex + (1 << 20), chunkCap = totalIn / cp.chunkLength() + 16;
                long summaryCap = totalIndex / 16 + (1 << 20);
                int nout = 1;
                if (maxSSTableBytes > 0 && maxSSTableBytes < dataCap)
                {
                    // the limit counts ON-DISK (compressed) bytes: the files are about the compressed input over the limit; a file holds the limit plus
                    // the partition that crosses it (a larger one comes back as ETOOSMALL with its size, and the retry below grows the slots)
                    long files = Math.max(1, totalCompressed / Math.max(1, maxSSTableBytes) + 2);
                    nout = (int) Math.min(4096, files);
                    dataCap = Math.min(dataCap, maxSSTableBytes + (16 << 20)); indexCap = Math.min(indexCap, indexCap / files * 2 + (1 << 20));
                    chunkCap = Math.min(chunkCap, 4 * dataCap / cp.chunkLength() + 16); summaryCap = Math.min(summaryCap, indexCap / 16 + (1 << 20));
                }
                Outputs outs = null;
                ByteBuffer res = B200C.struct(SIZEOF_RESULT);
                int rc;
                for (int attempt = 0; ; attempt++)
                {
                    if (outs != null) outs.close();
                    outs = new Outputs(nout, dataCap, indexCap, chunkCap, summaryCap, 8 + 8 * m.getLong(M_BLOOM_WORDS));
                    res.putInt(R_NOUTPUTS_CAP, nout).putLong(R_OUTPUTS, B200C.address(outs.slots));

                    // ---- the call; progress and stop requests travel through poll / cancel from the CompactionInfo.Holder ------------------------------
                    GpuCompactionInfo info = new GpuCompactionInfo(this, ctx, totalIn);
                    CompactionManager.instance.active.beginCompaction(info);
                    try
                    {
                        if (!cfs.getCompactionStrategyManager().isActive())
                            throw new CompactionInterruptedException(info.getCompactionInfo());
                        rc = B200C.compact(ctx, B200C.address(m), B200C.address(res), 0);
                    }
                    finally
                    {
                        CompactionManager.instance.active.finishCompaction(info);
                        outs.unregister();
                    }
                    if (rc != B200C.ETOOSMALL || attempt == 2) break;
                    nout = Math.max(nout, res.getInt(R_NOUTPUTS));
                    dataCap = Math.max(dataCap, res.getLong(R_REQUIRED_DATA_CAP)); indexCap = Math.max(indexCap, res.getLong(R_REQUIRED_INDEX_CAP));
                    chunkCap = Math.max(chunkCap, res.getLong(R_REQUIRED_CHUNK_CAP));
                    for (int k = 0; k < Math.min(nout, outs.n); k++) summaryCap = Math.max(summaryCap, outs.slot(k).getLong(O_SUMMARY_LEN));
                }
                switch (rc)
                {
                    case B200C.OK: break;
                    case B200C.ECORRUPT:
                    {
                        outs.close();
                        SSTableReader bad = inputs.get(res.getInt(R_CORRUPTION)).reader;         // corruption.input
                        bad.markSuspect();
                        throw new CorruptSSTableException(new IOException(B200C.lastError(ctx)), bad.getFilename());
                    }
                    case B200C.ECANCELLED: outs.close(); throw new CompactionInterruptedException(new GpuCompactionInfo(this, ctx, totalIn).getCompactionInfo());
                    case B200C.EUNSUPPORTED: outs.close(); super.runMayThrow(); return;          // an input used a feature outside the envelope: the stock task does it
                    default: outs.close(); throw new RuntimeException("b200c_compact failed (" + rc + "): " + B200C.lastError(ctx));
                }

                // ---- outputs -> component files of a new descriptor each, tracked by the transaction exactly like a writer's would be -----------------
                long written = 0;
                for (int k = 0; k < res.getInt(R_NOUTPUTS); k++)
                {
                    ByteBuffer out = outs.slot(k);
                    if (out.getLong(O_PARTITIONS) == 0) continue;
                    Descriptor d = cfs.newSSTableDescriptor(getDirectories().getWriteableLocationAsFile(cfs, null, out.getLong(O_DATA_LEN)));
                    Set<Component> components = new java.util.HashSet<>(d.getFormat().allComponents());
                    transaction.trackNew(new org.apache.cassandra.io.sstable.SSTable.Builder<>(d).setComponents(components).setTableMetadataRef(cfs.metadata).build(cfs));
                    write(d.fileFor(Components.DATA), outs.data[k], out.getLong(O_DATA_LEN));
                    write(d.fileFor(BigFormat.Components.PRIMARY_INDEX), outs.index[k], out.getLong(O_INDEX_LEN));
                    write(d.fileFor(Components.FILTER), outs.filter[k], out.getLong(O_FILTER_LEN));
                    write(d.fileFor(BigFormat.Components.SUMMARY), outs.summary[k], out.getLong(O_SUMMARY_LEN));
                    writeCompressionInfo(d, cp, out, outs.offsets[k]);
                    try (FileOutputStreamPlus o = new FileOutputStreamPlus(d.fileFor(Components.DIGEST)))
                    {
                        o.write(Long.toString(out.getInt(O_DIGEST) & 0xFFFFFFFFL).getBytes(java.nio.charset.StandardCharsets.UTF_8));
                    }
                    writeStatistics(d, table, header, outs.stats[k], outs.keys[k], out, (double) out.getLong(O_DATA_LEN) / Math.max(1, out.getLong(O_DATA_LENGTH)), actuallyCompact, fp);
                    d.getFormat().getWriterFactory();                                            // TOC.txt
                    org.apache.cassandra.io.sstable.format.TOCComponent.appendTOC(d, components);
                    SSTableReader reader = SSTableReader.open(cfs, d, components, cfs.metadata);
                    transaction.update(reader, false);
                    written += out.getLong(O_DATA_LEN);
                }
                outs.close();
                transaction.obsoleteOriginals();
                transaction.prepareToCommit();
                transaction.commit();

                long[] merged = new long[inputs.size()];
                for (int i = 0; i < merged.length; i++) merged[i] = res.getLong(R_MERGED_ROW_COUNTS + 8 * i);
                updateCompactionHistory(transaction.opId(), cfs.getKeyspaceName(), cfs.getTableName(), merged, totalIn, written,
                                        com.google.common.collect.ImmutableMap.of(COMPACTION_TYPE_PROPERTY, compactionType.type));
                cfs.metric.compactionBytesWritten.inc(written);
            }
            finally
            {
                for (Input s : inputs) s.close();
            }
        }
    }

    /** MaxSSTableSizeWriter.getTotalWriteSize: the expected output size, scaled by the estimated key count after compaction */
    private long expectedWriteSize(Collection<SSTableReader> sstables, long estimatedTotalKeys)
    {
        long before = 0;
        for (SSTableReader r : sstables) before += r.estimatedKeys();
        return Math.round((double) estimatedTotalKeys / Math.max(1, before) * cfs.getExpectedCompactedFileSize(sstables, compactionType));
    }

    /** caller-provided buffers of n output slots (b200c_output), pinned while the call runs */
    private static final class Outputs implements AutoCloseable
    {
        final int n;
        final ByteBuffer slots;
        final ByteBuffer[] data, index, offsets, keys, filter, summary, stats;

        Outputs(int n, long dataCap, long indexCap, long chunkCap, long summaryCap, long filterCap)
        {
            this.n = n;
            slots = B200C.struct(SIZEOF_OUTPUT * n);
            data = new ByteBuffer[n]; index = new ByteBuffer[n]; offsets = new ByteBuffer[n]; keys = new ByteBuffer[n];
            filter = new ByteBuffer[n]; summary = new ByteBuffer[n]; stats = new ByteBuffer[n];
            for (int k = 0; k < n; k++)
            {
                data[k] = ByteBuffer.allocateDirect(Math.toIntExact(Math.min(dataCap, Integer.MAX_VALUE - 8)));      // > 2 GiB outputs: use several buffers / Unsafe
                index[k] = ByteBuffer.allocateDirect(Math.toIntExact(indexCap));
                offsets[k] = B200C.struct(Math.toIntExact(8 * chunkCap));
                keys[k] = ByteBuffer.allocateDirect(2 * 65535);
                filter[k] = B200C.struct(Math.toIntExact(filterCap));
                summary[k] = ByteBuffer.allocateDirect(Math.toIntExact(summaryCap));
                stats[k] = B200C.struct(SIZEOF_STATS);
                ByteBuffer o = slot(k);
                o.putLong(O_DATA, B200C.address(data[k])).putLong(O_DATA_CAP, data[k].capacity());
                o.putLong(O_INDEX, B200C.address(index[k])).putLong(O_INDEX_CAP, index[k].capacity());
                o.putLong(O_CHUNK_OFFSETS, B200C.address(offsets[k])).putLong(O_CHUNK_CAP, offsets[k].capacity() / 8);
                o.putLong(O_KEY_BUF, B200C.address(keys[k])).putLong(O_KEY_CAP, keys[k].capacity());
                o.putLong(O_FILTER, B200C.address(filter[k])).putLong(O_FILTER_CAP, filter[k].capacity());
                o.putLong(O_SUMMARY, B200C.address(summary[k])).putLong(O_SUMMARY_CAP, summary[k].capacity());
                o.putLong(O_STATS, B200C.address(stats[k]));
                B200C.hostRegister(B200C.address(data[k]), data[k].capacity());
            }
        }

        /** view of slot k (native order, offsets from B200C.Layout) */
        ByteBuffer slot(int k)
        {
            ByteBuffer b = slots.duplicate().order(slots.order()); b.position(k * SIZEOF_OUTPUT).limit((k + 1) * SIZEOF_OUTPUT);
            return b.slice().order(slots.order());
        }

        private boolean registered = true;
        void unregister()
        {
            if (!registered) return;
            for (ByteBuffer b : data) B200C.hostUnregister(B200C.address(b));
            registered = false;
        }

        public void close() { unregister(); }
    }

    private static void write(File f, ByteBuffer b, long n) throws IOException
    {
        try (FileChannel ch = FileChannel.open(f.toPath(), StandardOpenOption.CREATE, StandardOpenOption.WRITE, StandardOpenOption.TRUNCATE_EXISTING))
        {
            ByteBuffer v = b.duplicate(); v.position(0).limit(Math.toIntExact(n));
            while (v.hasRemaining()) ch.write(v);
            ch.force(true);
        }
    }

    /** CompressionMetadata.Writer layout (S/io/compress/CompressionMetadata.java:375-398,423-431), offsets big-endian */
    private static void writeCompressionInfo(Descriptor d, CompressionParams cp, ByteBuffer out, ByteBuffer offsets) throws IOException
    {
        try (DataOutputStreamPlus o = new FileOutputStreamPlus(d.fileFor(Components.COMPRESSION_INFO)))
        {
            o.writeUTF(cp.getSstableCompressor().getClass().getSimpleName().replace("Gpu", ""));   // stock nodes must find LZ4Compressor / SnappyCompressor
            o.writeInt(cp.getOtherOptions().size());
            for (Map.Entry<String, String> e : cp.getOtherOptions().entrySet()) { o.writeUTF(e.getKey()); o.writeUTF(e.getValue()); }
            o.writeInt(cp.chunkLength()); o.writeInt(cp.maxCompressedLength()); o.writeLong(out.getLong(O_DATA_LENGTH));
            int n = Math.toIntExact(out.getLong(O_NCHUNKS));
            o.writeInt(n);
            for (int i = 0; i < n; i++) o.writeLong(offsets.getLong(8 * i));
        }
    }

    /** Statistics.db from the side band the kernels gathered (b200c_sstable_stats = MetadataCollector's reductions) */
    private void writeStatistics(Descriptor d, TableMetadata table, SerializationHeader header, ByteBuffer s, ByteBuffer keys, ByteBuffer out, double ratio,
                                 Collection<SSTableReader> inputs, double fpChance) throws IOException
    {
        long[] psizeOffsets = EstimatedHistogram.newOffsets(155, false), cellOffsets = EstimatedHistogram.newOffsets(118, false);
        long[] psize = new long[156], cells = new long[119];
        for (int i = 0; i < 156; i++) psize[i] = s.getLong(S_PARTITION_SIZE_HIST + 8 * i);
        for (int i = 0; i < 119; i++) cells[i] = s.getLong(S_CELLS_HIST + 8 * i);
        StreamingTombstoneHistogramBuilder th = new StreamingTombstoneHistogramBuilder(org.apache.cassandra.io.sstable.SSTable.TOMBSTONE_HISTOGRAM_BIN_SIZE,
                                                                                       org.apache.cassandra.io.sstable.SSTable.TOMBSTONE_HISTOGRAM_SPOOL_SIZE, 1);
        for (int i = 0; i < s.getInt(S_NTDROP); i++)                                   // points are already rounded to 60 s; replay them with their counts
            th.update(s.getLong(S_TDROP_POINT + 8 * i), (int) Math.min(Integer.MAX_VALUE, s.getLong(S_TDROP_COUNT + 8 * i)));
        IntervalSet.Builder<CommitLogPosition> intervals = new IntervalSet.Builder<>();
        for (SSTableReader r : inputs) intervals.addAll(r.getSSTableMetadata().commitLogIntervals);
        byte[] first = new byte[out.getInt(O_FIRST_KEY_LEN)], last = new byte[out.getInt(O_LAST_KEY_LEN)];
        ByteBuffer k = keys.duplicate(); k.position(0); k.get(first); k.get(last);
        ICardinality cardinality = new HyperLogLogPlus(13, 25);                        // CompactionMetadata: the sketch is rebuilt from Index.db keys by the caller if it needs
                                                                                       // more than the dense registers in b200c_sstable_stats.hll_registers (see INTEGRATION.md)
        Map<MetadataType, MetadataComponent> components = new EnumMap<>(MetadataType.class);
        components.put(MetadataType.VALIDATION, new ValidationMetadata(table.partitioner.getClass().getCanonicalName(), fpChance));
        components.put(MetadataType.STATS, new StatsMetadata(new EstimatedHistogram(psizeOffsets, psize), new EstimatedHistogram(cellOffsets, cells), intervals.build(),
                                                             s.getLong(S_MIN_TIMESTAMP), s.getLong(S_MAX_TIMESTAMP), s.getLong(S_MIN_LDT), s.getLong(S_MAX_LDT),
                                                             s.getInt(S_MIN_TTL), s.getInt(S_MAX_TTL), ratio, th.build(), level, table.comparator.subtypes(), Slice.ALL,
                                                             s.getInt(S_HAS_LEGACY_COUNTER_SHARDS) != 0, ActiveRepairService.UNREPAIRED_SSTABLE, s.getLong(S_TOTAL_COLUMNS_SET), s.getLong(S_TOTAL_ROWS), Double.NaN,
                                                             org.apache.cassandra.service.StorageService.instance.getLocalHostUUID(), null, false,
                                                             s.getInt(S_HAS_PARTITION_DELETIONS) != 0, ByteBuffer.wrap(first), ByteBuffer.wrap(last)));
        components.put(MetadataType.COMPACTION, new CompactionMetadata(cardinality));
        components.put(MetadataType.HEADER, header.toComponent());
        try (FileOutputStreamPlus o = new FileOutputStreamPlus(d.fileFor(Components.STATS)))
        {
            d.getMetadataSerializer().serialize(components, o, d.version);
        }
    }

    /** BloomCalculations.computeBloomSpec for (keys, fpChance): {K, bucketsPerElement} (S/utils/BloomCalculations.java) */
    static final class BloomSpec
    {
        static int[] of(long keys, double fp)
        {
            if (fp >= 1.0) return new int[]{ 0, 0 };
            int maxBuckets = org.apache.cassandra.utils.BloomCalculations.maxBucketsPerElement(keys);
            org.apache.cassandra.utils.BloomCalculations.BloomSpecification spec = org.apache.cassandra.utils.BloomCalculations.computeBloomSpec(maxBuckets, fp);
            return new int[]{ spec.K, spec.bucketsPerElement };
        }
    }

    /** CompactionInfo.Holder of the native call: progress from b200c_poll, stop() -> b200c_cancel (CompactionIterator.java:167-176,709-742) */
    static final class GpuCompactionInfo extends CompactionInfo.Holder
    {
        private final GpuCompactionTask task; private final long ctx, total;
        private final ByteBuffer progress = B200C.struct(SIZEOF_PROGRESS);

        GpuCompactionInfo(GpuCompactionTask task, long ctx, long total) { this.task = task; this.ctx = ctx; this.total = total; }

        @Override
        public CompactionInfo getCompactionInfo()
        {
            B200C.poll(ctx, B200C.address(progress));
            return new CompactionInfo(task.cfs.metadata(), task.compactionType, progress.getLong(0), total, task.transaction.opId(), task.transaction.originals());
        }

        @Override
        public boolean isGlobal() { return false; }

        @Override
        public void stop()
        {
            super.stop();
            B200C.cancel(ctx);
        }
    }
}
