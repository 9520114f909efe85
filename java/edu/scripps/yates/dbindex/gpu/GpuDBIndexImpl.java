package edu.scripps.yates.dbindex.gpu;

import java.io.File;
import java.util.Collection;
import java.util.List;
import java.util.Map;
import java.util.Set;

import edu.scripps.yates.dbindex.DBIndexImpl;
import edu.scripps.yates.dbindex.DBIndexer.IndexerMode;
import edu.scripps.yates.dbindex.DBIndexerException;
import edu.scripps.yates.utilities.fasta.dbindex.DBIndexSearchParams;
import edu.scripps.yates.utilities.fasta.dbindex.DBIndexStoreException;
import edu.scripps.yates.utilities.fasta.dbindex.IndexedProtein;
import edu.scripps.yates.utilities.fasta.dbindex.IndexedSequence;
import edu.scripps.yates.utilities.fasta.dbindex.MassRange;
import gnu.trove.map.hash.THashMap;

/**
 * The class a search engine holds: DBIndexInterface (DBIndexImpl.java:27) with the GPU index behind it.
 * It extends DBIndexImpl so that every factory, registry and memoisation of the reference stays as it
 * is (getDefaultDBIndexParams* DBIndexImpl.java:243-491, getProteins(String) cache :222-237,
 * getIndexedProteinById / getProteinSequenceById :501-513); the only difference is which indexer is
 * created: GpuDBIndexer with a GpuDBIndexStore instead of DBIndexer with DBIndexStoreSQLiteMult
 * (DBIndexImpl.java:117-145). NOT COMPILED HERE (no JDK, see DbiNative).
 */
public class GpuDBIndexImpl extends DBIndexImpl {
	private static final Map<String, GpuDBIndexImpl> gpuIndexByParamKey = new THashMap<>();

	/** DBIndexImpl.getByParam (DBIndexImpl.java:44-49) for GPU indexes: one per parameter key. */
	public static synchronized GpuDBIndexImpl getByParam(DBIndexSearchParams sParam) {
		final String key = sParam.getFullIndexFileName(null, null, false, null, false, null);
		final GpuDBIndexImpl hit = gpuIndexByParamKey.get(key);
		return hit != null ? hit : new GpuDBIndexImpl(sParam);
	}

	public GpuDBIndexImpl(File fastaFile) {
		this(getDefaultDBIndexParams(fastaFile));
	}

	/**
	 * Same sequence as DBIndexImpl(DBIndexSearchParams) (DBIndexImpl.java:117-145): indexer, init(), run().
	 * useIndex = false (default_use_index, dbindex.properties) selects SEARCH_UNINDEXED (DBIndexer.java:58-61): the
	 * proteins are uploaded and every query digests them again on the GPU (dbi_search_unindexed).
	 */
	public GpuDBIndexImpl(DBIndexSearchParams sParam) {
		super(); // the no-arg constructor builds nothing (DBIndexImpl.java:51-53)
		try {
			indexer = new GpuDBIndexer(sParam, sParam.isUseIndex() ? IndexerMode.INDEX : IndexerMode.SEARCH_UNINDEXED);
			indexer.init();
			indexer.run(); // FASTA streaming as in the reference; cutSeq only hands proteins to the GPU store
			synchronized (GpuDBIndexImpl.class) {
				gpuIndexByParamKey.put(sParam.getFullIndexFileName(null, null, false, null, false, null), this);
			}
		} catch (final DBIndexerException e) {
			throw new RuntimeException(e);
		}
	}

	// The six DBIndexInterface methods are inherited unchanged (DBIndexImpl.java:180-237, 501-513): they call
	// indexer.getSequencesUsingDaltonTolerance / getSequences / getProteins, which reach GpuDBIndexStore.
	// They are restated here so that the class reads as what it is.
	@Override
	public List<IndexedSequence> getSequences(double precursorMass, double massTolerance) throws DBIndexStoreException {
		return super.getSequences(precursorMass, massTolerance);
	}

	@Override
	public List<IndexedSequence> getSequences(List<MassRange> massRanges) throws DBIndexStoreException {
		return super.getSequences(massRanges);
	}

	@Override
	public List<IndexedProtein> getProteins(IndexedSequence seq) throws DBIndexStoreException {
		return super.getProteins(seq);
	}

	/** Memoised as in the reference; a miss reaches GpuDBIndexer.getProteins(String), one dbi_lookup_peptides. */
	@Override
	public Set<IndexedProtein> getProteins(String seq) throws DBIndexStoreException {
		return super.getProteins(seq);
	}

	/**
	 * getSequences(List<MassRange>) for every spectrum of a run in one device call. Not an overload of
	 * getSequences(List): both would erase to the same signature.
	 */
	public List<List<IndexedSequence>> getSequencesForSpectra(List<List<MassRange>> spectra) throws DBIndexStoreException {
		return ((GpuDBIndexer) indexer).getSequencesForSpectra(spectra);
	}

	/** getProteins(String) for a whole collection (e.g. every distinct identified peptide) in one device call. */
	public Map<String, Set<IndexedProtein>> getProteins(Collection<String> seqs) throws DBIndexStoreException {
		return ((GpuDBIndexer) indexer).getProteins(seqs);
	}
}
