package edu.scripps.yates.dbindex.gpu;

import java.io.IOException;
import java.util.ArrayList;
import java.util.Collection;
import java.util.LinkedHashMap;
import java.util.LinkedHashSet;
import java.util.List;
import java.util.Map;
import java.util.Set;

import edu.scripps.yates.dbindex.DBIndexer;
import edu.scripps.yates.utilities.fasta.dbindex.DBIndexSearchParams;
import edu.scripps.yates.utilities.fasta.dbindex.DBIndexStoreException;
import edu.scripps.yates.utilities.fasta.dbindex.IndexedProtein;
import edu.scripps.yates.utilities.fasta.dbindex.IndexedSequence;
import edu.scripps.yates.utilities.fasta.dbindex.MassRange;

/**
 * DBIndexer with the digestion moved to the GPU: run() still streams the FASTA and fills the
 * ProteinCache (DBIndexer.java:600-616), but cutSeq only hands the protein to the store; the windows,
 * masses and gates of DBIndexer.java:256-394 are computed by digest_count/emit_kernel when
 * stopAddSeq() calls dbi_build (in SEARCH_UNINDEXED mode: when a query calls dbi_search_unindexed). Uses the
 * reference's own plugin constructor (DBIndexer.java:143).
 * NOT COMPILED HERE (no JDK, see DbiNative).
 */
public class GpuDBIndexer extends DBIndexer {
	public GpuDBIndexer(DBIndexSearchParams sparam, IndexerMode mode) {
		super(sparam, mode, new GpuDBIndexStore(sparam, mode == IndexerMode.SEARCH_UNINDEXED));
	}

	@Override
	protected void cutSeq(final String protAccession, String protSeq) throws IOException {
		try {
			indexStore.addProteinDef(++protNum, protAccession, protSeq); // DBIndexer.java:251
		} catch (final DBIndexStoreException e) {
			throw new IOException(e);
		}
	}

	/**
	 * getSequencesUsingPPMTolerance (DBIndexer.java:787-844) as a batch of one: the window and the exact-mass
	 * probe walk run on the GPU in one call (on every GPU of a sharded index).
	 */
	@Override
	public List<IndexedSequence> getSequencesUsingPPMTolerance(double precursorMass, double massToleranceInPPM)
			throws DBIndexStoreException {
		return getSequencesUsingPPMTolerance(new double[] { precursorMass }, massToleranceInPPM).get(0);
	}

	/** getSequencesUsingPPMTolerance for every mass, one device call (dbi_query_spectra, DBI_TOL_PPM). */
	public List<List<IndexedSequence>> getSequencesUsingPPMTolerance(double[] masses, double massToleranceInPPM)
			throws DBIndexStoreException {
		final GpuDBIndexStore store = (GpuDBIndexStore) indexStore;
		final double[] ppm = new double[masses.length];
		java.util.Arrays.fill(ppm, massToleranceInPPM);
		return store.querySpectra(masses, ppm, null, DbiNative.DBI_TOL_PPM);
	}

	/** getSequences(List<MassRange>) for every spectrum, one device call (dbi_query_spectra, DBI_TOL_DA). */
	public List<List<IndexedSequence>> getSequencesForSpectra(List<List<MassRange>> spectra) throws DBIndexStoreException {
		final GpuDBIndexStore store = (GpuDBIndexStore) indexStore;
		final long[] rangeOff = new long[spectra.size() + 1];
		for (int s = 0; s < spectra.size(); ++s)
			rangeOff[s + 1] = rangeOff[s] + spectra.get(s).size();
		final double[] mass = new double[(int) rangeOff[spectra.size()]], tol = new double[mass.length];
		int r = 0;
		for (final List<MassRange> sp : spectra)
			for (final MassRange m : sp) {
				mass[r] = m.getPrecMass();
				tol[r++] = m.getTolerance();
			}
		return store.querySpectra(mass, tol, rangeOff, DbiNative.DBI_TOL_DA);
	}

	/** getProteins(String) (DBIndexer.java:925-947) through the batched device lookup (dbi_lookup_peptides). */
	@Override
	public Set<IndexedProtein> getProteins(String sequence) throws DBIndexStoreException {
		return getProteins(List.of(sequence)).get(sequence);
	}

	/** getProteins(String) for every distinct string of the collection, in one device call per GPU. */
	public Map<String, Set<IndexedProtein>> getProteins(Collection<String> sequences) throws DBIndexStoreException {
		final List<String> distinct = new ArrayList<>(new LinkedHashSet<>(sequences));
		final List<Set<IndexedProtein>> sets = ((GpuDBIndexStore) indexStore).lookupPeptides(distinct);
		final Map<String, Set<IndexedProtein>> ret = new LinkedHashMap<>();
		for (int i = 0; i < distinct.size(); ++i)
			ret.put(distinct.get(i), sets.get(i));
		return ret;
	}
}
