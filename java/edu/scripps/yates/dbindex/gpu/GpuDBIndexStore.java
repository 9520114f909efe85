package edu.scripps.yates.dbindex.gpu;

import java.lang.foreign.Arena;
import java.lang.foreign.MemorySegment;
import java.util.ArrayList;
import java.util.Iterator;
import java.util.List;

import edu.scripps.yates.dbindex.DBIndexStore;
import edu.scripps.yates.dbindex.Interval;
import edu.scripps.yates.dbindex.MergeIntervals;
import edu.scripps.yates.dbindex.ProteinCache;
import edu.scripps.yates.dbindex.Util;
import edu.scripps.yates.utilities.fasta.dbindex.DBIndexSearchParams;
import edu.scripps.yates.utilities.fasta.dbindex.DBIndexStoreException;
import edu.scripps.yates.utilities.fasta.dbindex.IndexedProtein;
import edu.scripps.yates.utilities.fasta.dbindex.IndexedSequence;
import edu.scripps.yates.utilities.fasta.dbindex.MassRange;
import edu.scripps.yates.utilities.fasta.dbindex.ResidueInfo;
import edu.scripps.yates.utilities.masses.AssignMass;

import static java.lang.foreign.ValueLayout.ADDRESS;
import static java.lang.foreign.ValueLayout.JAVA_BYTE;
import static java.lang.foreign.ValueLayout.JAVA_DOUBLE;
import static java.lang.foreign.ValueLayout.JAVA_INT;
import static java.lang.foreign.ValueLayout.JAVA_LONG;
import static java.lang.foreign.ValueLayout.JAVA_SHORT;

/**
 * The GPU store behind the reference's own plugin seam: DBIndexStore (DBIndexStore.java:19-194), handed
 * to the indexer through its 3-argument constructor (DBIndexer.java:143). Digestion, mass-ordering,
 * merging and range search run in libdbindex_gpu.so; this class only marshals and rebuilds the
 * IndexedSequence objects exactly as DBIndexStoreSQLiteByteIndexMerge.parseAddPeptideInfo does
 * (DBIndexStoreSQLiteByteIndexMerge.java:452-462). NOT COMPILED HERE (no JDK, see DbiNative).
 */
public class GpuDBIndexStore implements DBIndexStore {
	private static final int MAX_MASS = 8000; // Constants.MAX_PRECURSOR_MASS, DBIndexStoreSQLiteMult buckets
	private final DBIndexSearchParams sparam;
	private final Arena arena = Arena.ofShared();
	private MemorySegment handle = MemorySegment.NULL; // handles[0]
	// -Ddbindex.gpu.devices=N: ONE index sharded over N GPUs of this box (the reference's mass buckets,
	// DBIndexStoreSQLiteMult.java:55-56,215-217, as GPUs): handle r lives on device r and is given shard r of the proteins
	private final int nDevices = Math.max(1, Integer.getInteger("dbindex.gpu.devices", 1));
	private MemorySegment[] handles = new MemorySegment[0];
	private double[] splitMass = new double[0]; // masses at which the slices of the sharded index are cut
	private boolean inited = false, built = false;
	// SEARCH_UNINDEXED (DBIndexer.java:58-61, MassRangeFilteringIndex.java:90-108): no index, every query digests
	// the proteins again for its ranges (dbi_search_unindexed; with -Ddbindex.gpu.devices=N every GPU its shard,
	// dbi_mg_search_unindexed_local), at most maxCandidates candidate records per call (and GPU)
	private final boolean unindexed;
	private final long maxCandidates = Long.getLong("dbindex.gpu.maxCandidates", 1L << 25);
	private ProteinCache proteinCache;
	private String indexFile; // null = in-memory index only
	// proteins gathered by addProteinDef until stopAddSeq() (subsystem 1: packed residue buffer)
	private final java.io.ByteArrayOutputStream residues = new java.io.ByteArrayOutputStream();
	private final List<Long> offsets = new ArrayList<>(List.of(0L));
	// Search-engine threads (DBIndexer.java:468-469) query the built index through views (dbi_view_open): one per
	// thread and GPU, opened on the thread's first query, each with its own stream and pending results, so their
	// calls run in parallel.  The paths that need the owner handles (the unindexed searches, the sharded spectrum
	// batches) take ownerLock around every call pair, so no thread reads another one's pending result.
	private final ThreadLocal<MemorySegment[]> views = new ThreadLocal<>();
	private final java.util.concurrent.ConcurrentLinkedQueue<MemorySegment> openViews = new java.util.concurrent.ConcurrentLinkedQueue<>();
	private final Object ownerLock = new Object();

	public GpuDBIndexStore(DBIndexSearchParams sparam, boolean unindexed) {
		this.sparam = sparam;
		this.unindexed = unindexed;
	}

	private static void check(int rc) throws DBIndexStoreException {
		if (rc != DbiNative.DBI_OK)
			throw new DBIndexStoreException(DbiNative.lastError());
	}

	/** this thread's views of the built index, one per GPU (handles[d] -> views()[d]) */
	private MemorySegment[] views() throws Throwable {
		MemorySegment[] v = views.get();
		if (v == null) {
			v = new MemorySegment[handles.length];
			try (Arena a = Arena.ofConfined()) {
				final MemorySegment out = a.allocate(ADDRESS);
				for (int d = 0; d < handles.length; ++d) {
					final int rc = (int) DbiNative.dbi_view_open.invoke(handles[d], out);
					if (rc != DbiNative.DBI_OK) {
						final DBIndexStoreException e = new DBIndexStoreException(DbiNative.lastError());
						for (int k = 0; k < d; ++k) {
							openViews.remove(v[k]);
							DbiNative.dbi_destroy.invoke(v[k]);
						}
						throw e;
					}
					v[d] = out.get(ADDRESS, 0);
					openViews.add(v[d]);
				}
			}
			views.set(v);
		}
		return v;
	}

	/** dbi_params from the live AssignMass / Enzyme / search parameters (SURVEY.md 5.1). */
	private MemorySegment params() throws Throwable {
		final MemorySegment p = arena.allocate(DbiNative.PARAMS);
		DbiNative.dbi_default_params.invoke(p, sparam.isUseMonoParent() ? 1 : 0);
		final long massOff = DbiNative.PARAMS.byteOffset(java.lang.foreign.MemoryLayout.PathElement.groupElement("residue_mass"));
		for (int c = 0; c < 256; ++c) // the real table, static mods already applied by SearchParamReader
			p.set(JAVA_DOUBLE, massOff + 8L * c, AssignMass.getMass((char) c));
		set(p, "h2o_proton", AssignMass.H2O_PROTON);
		set(p, "nterm", AssignMass.getnTerm());
		set(p, "cterm", AssignMass.getcTerm());
		setInt(p, "add_h2o_proton", sparam.isH2OPlusProtonAdded() ? 1 : 0);
		final long enzOff = DbiNative.PARAMS.byteOffset(java.lang.foreign.MemoryLayout.PathElement.groupElement("is_enzyme"));
		final long nocOff = DbiNative.PARAMS.byteOffset(java.lang.foreign.MemoryLayout.PathElement.groupElement("is_nocut"));
		for (int c = 0; c < 256; ++c) {
			p.set(JAVA_BYTE, enzOff + c, (byte) (sparam.getEnzyme().isEnzyme((char) c) ? 1 : 0));
			p.set(JAVA_BYTE, nocOff + c, (byte) 0);
		}
		final String nocut = sparam.getEnzymeNocutResidues();
		if (nocut != null)
			for (final char c : nocut.toCharArray())
				p.set(JAVA_BYTE, nocOff + c, (byte) 1);
		setInt(p, "max_missed", sparam.getMaxMissedCleavages());
		setInt(p, "semi", sparam.isSemiCleavage() ? 1 : 0);
		set(p, "min_mass", sparam.getMinPrecursorMass());
		set(p, "max_mass", sparam.getMaxPrecursorMass());
		setInt(p, "mass_group_factor", sparam.getMassGroupFactor());
		// mandatoryInternalAAs (DBIndexer.java:248,334-344): null = no constraint, an empty array is legal
		final char[] mandatory = sparam.getMandatoryInternalAAs();
		if (mandatory != null) {
			setInt(p, "has_mandatory", 1);
			final long manOff = DbiNative.PARAMS.byteOffset(java.lang.foreign.MemoryLayout.PathElement.groupElement("is_mandatory"));
			for (final char c : mandatory)
				p.set(JAVA_BYTE, manOff + c, (byte) 1);
		}
		// PeptideFilterByMaxOccurrencies prints itself as <aa><max> (util/PeptideFilterByMaxOccurrencies.java:37-40)
		if (sparam.getPeptideFilter() != null) {
			final String pf = sparam.getPeptideFilter().toString();
			setInt(p, "filter_aa", pf.charAt(0));
			setInt(p, "filter_max", Integer.parseInt(pf.substring(1)));
		}
		// differential mods: the residue -> shift table SearchParamReader fills (io/SearchParamReader.java:631-667,
		// model/DiffModification.java:11-54) and max_num_differential_AA_per_mod (:322)
		final boolean[] isDiff = edu.scripps.yates.dbindex.model.DiffModification.getIsDiffMod();
		final double[] diff = edu.scripps.yates.dbindex.model.DiffModification.getDiffMod();
		int nMods = 0;
		try (Arena a = Arena.ofConfined()) {
			for (int c = 0; c < isDiff.length && c < 256; ++c)
				if (isDiff[c] && diff[c] != 0) {
					final MemorySegment res = a.allocateFrom(String.valueOf((char) c));
					check((int) DbiNative.dbi_params_add_diff_mod.invoke(p, res, diff[c])); // DBI_ERANGE past 16 entries
					++nMods;
				}
		}
		setInt(p, "max_mods_per_peptide", nMods > 0 ? edu.scripps.yates.dbindex.SearchParams.getInstance().getMaxNumDiffMod() : 0);
		return p;
	}

	private static void set(MemorySegment p, String f, double v) {
		p.set(JAVA_DOUBLE, DbiNative.PARAMS.byteOffset(java.lang.foreign.MemoryLayout.PathElement.groupElement(f)), v);
	}

	private static void setInt(MemorySegment p, String f, int v) {
		p.set(JAVA_INT, DbiNative.PARAMS.byteOffset(java.lang.foreign.MemoryLayout.PathElement.groupElement(f)), v);
	}

	@Override
	public void init(String databaseID) throws DBIndexStoreException {
		if (inited)
			throw new DBIndexStoreException("Already intialized"); // DBIndexStoreSQLiteMult.java:97-99
		try {
			handles = new MemorySegment[nDevices];
			for (int d = 0; d < nDevices; ++d) {
				final MemorySegment out = arena.allocate(ADDRESS);
				final MemorySegment p = params();
				setInt(p, "device", d);
				check((int) DbiNative.dbi_create.invoke(p, out));
				handles[d] = out.get(ADDRESS, 0);
			}
			handle = handles[0];
			// on-disk index (in_memory_index = false): <fasta>_<md5(params)> like the reference (IndexUtil.java:270-324);
			// if the file is there the index is loaded and DBIndexer.run() skips indexing (DBIndexer.java:522-531)
			if (!sparam.isInMemoryIndex() && nDevices == 1 && !unindexed) { // a sharded index is rebuilt (dbi_save holds one GPU's index)
				indexFile = sparam.getFullIndexFileName(null, null, false, null, false, null) + ".gpuidx";
				if (new java.io.File(indexFile).exists()) {
					check((int) DbiNative.dbi_load.invoke(handle, arena.allocateFrom(indexFile)));
					built = true;
				}
			}
		} catch (final DBIndexStoreException e) {
			throw e;
		} catch (final Throwable t) {
			throw new DBIndexStoreException("dbi_create failed", t);
		}
		inited = true;
	}

	private void requireInit() throws DBIndexStoreException {
		if (!inited)
			throw new DBIndexStoreException("Indexer is not initialized"); // Mult:153,273,316
	}

	@Override
	public boolean indexExists() {
		return built; // the index lives in HBM: it exists once stopAddSeq() has run
	}

	@Override
	public void startAddSeq() throws DBIndexStoreException {
		requireInit();
	}

	/** cutSeq is replaced by the digestion kernels: the indexer hands whole proteins over here. */
	@Override
	public long addProteinDef(long num, String accession, String protSequence) throws DBIndexStoreException {
		requireInit();
		final byte[] b = protSequence.getBytes(java.nio.charset.StandardCharsets.ISO_8859_1);
		residues.write(b, 0, b.length);
		offsets.add(offsets.get(offsets.size() - 1) + b.length);
		return num; // Mult:446-450
	}

	@Override
	public FilterResult filterSequence(double precMass, String sequence) {
		return FilterResult.INCLUDE; // gates are applied on the device (DBIndexer.java:327-331)
	}

	@Override
	public void addSequence(double precMass, int sequenceOffset, int sequenceLen, String sequence, String resLeft,
			String resRight, long proteinId) {
		// no-op: GpuDBIndexer never calls it, peptides are emitted by digest_emit_kernel
	}

	/** stopAddSeq = commit + mergePeptides + createIndex of the SQLite stack -> dbi_build. */
	@Override
	public void stopAddSeq() throws DBIndexStoreException {
		requireInit();
		try (Arena a = Arena.ofConfined()) {
			final byte[] res = residues.toByteArray();
			final MemorySegment r = a.allocate(Math.max(1, res.length));
			MemorySegment.copy(res, 0, r, JAVA_BYTE, 0, res.length);
			final MemorySegment o = a.allocate(JAVA_LONG, offsets.size());
			for (int i = 0; i < offsets.size(); ++i)
				o.setAtIndex(JAVA_LONG, i, offsets.get(i));
			if (nDevices == 1) {
				check((int) DbiNative.dbi_add_proteins.invoke(handle, r, o, offsets.size() - 1));
				if (unindexed) // the proteins are all there is: every query digests them (dbi_search_unindexed)
					return;
				check((int) DbiNative.dbi_build.invoke(handle));
			} else {
				// contiguous shards of about equal residue count, in protein order (ids stay global and in file order);
				// dbi_add_proteins takes offsets[first .. last] of the shared buffer as they are
				final int nProt = offsets.size() - 1;
				final long total = offsets.get(nProt);
				int first = 0;
				for (int d = 0; d < nDevices; ++d) {
					int last = nProt;
					if (d < nDevices - 1) {
						last = first;
						while (last < nProt && offsets.get(last) < total * (d + 1) / nDevices)
							++last;
					}
					check((int) DbiNative.dbi_add_proteins.invoke(handles[d], r, o.asSlice(8L * first), last - first));
					first = last;
				}
				if (unindexed) // every query digests the shards (dbi_mg_search_unindexed_local)
					return;
				// the whole exchange in one call: shard packing, NVLink pulls, own-shard digest, the two multisplit /
				// peer-memory scatter kernels into folded mass slices, per-GPU sort + merge + expansion
				final MemorySegment hs = a.allocate(ADDRESS, nDevices);
				for (int d = 0; d < nDevices; ++d)
					hs.setAtIndex(ADDRESS, d, handles[d]);
				check((int) DbiNative.dbi_mg_build_local.invoke(hs, nDevices));
				final int slices = (int) DbiNative.dbi_mg_slices.invoke(handle);
				final MemorySegment sm = a.allocate(JAVA_DOUBLE, Math.max(1, slices - 1));
				check((int) DbiNative.dbi_mg_split_masses.invoke(handle, sm));
				splitMass = new double[slices - 1];
				for (int i = 0; i < slices - 1; ++i)
					splitMass[i] = sm.getAtIndex(JAVA_DOUBLE, i);
			}
			built = true;
			if (indexFile != null)
				check((int) DbiNative.dbi_save.invoke(handle, a.allocateFrom(indexFile)));
		} catch (final DBIndexStoreException e) {
			throw e;
		} catch (final Throwable t) {
			throw new DBIndexStoreException("dbi_build failed", t);
		}
	}

	@Override
	public List<IndexedSequence> getSequences(double precMass, double tolerance) throws DBIndexStoreException {
		requireInit();
		double lo = precMass - tolerance; // Mult:324-329
		if (lo < 0)
			lo = 0;
		final double hi = precMass + tolerance;
		return query(new double[] { lo }, new double[] { hi });
	}

	@Override
	public List<IndexedSequence> getSequences(List<MassRange> ranges) throws DBIndexStoreException {
		if (ranges.size() == 1) // Mult:354-358
			return getSequences(ranges.get(0).getPrecMass(), ranges.get(0).getTolerance());
		requireInit();
		final ArrayList<Interval> intervals = new ArrayList<>();
		for (final MassRange r : ranges)
			intervals.add(Interval.massRangeToInterval(r)); // Interval.java:27-38
		final List<Interval> merged = MergeIntervals.mergeIntervals(intervals); // MergeIntervals.java:16-46
		final double[] lo = new double[merged.size()], hi = new double[merged.size()];
		for (int i = 0; i < merged.size(); ++i) {
			lo[i] = merged.get(i).getStart();
			hi[i] = merged.get(i).getEnd();
		}
		return query(lo, hi);
	}

	/**
	 * dbi_query_hits + dbi_query_hits_read: ONE device pass for all ranges of the call (bounds search, hit
	 * materialisation incl. peptide residues and flanks, one D2H per array), then the object assembly of
	 * parseAddPeptideInfo (Merge:452-477). The mod pattern (byte k = position + 1 of the k-th modified
	 * residue) travels in IndexedSequence.setModSequence-style notation so that variants of one peptide
	 * stay distinguishable.
	 */
	private List<IndexedSequence> query(double[] lo, double[] hi) throws DBIndexStoreException {
		final List<IndexedSequence> ret = new ArrayList<>();
		final int bucketRange = MAX_MASS / sparam.getIndexFactor();
		for (int i = 0; i < lo.length; ++i) // "Cannot query, unsupported precursor mass" -> empty (Mult:333-338)
			if ((int) lo[i] / bucketRange > sparam.getIndexFactor() - 1 || (int) hi[i] / bucketRange > sparam.getIndexFactor() - 1)
				return ret;
		if (unindexed) {
			// one range, or the merged intervals of getSequences(List<MassRange>), which are sorted by mass already: the
			// chunks of the mass-sorted batch come back in the caller's order
			searchUnindexed(lo, hi, (q, pep, resLeft, resRight, mass, off, pids, patterns) -> {
				for (final int mp : patterns)
					ret.add(sequence(pep, resLeft, resRight, mass, off, pids, mp));
			});
			return ret;
		}
		if (nDevices > 1) {
			// Mult.getSequences walks the buckets a range touches (:333-343); here: the GPUs owning the slices it
			// touches.  Slice s = [splitMass[s-1], splitMass[s]) lives on GPU s < N ? s : slices - 1 - s.
			final int slices = splitMass.length + 1;
			for (int d = 0; d < nDevices; ++d) {
				final List<Double> l = new ArrayList<>(), h = new ArrayList<>();
				for (int i = 0; i < lo.length; ++i) {
					boolean mine = false;
					for (int sl = 0; sl < slices && !mine; ++sl) {
						final int owner = sl < nDevices ? sl : slices - 1 - sl;
						final double left = sl == 0 ? Double.NEGATIVE_INFINITY : splitMass[sl - 1];
						final double right = sl == slices - 1 ? Double.POSITIVE_INFINITY : splitMass[sl];
						mine = owner == d && hi[i] >= left && lo[i] < right;
					}
					if (mine) {
						l.add(lo[i]);
						h.add(hi[i]);
					}
				}
				if (!l.isEmpty())
					queryOn(d, l.stream().mapToDouble(Double::doubleValue).toArray(),
							h.stream().mapToDouble(Double::doubleValue).toArray(), ret);
			}
			return ret;
		}
		queryOn(0, lo, hi, ret);
		return ret;
	}

	/** one dbi_query_hits + dbi_query_hits_read on this thread's view of GPU d; the hits are appended to ret */
	private void queryOn(int d, double[] lo, double[] hi, List<IndexedSequence> ret) throws DBIndexStoreException {
		try (Arena a = Arena.ofConfined()) {
			final MemorySegment handle = views()[d];
			final int nq = lo.length;
			final MemorySegment dlo = a.allocate(JAVA_DOUBLE, nq), dhi = a.allocate(JAVA_DOUBLE, nq);
			MemorySegment.copy(lo, 0, dlo, JAVA_DOUBLE, 0, nq);
			MemorySegment.copy(hi, 0, dhi, JAVA_DOUBLE, 0, nq);
			final MemorySegment cnt = a.allocate(DbiNative.HIT_COUNTS);
			check((int) DbiNative.dbi_query_hits.invoke(handle, dlo, dhi, (long) nq, cnt));
			readHits(handle, a, cnt, null, (q, pep, resLeft, resRight, mass, off, pids, patterns) -> {
				for (final int mp : patterns)
					ret.add(sequence(pep, resLeft, resRight, mass, off, pids, mp));
			});
		} catch (final DBIndexStoreException e) {
			throw e;
		} catch (final Throwable t) {
			throw new DBIndexStoreException("Error getting peptides ", t);
		}
	}

	/**
	 * A batch of spectra in one device call per chunk: tolMode DBI_TOL_DA, spectrum s = the ranges
	 * [rangeOff[s], rangeOff[s+1]) of (mass, tol in Da), answered as getSequences(List<MassRange>); DBI_TOL_PPM
	 * (rangeOff null), mass[s] at tol[s] ppm, answered as DBIndexer.getSequencesUsingPPMTolerance. The bucket rule
	 * of sparam.getIndexFactor() is applied on the device (dbi_query_spectra; SEARCH_UNINDEXED:
	 * dbi_search_unindexed_spectra, spectra sorted by mass and split into chunks like searchUnindexed, never inside
	 * a spectrum). With -Ddbindex.gpu.devices=N > 1: dbi_mg_query_spectra_local (SEARCH_UNINDEXED:
	 * dbi_mg_search_unindexed_spectra_local, chunked on the largest per-GPU N_c), then every GPU's share is read.
	 */
	public List<List<IndexedSequence>> querySpectra(double[] mass, double[] tol, long[] rangeOff, int tolMode)
			throws DBIndexStoreException {
		requireInit();
		final int n = rangeOff == null ? mass.length : rangeOff.length - 1;
		final List<List<IndexedSequence>> ret = new ArrayList<>();
		for (int i = 0; i < n; ++i)
			ret.add(new ArrayList<>());
		final RunSink sink = (q, pep, resLeft, resRight, m, off, pids, patterns) -> {
			for (final int mp : patterns)
				ret.get(q).add(sequence(pep, resLeft, resRight, m, off, pids, mp));
		};
		final Integer[] order = new Integer[n];
		for (int i = 0; i < n; ++i)
			order[i] = i;
		if (unindexed) { // by mass (a range list by its first range), as searchUnindexed sorts its ranges
			final double[] key = new double[n];
			for (int i = 0; i < n; ++i)
				key[i] = rangeOff == null ? mass[i] : rangeOff[i + 1] > rangeOff[i] ? mass[(int) rangeOff[i]] : 0;
			java.util.Arrays.sort(order, (x, y) -> Double.compare(key[x], key[y]));
		}
		final int[] ids = new int[n];
		for (int i = 0; i < n; ++i)
			ids[i] = order[i];
		spectraChunk(mass, tol, rangeOff, tolMode, ids, sink);
		return ret;
	}

	private void spectraChunk(double[] mass, double[] tol, long[] rangeOff, int tolMode, int[] ids, RunSink sink)
			throws DBIndexStoreException {
		if (unindexed || nDevices > 1)
			synchronized (ownerLock) {
				spectraChunkOn(mass, tol, rangeOff, tolMode, ids, sink);
			}
		else
			spectraChunkOn(mass, tol, rangeOff, tolMode, ids, sink);
	}

	private void spectraChunkOn(double[] mass, double[] tol, long[] rangeOff, int tolMode, int[] ids, RunSink sink)
			throws DBIndexStoreException {
		try (Arena a = Arena.ofConfined()) {
			final int n = ids.length;
			long nr = 0;
			for (final int i : ids)
				nr += rangeOff == null ? 1 : rangeOff[i + 1] - rangeOff[i];
			final MemorySegment dm = a.allocate(JAVA_DOUBLE, Math.max(1, nr)), dt = a.allocate(JAVA_DOUBLE, Math.max(1, nr));
			final MemorySegment dro = rangeOff == null ? MemorySegment.NULL : a.allocate(JAVA_LONG, n + 1);
			long r = 0;
			for (int k = 0; k < n; ++k) {
				final long r0 = rangeOff == null ? ids[k] : rangeOff[ids[k]];
				final long r1 = rangeOff == null ? ids[k] + 1 : rangeOff[ids[k] + 1];
				if (rangeOff != null)
					dro.setAtIndex(JAVA_LONG, k, r);
				for (long j = r0; j < r1; ++j, ++r) {
					dm.setAtIndex(JAVA_DOUBLE, r, mass[(int) j]);
					dt.setAtIndex(JAVA_DOUBLE, r, tol[(int) j]);
				}
			}
			if (rangeOff != null)
				dro.setAtIndex(JAVA_LONG, n, r);
			final MemorySegment cnt = a.allocate(DbiNative.HIT_COUNTS, nDevices), nCand = a.allocate(JAVA_LONG, nDevices);
			final MemorySegment hs = a.allocate(ADDRESS, nDevices);
			for (int d = 0; d < nDevices; ++d)
				hs.setAtIndex(ADDRESS, d, handles[d]);
			final int factor = sparam.getIndexFactor();
			final MemorySegment[] readFrom = !unindexed && nDevices == 1 ? views() : handles;
			if (!unindexed) {
				if (nDevices == 1)
					check((int) DbiNative.dbi_query_spectra.invoke(readFrom[0], dm, dt, dro, (long) n, tolMode, factor, cnt));
				else
					check((int) DbiNative.dbi_mg_query_spectra_local.invoke(hs, nDevices, dm, dt, dro, (long) n, tolMode,
							factor, cnt));
			} else {
				final int rc;
				if (nDevices == 1)
					rc = (int) DbiNative.dbi_search_unindexed_spectra.invoke(handle, dm, dt, dro, (long) n, tolMode, factor,
							maxCandidates, cnt, nCand);
				else
					rc = (int) DbiNative.dbi_mg_search_unindexed_spectra_local.invoke(hs, nDevices, dm, dt, dro, (long) n,
							tolMode, factor, maxCandidates, cnt, nCand);
				long nc = 0;
				for (int d = 0; d < nDevices; ++d)
					nc = Math.max(nc, nCand.getAtIndex(JAVA_LONG, d));
				if (rc == DbiNative.DBI_ERANGE && nc > maxCandidates && n > 1) {
					final int chunks = (int) Math.min(n, (nc + maxCandidates - 1) / maxCandidates + 1);
					for (int c = 0; c < chunks; ++c)
						spectraChunk(mass, tol, rangeOff, tolMode, java.util.Arrays.copyOfRange(ids,
								(int) ((long) n * c / chunks), (int) ((long) n * (c + 1) / chunks)), sink);
					return;
				}
				check(rc);
			}
			final long cb = DbiNative.HIT_COUNTS.byteSize();
			for (int d = 0; d < nDevices; ++d) // every GPU answers for the mass slices it owns
				readHits(readFrom[d], a, cnt.asSlice(d * cb, cb), ids, sink);
		} catch (final DBIndexStoreException e) {
			throw e;
		} catch (final Throwable t) {
			throw new DBIndexStoreException("Error getting peptides ", t);
		}
	}

	/** IndexedSequence as parseAddPeptideInfo builds it (Merge:452-462), the mod pattern as a mod sequence */
	private static IndexedSequence sequence(String pep, String resLeft, String resRight, double mass, int off,
			List<Integer> pids, int modPattern) {
		final IndexedSequence s = new IndexedSequence(0, mass, pep, resLeft, resRight);
		s.setProteinIds(pids);
		s.setSequenceOffset(off); // SURVEY Q10: the offset is known, hand it over
		if (modPattern != 0)
			s.setModSequence(modNotation(pep, modPattern));
		return s;
	}

	/** what readHits hands over per run: the caller's query number, the peptide, and the mod pattern of every hit */
	private interface RunSink {
		void run(int query, String pep, String resLeft, String resRight, double mass, int off, List<Integer> pids,
				int[] patterns) throws DBIndexStoreException;
	}

	/**
	 * SEARCH_UNINDEXED: the ranges sorted by mass go to dbi_search_unindexed (sharded: dbi_mg_search_unindexed_local,
	 * N_c = the largest per-GPU count); a batch whose candidate records exceed maxCandidates (DBI_ERANGE, N_c
	 * reported) is split into ceil(N_c / cap) + 1 contiguous chunks, again if needed.
	 * The sink sees the runs of every query, chunk by chunk in mass order, with the caller's query numbers.
	 */
	private void searchUnindexed(double[] lo, double[] hi, RunSink sink) throws DBIndexStoreException {
		final Integer[] order = new Integer[lo.length];
		for (int i = 0; i < order.length; ++i)
			order[i] = i;
		java.util.Arrays.sort(order, (x, y) -> Double.compare(lo[x], lo[y]));
		final int[] ids = new int[order.length];
		for (int i = 0; i < ids.length; ++i)
			ids[i] = order[i];
		synchronized (ownerLock) {
			searchChunk(lo, hi, ids, sink);
		}
	}

	private void searchChunk(double[] lo, double[] hi, int[] ids, RunSink sink) throws DBIndexStoreException {
		try (Arena a = Arena.ofConfined()) {
			final int nq = ids.length;
			final MemorySegment dlo = a.allocate(JAVA_DOUBLE, Math.max(1, nq)), dhi = a.allocate(JAVA_DOUBLE, Math.max(1, nq));
			for (int i = 0; i < nq; ++i) {
				dlo.setAtIndex(JAVA_DOUBLE, i, lo[ids[i]]);
				dhi.setAtIndex(JAVA_DOUBLE, i, hi[ids[i]]);
			}
			final MemorySegment cnt = a.allocate(DbiNative.HIT_COUNTS, nDevices), nCand = a.allocate(JAVA_LONG, nDevices);
			final int rc;
			if (nDevices == 1) {
				rc = (int) DbiNative.dbi_search_unindexed.invoke(handle, dlo, dhi, (long) nq, maxCandidates, cnt, nCand);
			} else {
				final MemorySegment hs = a.allocate(ADDRESS, nDevices);
				for (int d = 0; d < nDevices; ++d)
					hs.setAtIndex(ADDRESS, d, handles[d]);
				rc = (int) DbiNative.dbi_mg_search_unindexed_local.invoke(hs, nDevices, dlo, dhi, (long) nq, maxCandidates,
						cnt, nCand);
			}
			long nc = 0;
			for (int d = 0; d < nDevices; ++d)
				nc = Math.max(nc, nCand.getAtIndex(JAVA_LONG, d));
			if (rc == DbiNative.DBI_ERANGE && nc > maxCandidates && nq > 1) {
				final int chunks = (int) Math.min(nq, (nc + maxCandidates - 1) / maxCandidates + 1);
				for (int c = 0; c < chunks; ++c)
					searchChunk(lo, hi, java.util.Arrays.copyOfRange(ids, (int) ((long) nq * c / chunks),
							(int) ((long) nq * (c + 1) / chunks)), sink);
				return;
			}
			check(rc);
			final long cb = DbiNative.HIT_COUNTS.byteSize();
			for (int d = 0; d < nDevices; ++d) // every GPU answers for the mass slices it owns in this call
				readHits(handles[d], a, cnt.asSlice(d * cb, cb), ids, sink);
		} catch (final DBIndexStoreException e) {
			throw e;
		} catch (final Throwable t) {
			throw new DBIndexStoreException("Error getting peptides ", t);
		}
	}

	/** dbi_query_hits_read of the pending result; queryIds: the caller's number of every query (null = itself) */
	private void readHits(MemorySegment handle, Arena a, MemorySegment cnt, int[] queryIds, RunSink sink)
			throws Throwable {
		{
			// the answer comes back grouped in RUNS (consecutive hits that are variants of one peptide with one
			// mass): peptide string, flanks, first occurrence and protein list once per run, the mod pattern per hit
			final long nq = cnt.get(JAVA_LONG, 0), nHits = cnt.get(JAVA_LONG, 8), nPeps = cnt.get(JAVA_LONG, 16),
					nSeq = cnt.get(JAVA_LONG, 24), nIds = cnt.get(JAVA_LONG, 32);
			final MemorySegment pat = a.allocate(JAVA_INT, Math.max(1, nHits));
			final MemorySegment pepHitOff = a.allocate(JAVA_LONG, nPeps + 1);
			final MemorySegment mass = a.allocate(JAVA_DOUBLE, Math.max(1, nPeps));
			final MemorySegment prot = a.allocate(JAVA_INT, Math.max(1, nPeps)), off = a.allocate(JAVA_INT, Math.max(1, nPeps));
			final MemorySegment len = a.allocate(JAVA_SHORT, Math.max(1, nPeps));
			final MemorySegment flanks = a.allocate(Math.max(1, 6 * nPeps));
			final MemorySegment seqOff = a.allocate(JAVA_LONG, nPeps + 1), seq = a.allocate(Math.max(1, nSeq));
			final MemorySegment plo = a.allocate(JAVA_LONG, nPeps + 1), ids = a.allocate(JAVA_INT, Math.max(1, nIds));
			final MemorySegment pepOff = a.allocate(JAVA_LONG, nq + 1);
			final MemorySegment bufs = a.allocate(DbiNative.HIT_BUFFERS);
			final MemorySegment[] order = { MemorySegment.NULL /* hit_off */, pepOff, pat, pepHitOff, mass, prot, off, len,
					flanks, seqOff, seq, plo, ids };
			for (int k = 0; k < order.length; ++k)
				bufs.setAtIndex(ADDRESS, k, order[k]);
			check((int) DbiNative.dbi_query_hits_read.invoke(handle, bufs));
			final byte[] seqBytes = seq.asSlice(0, nSeq).toArray(JAVA_BYTE);
			final byte[] flankBytes = flanks.asSlice(0, 6 * nPeps).toArray(JAVA_BYTE);
			int q = 0;
			for (long p = 0; p < nPeps; ++p) {
				while (pepOff.getAtIndex(JAVA_LONG, q + 1) <= p) // the query this run belongs to
					++q;
				final int s0 = (int) seqOff.getAtIndex(JAVA_LONG, p), s1 = (int) seqOff.getAtIndex(JAVA_LONG, p + 1);
				final String pep = new String(seqBytes, s0, s1 - s0, java.nio.charset.StandardCharsets.ISO_8859_1);
				final String resLeft = new String(flankBytes, (int) (6 * p), 3, java.nio.charset.StandardCharsets.ISO_8859_1);
				final String resRight = new String(flankBytes, (int) (6 * p + 3), 3, java.nio.charset.StandardCharsets.ISO_8859_1);
				final List<Integer> pids = new ArrayList<>();
				for (long k = plo.getAtIndex(JAVA_LONG, p); k < plo.getAtIndex(JAVA_LONG, p + 1); ++k)
					pids.add(ids.getAtIndex(JAVA_INT, k));
				final long h0 = pepHitOff.getAtIndex(JAVA_LONG, p), h1 = pepHitOff.getAtIndex(JAVA_LONG, p + 1);
				final int[] patterns = new int[(int) (h1 - h0)];
				for (long i = h0; i < h1; ++i)
					patterns[(int) (i - h0)] = pat.getAtIndex(JAVA_INT, i);
				sink.run(queryIds == null ? q : queryIds[q], pep, resLeft, resRight, mass.getAtIndex(JAVA_DOUBLE, p),
						off.getAtIndex(JAVA_INT, p), pids, patterns);
			}
		}
	}

	/** pattern byte k = position + 1 of the k-th modified residue -> "PEPT(+79.9663)IDE". */
	private static String modNotation(String pep, int pattern) {
		final double[] diff = edu.scripps.yates.dbindex.model.DiffModification.getDiffMod();
		final StringBuilder sb = new StringBuilder();
		for (int i = 0; i < pep.length(); ++i) {
			sb.append(pep.charAt(i));
			for (int k = 0; k < 4; ++k)
				if (((pattern >>> (8 * k)) & 0xff) == i + 1)
					sb.append("(").append(String.format(java.util.Locale.ROOT, "%+.4f", diff[pep.charAt(i)])).append(")");
		}
		return sb.toString();
	}

	/**
	 * getProteins(String) (DBIndexer.java:925-947) for a whole list in one dbi_lookup_peptides + _read per GPU: the
	 * proteins of the unmodified entry whose peptide equals each string (its mass computed on the device the way
	 * the index computes it), an empty set when there is none or when that mass has no bucket (Mult:333-338). A
	 * sharded index asks every GPU: a row is found at most once, by the owner of the slice holding its mass.
	 */
	public List<java.util.Set<IndexedProtein>> lookupPeptides(List<String> peptides) throws DBIndexStoreException {
		requireInit();
		final int n = peptides.size();
		final List<java.util.Set<IndexedProtein>> ret = new ArrayList<>(n);
		for (int i = 0; i < n; ++i)
			ret.add(new java.util.HashSet<>());
		final int bucketRange = MAX_MASS / sparam.getIndexFactor();
		if (unindexed)
			return lookupUnindexed(peptides, ret, bucketRange);
		try (Arena a = Arena.ofConfined()) {
			final java.io.ByteArrayOutputStream packed = new java.io.ByteArrayOutputStream();
			final MemorySegment off = a.allocate(JAVA_LONG, n + 1L);
			for (int i = 0; i < n; ++i) {
				final byte[] b = peptides.get(i).getBytes(java.nio.charset.StandardCharsets.ISO_8859_1);
				packed.write(b, 0, b.length);
				off.setAtIndex(JAVA_LONG, i + 1, packed.size());
			}
			final byte[] res = packed.toByteArray();
			final MemorySegment r = a.allocate(Math.max(1, res.length));
			MemorySegment.copy(res, 0, r, JAVA_BYTE, 0, res.length);
			final boolean[] found = new boolean[n];
			for (final MemorySegment h : views()) {
				final MemorySegment cnt = a.allocate(DbiNative.LOOKUP_COUNTS);
				check((int) DbiNative.dbi_lookup_peptides.invoke(h, r, off, MemorySegment.NULL, (long) n, cnt));
				final long nIds = cnt.get(JAVA_LONG, 16);
				final MemorySegment status = a.allocate(Math.max(1, n)), mass = a.allocate(JAVA_DOUBLE, Math.max(1, n));
				final MemorySegment plo = a.allocate(JAVA_LONG, n + 1L), ids = a.allocate(JAVA_INT, Math.max(1, nIds));
				final MemorySegment bufs = a.allocate(DbiNative.LOOKUP_BUFFERS);
				final MemorySegment[] order = { status, mass, MemorySegment.NULL /* entry */, MemorySegment.NULL /* first_prot */,
						MemorySegment.NULL /* first_off */, plo, ids };
				for (int k = 0; k < order.length; ++k)
					bufs.setAtIndex(ADDRESS, k, order[k]);
				check((int) DbiNative.dbi_lookup_peptides_read.invoke(h, bufs));
				for (int i = 0; i < n; ++i) {
					if (status.get(JAVA_BYTE, i) != 1)
						continue;
					if (found[i])
						throw new DBIndexStoreException("peptide " + peptides.get(i) + " found on two GPUs");
					found[i] = true;
					final double m = mass.getAtIndex(JAVA_DOUBLE, i);
					if ((int) m / bucketRange > sparam.getIndexFactor() - 1)
						continue; // the zero-tolerance query of the reference returns nothing there
					for (long k = plo.getAtIndex(JAVA_LONG, i); k < plo.getAtIndex(JAVA_LONG, i + 1); ++k) {
						final int id = ids.getAtIndex(JAVA_INT, k);
						ret.get(i).add(new IndexedProtein(proteinCache.getProteinDef(id), id));
					}
				}
			}
		} catch (final DBIndexStoreException e) {
			throw e;
		} catch (final Throwable t) {
			throw new DBIndexStoreException("Error looking peptides up ", t);
		}
		return ret;
	}

	/**
	 * SEARCH_UNINDEXED getProteins(String): the reference's own route (DBIndexer.java:925-947) -- the mass by
	 * IndexUtil.calculateMass (dbi_calculate_mass), one search with zero-width windows, and the proteins of the
	 * unmodified hit whose peptide equals the string.
	 */
	private List<java.util.Set<IndexedProtein>> lookupUnindexed(List<String> peptides, List<java.util.Set<IndexedProtein>> ret,
			int bucketRange) throws DBIndexStoreException {
		final int n = peptides.size();
		final double[] m = new double[n];
		try (Arena a = Arena.ofConfined()) {
			final MemorySegment out = a.allocate(JAVA_DOUBLE);
			for (int i = 0; i < n; ++i) {
				final byte[] b = peptides.get(i).getBytes(java.nio.charset.StandardCharsets.ISO_8859_1);
				final MemorySegment seg = a.allocate(Math.max(1, b.length));
				MemorySegment.copy(b, 0, seg, JAVA_BYTE, 0, b.length);
				check((int) DbiNative.dbi_calculate_mass.invoke(handle, seg, (long) b.length, out));
				m[i] = out.get(JAVA_DOUBLE, 0);
			}
		} catch (final DBIndexStoreException e) {
			throw e;
		} catch (final Throwable t) {
			throw new DBIndexStoreException("dbi_calculate_mass failed", t);
		}
		searchUnindexed(m, m, (q, pep, resLeft, resRight, mass, off, pids, patterns) -> {
			if ((int) m[q] / bucketRange > sparam.getIndexFactor() - 1 || !pep.equals(peptides.get(q)))
				return;
			for (final int mp : patterns)
				if (mp == 0)
					for (final int id : pids)
						ret.get(q).add(new IndexedProtein(proteinCache.getProteinDef(id), id));
		});
		return ret;
	}

	@Override
	public Iterator<IndexedSequence> getSequencesIterator(List<MassRange> ranges) throws DBIndexStoreException {
		return getSequences(ranges).iterator(); // Mult:634-636
	}

	@Override
	public void setProteinCache(ProteinCache proteinCache) {
		this.proteinCache = proteinCache;
	}

	@Override
	public boolean supportsProteinCache() {
		return true; // Mult:433-436
	}

	@Override
	public List<IndexedProtein> getProteins(IndexedSequence sequence) {
		final List<IndexedProtein> ret = new ArrayList<>(); // Mult:453-463
		for (final int id : sequence.getProteinIds())
			ret.add(new IndexedProtein(proteinCache.getProteinDef(id), id));
		return ret;
	}

	@Override
	public long getNumberSequences() throws DBIndexStoreException {
		requireInit();
		if (unindexed)
			throw new DBIndexStoreException("not available in unindexed search mode (useIndex = false): there is no index");
		try (Arena a = Arena.ofConfined()) {
			long total = 0;
			for (final MemorySegment h : handles) {
				final MemorySegment st = a.allocate(512);
				check((int) DbiNative.dbi_stats_get.invoke(h, st));
				total += st.get(JAVA_LONG, 32); // dbi_stats.n_entries
			}
			return total;
		} catch (final DBIndexStoreException e) {
			throw e;
		} catch (final Throwable t) {
			throw new DBIndexStoreException("dbi_stats_get failed", t);
		}
	}

	@Override
	public ResidueInfo getResidues(IndexedSequence peptideSequence, IndexedProtein protein) {
		final String protSeq = proteinCache.getProteinSequence((int) protein.getId());
		int off = peptideSequence.getSequenceOffset();
		if (off == IndexedSequence.OFFSET_UNKNOWN)
			off = protSeq.indexOf(peptideSequence.getSequence()); // Mult:303-312
		return Util.getResidues(peptideSequence, off, peptideSequence.getSequenceLen(), protSeq);
	}

	@Override
	public List<Integer> getEntryKeys() throws DBIndexStoreException {
		requireInit();
		if (unindexed)
			throw new DBIndexStoreException("not available in unindexed search mode (useIndex = false): there is no index");
		try (Arena a = Arena.ofConfined()) {
			final List<Integer> ret = new ArrayList<>();
			for (final MemorySegment h : handles) { // Mult.getEntryKeys concatenates its buckets the same way (:196-201)
				final MemorySegment n = a.allocate(JAVA_LONG);
				check((int) DbiNative.dbi_entry_keys.invoke(h, MemorySegment.NULL, 0L, n));
				final long k = n.get(JAVA_LONG, 0);
				final MemorySegment keys = a.allocate(JAVA_INT, Math.max(1, k));
				check((int) DbiNative.dbi_entry_keys.invoke(h, keys, k, n));
				for (long i = 0; i < k; ++i)
					ret.add(keys.getAtIndex(JAVA_INT, i));
			}
			return ret;
		} catch (final DBIndexStoreException e) {
			throw e;
		} catch (final Throwable t) {
			throw new DBIndexStoreException("dbi_entry_keys failed", t);
		}
	}

	@Override
	public void lastBuffertoDatabase() {
		throw new UnsupportedOperationException("Not supported yet."); // Mult:620-622
	}

	public void close() {
		for (MemorySegment v; (v = openViews.poll()) != null;)
			try {
				DbiNative.dbi_destroy.invoke(v);
			} catch (final Throwable ignored) {
			}
		for (final MemorySegment h : handles)
			try {
				if (h != null && !h.equals(MemorySegment.NULL))
					DbiNative.dbi_destroy.invoke(h);
			} catch (final Throwable ignored) {
			}
		handles = new MemorySegment[0];
		handle = MemorySegment.NULL;
		arena.close();
	}
}
