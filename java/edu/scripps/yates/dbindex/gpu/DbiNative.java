package edu.scripps.yates.dbindex.gpu;

import java.lang.foreign.Arena;
import java.lang.foreign.FunctionDescriptor;
import java.lang.foreign.Linker;
import java.lang.foreign.MemoryLayout;
import java.lang.foreign.MemorySegment;
import java.lang.foreign.StructLayout;
import java.lang.foreign.SymbolLookup;
import java.lang.invoke.MethodHandle;

import static java.lang.foreign.ValueLayout.ADDRESS;
import static java.lang.foreign.ValueLayout.JAVA_BYTE;
import static java.lang.foreign.ValueLayout.JAVA_DOUBLE;
import static java.lang.foreign.ValueLayout.JAVA_INT;
import static java.lang.foreign.ValueLayout.JAVA_LONG;

/**
 * Panama FFM (java.lang.foreign, JDK 22+) binding of include/dbindex_gpu.h. No jni.h and no generated
 * glue: every entry point is a downcall handle on the C ABI of libdbindex_gpu.so.
 *
 * NOT COMPILED IN THIS REPOSITORY: the build image has no JDK and the reference's core dependency
 * (edu.scripps.yates:utilities:1.6-SNAPSHOT) is not vendored. The same calls are exercised from Python
 * (dbindex_b200/capi.py); this file is what a dbIndex maintainer drops next to DBIndexStoreSQLiteMult.
 * tests/test_java_layout.py and tests/test_peptide_lookup.py parse the layouts below and checks every field offset against
 * offsetof() of the compiled C structs, so a drift fails in CI without a JDK.
 */
public final class DbiNative {
	public static final int DBI_OK = 0, DBI_ENOTINIT = -1, DBI_EALREADY = -2, DBI_EINVAL = -3, DBI_ENOMEM = -4,
			DBI_ECUDA = -5, DBI_ENCCL = -6, DBI_ERANGE = -7;
	public static final int DBI_ABI_VERSION = 3, DBI_MAX_MODS = 16;

	/** struct dbi_mod { uint8_t residue; uint8_t _pad[7]; double delta; } */
	static final StructLayout MOD = MemoryLayout.structLayout(JAVA_BYTE.withName("residue"),
			MemoryLayout.paddingLayout(7), JAVA_DOUBLE.withName("delta"));

	/** struct dbi_params, field for field; the only padding is the 4 bytes before mods[] (see dbi_abi_sizes). */
	static final StructLayout PARAMS = MemoryLayout.structLayout(JAVA_INT.withName("abi_version"),
			JAVA_INT.withName("device"), MemoryLayout.sequenceLayout(256, JAVA_DOUBLE).withName("residue_mass"),
			JAVA_DOUBLE.withName("h2o_proton"), JAVA_DOUBLE.withName("nterm"), JAVA_DOUBLE.withName("cterm"),
			JAVA_INT.withName("add_h2o_proton"), MemoryLayout.sequenceLayout(256, JAVA_BYTE).withName("is_enzyme"),
			MemoryLayout.sequenceLayout(256, JAVA_BYTE).withName("is_nocut"), JAVA_INT.withName("max_missed"),
			JAVA_INT.withName("semi"), JAVA_INT.withName("min_len"),
			JAVA_DOUBLE.withName("min_mass"), JAVA_DOUBLE.withName("max_mass"), JAVA_INT.withName("mass_group_factor"),
			JAVA_INT.withName("n_mods"), JAVA_INT.withName("max_mods_per_peptide"), MemoryLayout.paddingLayout(4),
			MemoryLayout.sequenceLayout(DBI_MAX_MODS, MOD).withName("mods"),
			MemoryLayout.sequenceLayout(256, JAVA_BYTE).withName("is_mandatory"), JAVA_INT.withName("has_mandatory"),
			JAVA_INT.withName("filter_aa"), JAVA_INT.withName("filter_max"), JAVA_INT.withName("_pad_filters"),
			JAVA_INT.withName("keep_emitted"), JAVA_INT.withName("profile"),
			MemoryLayout.sequenceLayout(6, JAVA_INT).withName("reserved"));

	/** struct dbi_hit_counts */
	static final StructLayout HIT_COUNTS = MemoryLayout.structLayout(JAVA_LONG.withName("nq"),
			JAVA_LONG.withName("n_hits"), JAVA_LONG.withName("n_peps"), JAVA_LONG.withName("n_seq_bytes"),
			JAVA_LONG.withName("n_prot_ids"));

	/** struct dbi_hit_buffers: thirteen caller-owned output pointers (hits grouped in runs of one peptide and mass) */
	static final StructLayout HIT_BUFFERS = MemoryLayout.structLayout(ADDRESS.withName("hit_off"),
			ADDRESS.withName("pep_off"), ADDRESS.withName("modpat"), ADDRESS.withName("pep_hit_off"),
			ADDRESS.withName("mass"), ADDRESS.withName("first_prot"), ADDRESS.withName("first_off"),
			ADDRESS.withName("len"), ADDRESS.withName("flanks"), ADDRESS.withName("seq_off"), ADDRESS.withName("seq"),
			ADDRESS.withName("prot_list_off"), ADDRESS.withName("prot_ids"));

	/** struct dbi_lookup_counts */
	static final StructLayout LOOKUP_COUNTS = MemoryLayout.structLayout(JAVA_LONG.withName("n"),
			JAVA_LONG.withName("n_found"), JAVA_LONG.withName("n_prot_ids"));

	/** struct dbi_lookup_buffers: seven caller-owned output pointers (one row per looked-up peptide) */
	static final StructLayout LOOKUP_BUFFERS = MemoryLayout.structLayout(ADDRESS.withName("status"),
			ADDRESS.withName("mass"), ADDRESS.withName("entry"), ADDRESS.withName("first_prot"),
			ADDRESS.withName("first_off"), ADDRESS.withName("prot_list_off"), ADDRESS.withName("prot_ids"));

	private static final Linker LINKER = Linker.nativeLinker();
	private static final SymbolLookup LIB = SymbolLookup
			.libraryLookup(System.getProperty("dbindex.gpu.lib", "libdbindex_gpu.so"), Arena.global());

	private static MethodHandle h(String name, FunctionDescriptor fd) {
		return LINKER.downcallHandle(LIB.find(name).orElseThrow(() -> new UnsatisfiedLinkError(name)), fd);
	}

	static final MethodHandle dbi_default_params = h("dbi_default_params", FunctionDescriptor.ofVoid(ADDRESS, JAVA_INT));
	static final MethodHandle dbi_params_add_diff_mod = h("dbi_params_add_diff_mod",
			FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_DOUBLE));
	static final MethodHandle dbi_abi_sizes = h("dbi_abi_sizes", FunctionDescriptor.ofVoid(ADDRESS, ADDRESS));
	static final MethodHandle dbi_create = h("dbi_create", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
	static final MethodHandle dbi_add_proteins = h("dbi_add_proteins",
			FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_INT));
	static final MethodHandle dbi_build = h("dbi_build", FunctionDescriptor.of(JAVA_INT, ADDRESS));
	static final MethodHandle dbi_save = h("dbi_save", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
	static final MethodHandle dbi_load = h("dbi_load", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
	static final MethodHandle dbi_query = h("dbi_query",
			FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS, ADDRESS));
	// batched parseAddPeptideInfo: every hit of every range of one call, materialised on the device
	static final MethodHandle dbi_query_hits = h("dbi_query_hits",
			FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS));
	static final MethodHandle dbi_query_hits_read = h("dbi_query_hits_read",
			FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
	// SEARCH_UNINDEXED: the hits of a batch from the proteins, no index kept; read with dbi_query_hits_read
	static final MethodHandle dbi_search_unindexed = h("dbi_search_unindexed",
			FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, JAVA_LONG, ADDRESS, ADDRESS));
	// batched getProteins(String): which entry (and so which proteins) every peptide of a list is
	// a batch of spectra (Dalton range lists or PPM masses) answered as getSequences(List<MassRange>) /
	// getSequencesUsingPPMTolerance answer one; read with dbi_query_hits_read, one query per spectrum
	static final int DBI_TOL_DA = 0, DBI_TOL_PPM = 1;
	static final MethodHandle dbi_query_spectra = h("dbi_query_spectra",
			FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, JAVA_INT, JAVA_INT, ADDRESS));
	static final MethodHandle dbi_search_unindexed_spectra = h("dbi_search_unindexed_spectra",
			FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, JAVA_INT, JAVA_INT, JAVA_LONG,
					ADDRESS, ADDRESS));
	static final MethodHandle dbi_lookup_peptides = h("dbi_lookup_peptides",
			FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS));
	static final MethodHandle dbi_lookup_peptides_read = h("dbi_lookup_peptides_read",
			FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
	static final MethodHandle dbi_host_alloc = h("dbi_host_alloc", FunctionDescriptor.of(JAVA_INT, JAVA_LONG, ADDRESS));
	static final MethodHandle dbi_host_free = h("dbi_host_free", FunctionDescriptor.of(JAVA_INT, ADDRESS));
	static final MethodHandle dbi_fetch = h("dbi_fetch", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_LONG, JAVA_LONG,
			ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS));
	static final MethodHandle dbi_entry_keys = h("dbi_entry_keys",
			FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS));
	static final MethodHandle dbi_stats_get = h("dbi_stats_get", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
	static final MethodHandle dbi_calculate_mass = h("dbi_calculate_mass",
			FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS));
	// host-side FASTA ingest (csrc/fasta.cpp): packed residues + offsets + deflines for dbi_add_proteins
	static final MethodHandle dbi_fasta_open = h("dbi_fasta_open", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, ADDRESS));
	static final MethodHandle dbi_fasta_counts = h("dbi_fasta_counts",
			FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS));
	static final MethodHandle dbi_fasta_read = h("dbi_fasta_read",
			FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS));
	static final MethodHandle dbi_fasta_close = h("dbi_fasta_close", FunctionDescriptor.ofVoid(ADDRESS));
	// sharded build with one handle per GPU inside this JVM: the whole exchange (shard packing, NVLink pulls, the
	// two multisplit / peer-memory scatter kernels) is one call; afterwards every handle answers for its mass slice
	// and reads base peptides owned by another GPU through the mapped window of that GPU
	static final MethodHandle dbi_mg_build_local = h("dbi_mg_build_local", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT));
	// SEARCH_UNINDEXED over those handles: every GPU digests its shard, indexes its mass slices for this batch only and
	// keeps its hits pending (dbi_query_hits_read on each handle)
	static final MethodHandle dbi_mg_search_unindexed_local = h("dbi_mg_search_unindexed_local", FunctionDescriptor.of(
			JAVA_INT, ADDRESS, JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, JAVA_LONG, ADDRESS, ADDRESS));
	// spectrum batches over those handles (built index / SEARCH_UNINDEXED): every GPU keeps its share of every
	// spectrum pending, the PPM probe walk ending where the GPU owning the first empty probe says
	static final MethodHandle dbi_mg_query_spectra_local = h("dbi_mg_query_spectra_local", FunctionDescriptor.of(
			JAVA_INT, ADDRESS, JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, JAVA_INT, JAVA_INT, ADDRESS));
	static final MethodHandle dbi_mg_search_unindexed_spectra_local = h("dbi_mg_search_unindexed_spectra_local",
			FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, JAVA_INT, JAVA_INT,
					JAVA_LONG, ADDRESS, ADDRESS));
	static final MethodHandle dbi_mg_slices = h("dbi_mg_slices", FunctionDescriptor.of(JAVA_INT, ADDRESS));
	static final MethodHandle dbi_mg_split_masses = h("dbi_mg_split_masses", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
	static final MethodHandle dbi_destroy = h("dbi_destroy", FunctionDescriptor.ofVoid(ADDRESS));
	static final MethodHandle dbi_last_error = h("dbi_last_error", FunctionDescriptor.of(ADDRESS));

	static {
		try (Arena a = Arena.ofConfined()) {
			MemorySegment sp = a.allocate(JAVA_LONG), ss = a.allocate(JAVA_LONG);
			dbi_abi_sizes.invoke(sp, ss);
			if (sp.get(JAVA_LONG, 0) != PARAMS.byteSize())
				throw new IllegalStateException("dbi_params layout mismatch: native " + sp.get(JAVA_LONG, 0)
						+ " vs " + PARAMS.byteSize());
		} catch (Throwable t) {
			throw new ExceptionInInitializerError(t);
		}
	}

	static String lastError() {
		try {
			MemorySegment p = (MemorySegment) dbi_last_error.invoke();
			return p.reinterpret(512).getString(0);
		} catch (Throwable t) {
			return t.toString();
		}
	}

	private DbiNative() {
	}
}
