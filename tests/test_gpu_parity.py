"""GPU parity: the CUDA path through the C ABI versus the CPU oracle, bit-exact (-m gpu)."""
import numpy as np
import pytest

from oracle import oracle
from tests import inputs

pytestmark = pytest.mark.gpu


def gpu_build(genomes, k, min_abundance=1, keep_singletons=False, kind=0, **kw):
    from grm_b200.builder import KmerMatrixBuilder
    with KmerMatrixBuilder(k=k, min_abundance=min_abundance, keep_singletons=keep_singletons, input_kind=kind, **kw) as b:
        b.set_genome_count(len(genomes))
        for row, files in enumerate(genomes):
            for f in files:
                b.add_genome_bytes(row, f)
        b.build()
        return b.kmers(), b.matrix(), b.stats


def check(genomes, k, min_abundance=1, keep_singletons=False, kind=0, **kw):
    ref = oracle.build([[(f, kind) for f in files] for files in genomes], k, min_abundance, keep_singletons)
    kmers, mat, stats = gpu_build(genomes, k, min_abundance, keep_singletons, kind, **kw)
    assert stats["n_bases"] == ref.n_bases, (stats, ref.n_bases)
    assert stats["n_windows"] == ref.n_windows, (stats, ref.n_windows)
    assert kmers.shape == ref.kmers.shape, (kmers.shape, ref.kmers.shape, stats)
    assert np.array_equal(kmers, ref.kmers)
    assert mat.shape == ref.matrix.shape
    assert np.array_equal(mat, ref.matrix)
    return stats


def test_known_answer_k4(gpu):
    fa = b">r1\nGATTACAGGTNACCTGTAATC\n"
    kmers, mat, stats = gpu_build([[fa]], 5, keep_singletons=True)
    want = np.array([0x4F, 0x5B, 0xA1, 0x1B8, 0x209, 0x284], dtype=np.uint64)
    assert np.array_equal(kmers, want[oracle.column_order(want)])          # default column order: ascending hash
    assert np.array_equal(np.sort(kmers), want)
    assert stats["n_windows"] == 12 and stats["n_bases"] == 21 and stats["n_records"] == 1
    assert (mat == np.uint64(1) << np.uint64(63)).all()


@pytest.mark.parametrize("k", [1, 5, 15, 21, 31, 32])
@pytest.mark.parametrize("keep", [False, True])
def test_random_small(gpu, k, keep):
    rng = np.random.default_rng(1000 + k)
    shared = [inputs.rand_seq(rng, 700), inputs.rand_seq(rng, 300)]
    genomes = [[inputs.fasta(rng, n_records=int(rng.integers(1, 6)), shared=shared, blank=True)] for _ in range(7)]
    check(genomes, k, keep_singletons=keep)


@pytest.mark.parametrize("G", [1, 2, 63, 64, 65, 130])
def test_genome_counts_cross_word(gpu, G):
    rng = np.random.default_rng(G)
    shared = [inputs.rand_seq(rng, 400)]
    genomes = [[inputs.fasta(rng, n_records=2, max_len=150, shared=shared)] for _ in range(G)]
    check(genomes, 11, keep_singletons=(G % 2 == 0))


def test_text_quirks(gpu):
    rng = np.random.default_rng(7)
    shared = [inputs.rand_seq(rng, 500)]
    variants = [
        dict(crlf=True), dict(final_nl=False), dict(junk_prefix=True), dict(width=7), dict(width=0),
        dict(width=4096 + 37, max_len=20000), dict(p_n=0.2), dict(p_lower=1.0), dict(blank=True, crlf=True),
        dict(min_len=0, max_len=12), dict(p_iupac=0.1),
    ]
    genomes = [[inputs.fasta(rng, n_records=4, shared=shared, **v)] for v in variants]
    check(genomes, 9, keep_singletons=True)
    check(genomes, 31, keep_singletons=False)


def test_degenerate_inputs(gpu):
    long_header = b">" + b"x" * 10000 + b"\nACGTACGTACGTACGTTTGACCA\n"
    genomes = [
        [b""],                                  # empty file
        [b"no header at all\nACGTACGT\n"],      # never starts a record
        [b">only header"],
        [b">h\n"],
        [long_header],
        [b">a\nACGT\n>b\nACGTACGTACGTACGTTTGACCA"],  # no trailing newline
        [b"\n\n\n>x\n\nACGTACG\n\nTACGTACGTTTGACCA\n\n"],
        [b">e1\n>e2\n>e3\nACGTACGTACGTACGTTTGACCA\n>e4\n"],
    ]
    check(genomes, 8, keep_singletons=True)
    check(genomes, 8, keep_singletons=False)


def test_multiple_files_and_empty_rows(gpu):
    rng = np.random.default_rng(3)
    shared = [inputs.rand_seq(rng, 600)]
    genomes = [
        [inputs.fasta(rng, shared=shared), inputs.fasta(rng, shared=shared), inputs.fasta(rng, shared=shared)],
        [],
        [inputs.fasta(rng, shared=shared)],
        [],
    ]
    check(genomes, 13, keep_singletons=True)


def test_large_tiles_and_overflow_splits(gpu):
    # several tiles / scan blocks per file, and a bucket count too small for the table -> sub-range splits
    rng = np.random.default_rng(11)
    shared = [inputs.rand_seq(rng, 300_000)]
    genomes = [[inputs.fasta(rng, n_records=3, min_len=100_000, max_len=200_000, shared=shared, p_shared=0.5)]
               for _ in range(5)]
    stats = check(genomes, 31, keep_singletons=True, bucket_bits=4)
    assert stats["n_splits"] > 0
    check(genomes, 31, keep_singletons=False)


@pytest.mark.parametrize("min_ab", [1, 2, 3])
def test_fastq_reads(gpu, min_ab):
    rng = np.random.default_rng(50 + min_ab)
    src = [inputs.rand_seq(rng, 3000) for _ in range(3)]
    genomes = []
    for g in range(6):
        s = src[g % 3]
        genomes.append([inputs.fastq(rng, s, n_reads=400, read_len=60, crlf=(g == 1), final_nl=(g != 2)),
                        inputs.fastq(rng, s, n_reads=100, read_len=45)])
    check(genomes, 21, min_abundance=min_ab, keep_singletons=False, kind=1)
    check(genomes, 21, min_abundance=min_ab, keep_singletons=True, kind=1)


def test_tsv_and_strings(gpu):
    from grm_b200.builder import KmerMatrixBuilder
    rng = np.random.default_rng(5)
    shared = [inputs.rand_seq(rng, 800)]
    genomes = [[inputs.fasta(rng, shared=shared)] for _ in range(5)]
    names = ["562.1", "my genome", "b", "c", "d"]
    ref = oracle.build([[(f, 0) for f in files] for files in genomes], 17, 1, True, want_tsv_names=names)
    with KmerMatrixBuilder(k=17, keep_singletons=True) as b:
        for row, files in enumerate(genomes):
            b.add_genome_bytes(row, files[0])
        b.build()
        assert b.tsv(names).tobytes() == ref.tsv
        strs = b.kmer_strings()
        assert [s.decode() for s in strs] == [oracle.py_kmer_string(int(x), 17) for x in ref.kmers]


def test_synth_device_matches_numpy_and_oracle(gpu):
    import ctypes as C
    import torch
    from grm_b200 import synth
    from grm_b200.builder import KmerMatrixBuilder
    cfg = synth.SynthConfig(seed=synth.MASTER_SEED + 1, core_len=30_000, island_len=500, n_islands=40, n_contigs=7)
    ids = list(range(6))
    lay, total, spans = synth.build_layout(cfg, ids)
    buf = torch.empty(total, dtype=torch.uint8, device="cuda")
    with KmerMatrixBuilder(k=31, keep_singletons=False) as b:
        b._check(b._lib.grmkm_synth_fasta_device(b._ctx, C.c_void_p(lay.ctypes.data), lay.nbytes,
                                                 C.c_void_p(buf.data_ptr()), total))
        host = buf.cpu().numpy()
        texts = []
        for g, (off, ln) in zip(ids, spans):
            ref = synth.genome_fasta(cfg, g)
            assert host[off:off + ln].tobytes() == ref, f"genome {g} differs"
            texts.append(ref)
        # device-resident inputs, no host copy
        for row, (off, ln) in enumerate(spans):
            b.add_genome_device(row, buf.data_ptr() + off, ln)
        b.build()
        assert b.stats["h2d_bytes"] == 0
        ref = oracle.build([[(t, 0)] for t in texts], 31, 1, False)
        assert np.array_equal(b.kmers(), ref.kmers)
        assert np.array_equal(b.matrix(), ref.matrix)
        assert b.stats["n_bases"] == synth.n_bases_of(cfg, ids)


def test_rebuild_reuses_context(gpu):
    from grm_b200.builder import KmerMatrixBuilder
    rng = np.random.default_rng(9)
    with KmerMatrixBuilder(k=15, keep_singletons=True) as b:
        for it in range(3):
            genomes = [[inputs.fasta(rng, max_len=2000 * (it + 1))] for _ in range(3)]
            b.reset()
            for row, files in enumerate(genomes):
                b.add_genome_bytes(row, files[0])
            b.build()
            ref = oracle.build([[(f, 0) for f in files] for files in genomes], 15, 1, True)
            assert np.array_equal(b.kmers(), ref.kmers) and np.array_equal(b.matrix(), ref.matrix)


def test_pipelined_host_batches(gpu, monkeypatch):
    """Host inputs are staged in batches whose H2D copy overlaps the previous batch's kernels; a tiny batch
    size forces many batches (and both staging halves to be reused) on a small input."""
    monkeypatch.setenv("GRMKM_BATCH_BYTES", "3000")
    rng = np.random.default_rng(41)
    shared = [inputs.rand_seq(rng, 4000), inputs.rand_seq(rng, 900)]
    genomes = [[inputs.fasta(rng, n_records=3, shared=shared, max_len=2500), inputs.fasta(rng, shared=shared, max_len=700)]
               for _ in range(23)]
    genomes[5] = [b""]
    genomes[9] = [inputs.fasta(rng, n_records=6, min_len=3000, max_len=9000)]         # larger than a batch
    st = check(genomes, 31, keep_singletons=True)
    assert st["h2d_bytes"] == sum(len(f) for g in genomes for f in g)
    check(genomes, 15, keep_singletons=False)
    monkeypatch.setenv("GRMKM_EXACT_OFFSETS", "1")
    check(genomes, 21, keep_singletons=True)                                        # single-batch fallback path
    monkeypatch.delenv("GRMKM_EXACT_OFFSETS")
    fq = [[inputs.fastq(rng, shared[0], n_reads=120, read_len=70)] for _ in range(9)]
    check(fq, 21, min_abundance=2, keep_singletons=True, kind=1)


def test_result_host_is_the_same_result(gpu):
    from grm_b200.builder import KmerMatrixBuilder
    rng = np.random.default_rng(31)
    shared = [inputs.rand_seq(rng, 3000)]
    with KmerMatrixBuilder(k=21, keep_singletons=True) as b:
        for n_gen in (70, 3):                       # the pinned buffer is reused (and re-sized) across builds
            b.reset()
            for row in range(n_gen):
                b.add_genome_bytes(row, inputs.fasta(rng, shared=shared, max_len=900))
            b.build()
            km, mat = b.result_host()
            assert km.dtype == np.uint64 and mat.shape == (b.dims[1], b.dims[0])
            assert np.array_equal(km, b.kmers()) and np.array_equal(mat, b.matrix())
        b.reset()
        b.set_genome_count(2)
        b.build()                                    # no input at all
        km, mat = b.result_host()
        assert km.size == 0 and mat.shape == (1, 0)


def test_errors(gpu):
    from grm_b200.builder import KmerMatrixBuilder, GrmkmError
    with pytest.raises(GrmkmError) as e:
        KmerMatrixBuilder(k=33)
    assert e.value.code == -2
    with KmerMatrixBuilder(k=5) as b:
        with pytest.raises(GrmkmError):
            b.dims
        with pytest.raises(GrmkmError) as e2:
            b.add_genome_files(0, ["/nonexistent/file.fna"])
        assert e2.value.code == -5


@pytest.mark.parametrize("world,G,keep", [(2, 130, False), (4, 300, True), (3, 70, False), (8, 1000, False)])
def test_partial_merge_emulated_ranks(gpu, world, G, keep):
    """The CUDA partial/export/merge entry points, with the all-to-all emulated by tensor slicing:
    P contexts on one GPU, one after the other (never concurrently)."""
    _emulated_ranks(world, G, keep)


@pytest.mark.parametrize("world,G,merge_bits", [(3, 200, 14), (5, 330, 13), (6, 400, 16), (7, 460, 12), (3, 200, 6)])
def test_owner_slice_on_a_finer_merge_grid(gpu, monkeypatch, world, G, merge_bits):
    """Owner ranges are cut on the grid of the partial builds (floor(B r / P) of 2^bits buckets); the owner-side merge
    sizes its own grid from what it received.  With a world size that is not a power of two the two grids' boundaries
    differ unless the merge derives its slice from the owners' grid: forced here with a merge grid much finer (and, last
    case, coarser) than the owners'."""
    monkeypatch.setenv("GRMKM_MERGE_BITS", str(merge_bits))
    _emulated_ranks(world, G, False)


def _emulated_ranks(world, G, keep):
    import torch
    from grm_b200.builder import KmerMatrixBuilder
    from grm_b200.distributed import CudaEngine, row_partition, words_per_rank
    rng = np.random.default_rng(G)
    shared = [inputs.rand_seq(rng, 2000), inputs.rand_seq(rng, 500)]
    genomes = [inputs.fasta(rng, n_records=2, max_len=300, shared=shared) for _ in range(G)]
    parts, sw = row_partition(G, world), words_per_rank(G, world)
    engines, sends, counts = [], [], []
    for r in range(world):
        b = KmerMatrixBuilder(k=19, keep_singletons=keep)
        b.set_genome_count(len(parts[r]))
        for i, g in enumerate(parts[r]):
            b.add_genome_bytes(i, genomes[g])
        e = CudaEngine(b)
        engines.append(e)
    bits = max(e.plan_bucket_bits() for e in engines)
    for r, e in enumerate(engines):
        e.set_bucket_bits(bits)
        c, s = e.build_partial(world, sw[r])
        counts.append(c); sends.append(s)
    slices_k, slices_m = [], []
    for dst in range(world):
        chunks, src_counts = [], []
        for src in range(world):
            width = 1 + sw[src]
            off = sum(counts[src][:dst]) * width
            chunks.append(sends[src][off: off + counts[src][dst] * width])
            src_counts.append(counts[src][dst])
        recv = torch.cat(chunks) if chunks else torch.empty(0, dtype=torch.int64, device="cuda")
        engines[dst].merge(recv, world, dst, src_counts, sw, G)
        k_, m_ = engines[dst].result()
        slices_k.append(k_); slices_m.append(m_)
    # owner slices concatenated in rank order = the one-GPU column order (ascending hash), byte for byte
    allk = np.concatenate(slices_k); allm = np.concatenate(slices_m, axis=1)
    ref = oracle.build([[(g, 0)] for g in genomes], 19, 1, keep)
    assert np.array_equal(allk, ref.kmers)
    assert np.array_equal(allm, ref.matrix)
    for e in engines:
        e.b.close()


@pytest.mark.parametrize("world,G,keep", [(2, 130, True), (3, 200, False), (8, 1000, False)])
def test_partial_export_into_peer_buffers(gpu, world, G, keep):
    """grmkm_export_partials_peers (the export fused with the all-to-all: every owner's slice is stored straight into
    that owner's receive buffer at the offset the counts assign) with the P receive buffers as local tensors."""
    import torch
    from grm_b200.builder import KmerMatrixBuilder
    from grm_b200.distributed import CudaEngine, row_partition, words_per_rank
    rng = np.random.default_rng(1000 + G)
    shared = [inputs.rand_seq(rng, 3000), inputs.rand_seq(rng, 700)]
    genomes = [inputs.fasta(rng, n_records=2, max_len=400, shared=shared) for _ in range(G)]
    parts, sw = row_partition(G, world), words_per_rank(G, world)
    engines = []
    for r in range(world):
        b = KmerMatrixBuilder(k=21, keep_singletons=keep)
        b.set_genome_count(len(parts[r]))
        b.add_genomes(list(range(len(parts[r]))), [genomes[g] for g in parts[r]])
        engines.append(CudaEngine(b))
    bits = max(e.plan_bucket_bits() for e in engines)
    M = []
    for e in engines:
        e.set_bucket_bits(bits)
        M.append(e.build_local(world))                     # M[s][d]
    width = [1 + w for w in sw]
    need = [sum(M[s][d] * width[s] for s in range(world)) for d in range(world)]
    recv = [torch.full((max(n, 1),), -1, dtype=torch.int64, device="cuda") for n in need]
    for r, e in enumerate(engines):
        offs = [sum(M[s][d] * width[s] for s in range(r)) for d in range(world)]
        e.export_peers(world, [t.data_ptr() for t in recv], offs)
    torch.cuda.synchronize()
    slices_k, slices_m = [], []
    for d, e in enumerate(engines):
        e.merge(recv[d][:need[d]], world, d, [M[s][d] for s in range(world)], sw, G)
        k_, m_ = e.result()
        slices_k.append(k_); slices_m.append(m_)
    ref = oracle.build([[(g, 0)] for g in genomes], 21, 1, keep)
    assert np.array_equal(np.concatenate(slices_k), ref.kmers)
    assert np.array_equal(np.concatenate(slices_m, axis=1), ref.matrix)
    for e in engines:
        e.b.close()


def test_exact_offset_fallback(gpu, monkeypatch):
    """GRMKM_EXACT_OFFSETS=1 forces the path a region overflow falls back to (count pass + exact offsets for the unit
    scatter and the expansion); results must not change."""
    rng = np.random.default_rng(21)
    shared = [inputs.rand_seq(rng, 50_000)]
    genomes = [[inputs.fasta(rng, n_records=3, min_len=20_000, max_len=40_000, shared=shared)] for _ in range(4)]
    monkeypatch.setenv("GRMKM_EXACT_OFFSETS", "1")
    check(genomes, 31, keep_singletons=True)
    check(genomes, 32, keep_singletons=False)
    fq = [[inputs.fastq(rng, shared[0], n_reads=800, read_len=90)] for _ in range(5)]
    check(fq, 21, min_abundance=2, keep_singletons=True, kind=1)


def test_single_pass_parser_chains(gpu):
    """The parse tiles (16 KiB) are resolved by look-back along per-file chains with the tickets dealt round-robin
    over the files: files of 1 .. 40 tiles, headers and sequence lines longer than several tiles, a file that is
    one header only, CRLF, and states that differ at every tile boundary."""
    rng = np.random.default_rng(4242)
    shared = [inputs.rand_seq(rng, 60000), inputs.rand_seq(rng, 9000)]
    big_header = b">" + bytes(rng.choice(np.frombuffer(b"ACGT>@ \t", dtype=np.uint8), size=70000)) + b"\n"
    one_line = b">one line\n" + shared[0] + shared[1] + b"\n"                     # 69 kB sequence line, no breaks
    genomes = [
        [inputs.fasta(rng, n_records=40, max_len=30000, shared=shared, width=60)],   # ~40 tiles
        [big_header + inputs.fasta(rng, n_records=3, max_len=3000, shared=shared)],  # header spans 5 tiles
        [one_line],
        [big_header.rstrip(b"\n")],                                                  # a header and nothing else
        [inputs.fasta(rng, n_records=12, max_len=20000, shared=shared, width=17, crlf=True)],
        [inputs.fasta(rng, n_records=2, max_len=100, shared=shared)],                # one tile
        [b""],
        [inputs.fasta(rng, n_records=25, max_len=9000, shared=shared, width=0),      # two files in one row
         inputs.fasta(rng, n_records=5, max_len=50000, shared=shared, width=251, blank=True)],
    ]
    check(genomes, 31, keep_singletons=True)
    check(genomes, 15, keep_singletons=False)


def test_single_pass_parser_fastq_chains(gpu):
    rng = np.random.default_rng(4243)
    src = inputs.rand_seq(rng, 30000)
    genomes = [
        [inputs.fastq(rng, src, n_reads=900, read_len=150)],                        # ~20 tiles
        [inputs.fastq(rng, src, n_reads=40, read_len=20000, crlf=True)],            # reads longer than a tile
        [inputs.fastq(rng, src, n_reads=3, read_len=70)],
        [inputs.fastq(rng, src, n_reads=300, read_len=250, final_nl=False)],
    ]
    check(genomes, 21, keep_singletons=True, kind=1)
    check(genomes, 21, min_abundance=2, keep_singletons=True, kind=1)


def test_add_genomes_in_one_call(gpu):
    """grmkm_add_genomes (the whole file list at once) gives the same build as one call per input, for host and
    for device-resident inputs."""
    import torch
    from grm_b200.builder import KmerMatrixBuilder
    rng = np.random.default_rng(99)
    shared = [inputs.rand_seq(rng, 3000)]
    files = [inputs.fasta(rng, n_records=4, max_len=1500, shared=shared) for _ in range(9)]
    rows = [0, 1, 1, 2, 3, 4, 4, 4, 6]                                   # pooled rows, an empty row 5
    ref = oracle.build([[(f, 0) for f, r in zip(files, rows) if r == g] for g in range(7)], 19, 1, False)
    with KmerMatrixBuilder(k=19) as b:
        b.add_genomes(rows, files)
        b.build()
        assert np.array_equal(b.kmers(), ref.kmers) and np.array_equal(b.matrix(), ref.matrix)
        b.reset()
        dev = [torch.frombuffer(bytearray(f + b"\0" * 16), dtype=torch.uint8).cuda() for f in files]
        b.add_genomes(rows, [d.data_ptr() for d in dev], [len(f) for f in files], on_device=True)
        b.build()
        assert np.array_equal(b.kmers(), ref.kmers) and np.array_equal(b.matrix(), ref.matrix)


def test_full_size_c2_workload(gpu):
    """BASELINE.json configs[1] at full size (100 synthetic 5 Mbp genomes, k = 31, singletons kept): bit-exact against the
    oracle (6 s on 16 cores), plus the properties that do not need it -- every valid window in exactly one unit, columns
    strictly ascending in hash order, padding bits clear, the same bytes from a second build and from permuted rows."""
    import ctypes as C
    import torch
    from grm_b200 import synth
    from grm_b200.builder import KmerMatrixBuilder
    cfg = synth.SynthConfig(seed=synth.MASTER_SEED + 1)
    G, k = 100, 31
    ids = list(range(G))
    lay, total, spans = synth.build_layout(cfg, ids)
    buf = torch.empty(total, dtype=torch.uint8, device="cuda")
    with KmerMatrixBuilder(k=k, keep_singletons=True) as b:
        b._check(b._lib.grmkm_synth_fasta_device(b._ctx, C.c_void_p(lay.ctypes.data), lay.nbytes,
                                                 C.c_void_p(buf.data_ptr()), total))
        ptrs = [buf.data_ptr() + off for off, _ in spans]
        lens = [ln for _, ln in spans]
        b.add_genomes(list(range(G)), ptrs, lens, on_device=True)
        b.build()
        st = b.stats
        km, mat = b.kmers(), b.matrix()
        assert st["n_bases"] == synth.n_bases_of(cfg, ids)
        assert st["n_windows"] == st["n_bases"] - (k - 1) * st["n_records"]          # ACGT only: every window is valid
        h = km * np.uint64(0x9E3779B97F4A7C15)
        assert (h[1:] > h[:-1]).all()                                                  # strictly ascending hash order
        assert mat.shape == (2, len(km)) and (mat[0] | mat[1]).all()                   # no empty column
        assert not (mat[1] & np.uint64((1 << 28) - 1)).any()                           # rows 100..127 do not exist
        # a second build of the same context, then the rows in reverse order
        b.reset(); b.add_genomes(list(range(G)), ptrs, lens, on_device=True); b.build()
        assert np.array_equal(b.kmers(), km) and np.array_equal(b.matrix(), mat)
        b.reset(); b.add_genomes([G - 1 - r for r in range(G)], ptrs, lens, on_device=True); b.build()
        km2, mat2 = b.kmers(), b.matrix()
        assert np.array_equal(km2, km)
        def rows_of(m):                                                                # [row][sampled column] presence bits
            sub = np.ascontiguousarray(m[:, ::997])
            by = sub.view(np.uint8).reshape(2, -1, 8)[:, :, ::-1]                      # most significant byte first
            return np.unpackbits(by, axis=2).transpose(0, 2, 1).reshape(128, -1)[:G]
        assert np.array_equal(rows_of(mat2), rows_of(mat)[::-1])
        # the oracle on the same bytes
        host = buf.cpu().numpy()
        ref = oracle.build([[(host[o:o + n].tobytes(), 0)] for o, n in spans], k, 1, True)
        assert st["n_bases"] == ref.n_bases and st["n_windows"] == ref.n_windows
        assert np.array_equal(km, ref.kmers) and np.array_equal(mat, ref.matrix)


@pytest.mark.parametrize("k", [15, 21, 31])
def test_c1_size_contigs_singletons_dropped(gpu, k):
    """BASELINE.json configs[0] / configs[4] shape: 20 synthetic 5 Mbp genomes through the from-contigs settings (min
    abundance 1, singleton k-mers dropped) at k = 15 / 21 / 31, full size, bit-exact against the oracle."""
    import ctypes as C
    import torch
    from grm_b200 import synth
    from grm_b200.builder import KmerMatrixBuilder
    cfg = synth.SynthConfig(seed=synth.MASTER_SEED)
    ids = list(range(20))
    lay, total, spans = synth.build_layout(cfg, ids)
    buf = torch.empty(total, dtype=torch.uint8, device="cuda")
    with KmerMatrixBuilder(k=k, keep_singletons=False) as b:
        b._check(b._lib.grmkm_synth_fasta_device(b._ctx, C.c_void_p(lay.ctypes.data), lay.nbytes,
                                                 C.c_void_p(buf.data_ptr()), total))
        b.add_genomes(ids, [buf.data_ptr() + off for off, _ in spans], [ln for _, ln in spans], on_device=True)
        b.build()
        host = buf.cpu().numpy()
        ref = oracle.build([[(host[o:o + n].tobytes(), 0)] for o, n in spans], k, 1, False)
        assert b.stats["n_windows"] == ref.n_windows
        assert np.array_equal(b.kmers(), ref.kmers) and np.array_equal(b.matrix(), ref.matrix)


def test_c4_style_read_sets(gpu):
    """BASELINE.json configs[3] shape at a size the oracle finishes in seconds: 30x read sets (150 bp, 0.5 % substitution
    errors) of 6 synthetic genomes, each one multi-megabyte FASTQ file (a long single-file look-back chain), min abundance
    2 drops the error k-mers; also min abundance 1 (the unit path on reads)."""
    from grm_b200 import synth
    cfg = synth.SynthConfig(seed=synth.MASTER_SEED + 3).scaled(0.02)          # 90 kbp core
    genomes = []
    for g in range(6):
        n_reads = 30 * len(synth.genome_sequence(cfg, g)) // 150
        genomes.append([synth.genome_reads_fastq(cfg, g, n_reads)])
    st2 = check(genomes, 31, min_abundance=2, keep_singletons=True, kind=1)
    st1 = check(genomes, 31, min_abundance=1, keep_singletons=True, kind=1)
    assert st1["n_kmers"] > 3 * st2["n_kmers"]                                # the error k-mers are most of the unfiltered set
    check(genomes, 31, min_abundance=2, keep_singletons=False, kind=1)


@pytest.mark.parametrize("G,k,keep,bucket_bits,kind,min_ab", [
    (5, 31, True, 4, 0, 1),        # table overflow: the bucket's offset is reserved after the counting sweep
    (130, 21, False, 0, 0, 1),     # three word rows: rows 1 and 2 go through the 2-D copy
    (3, 15, True, 12, 0, 1),       # far more buckets than columns: most of the look-back chain is empty buckets
    (4, 21, False, 0, 1, 2),       # reads with an abundance filter: rounds + the presence merge of their records
])
def test_ordered_emission_equals_gather_path(gpu, monkeypatch, G, k, keep, bucket_bits, kind, min_ab):
    """A final build writes its columns in place (buckets dealt by ticket, offsets by look-back over the published
    bucket counts); GRMKM_UNORDERED=1 is the chunk + gather path it replaced.  Same bytes, and both equal the oracle."""
    rng = np.random.default_rng(100 + G)
    shared = [inputs.rand_seq(rng, 60_000)]
    if kind == 0:
        genomes = [[inputs.fasta(rng, n_records=3, min_len=20_000, max_len=50_000, shared=shared, p_shared=0.6)] for _ in range(G)]
    else:
        genomes = [[inputs.fastq(rng, shared[0], n_reads=3000)] for _ in range(G)]
    kw = {"bucket_bits": bucket_bits} if bucket_bits else {}
    stats = check(genomes, k, min_abundance=min_ab, keep_singletons=keep, kind=kind, **kw)
    if bucket_bits == 4:
        assert stats["n_splits"] > 0
    km, mat, _ = gpu_build(genomes, k, min_ab, keep, kind, **kw)
    monkeypatch.setenv("GRMKM_UNORDERED", "1")
    km2, mat2, _ = gpu_build(genomes, k, min_ab, keep, kind, **kw)
    assert np.array_equal(km, km2) and np.array_equal(mat, mat2)


@pytest.mark.parametrize("G,keep", [(257, False), (300, True), (600, False)])
def test_row_blocks_for_more_than_256_genomes(gpu, monkeypatch, G, keep):
    """More than 256 genomes: the rows are built in blocks of 256 (partial columns per block) and the blocks are merged
    with one entry reference per block in the table; GRMKM_NO_ROW_BLOCKS=1 is the single-pass build it replaces.
    Same bytes, and both equal the oracle."""
    rng = np.random.default_rng(G)
    shared = [inputs.rand_seq(rng, 2500), inputs.rand_seq(rng, 600)]
    genomes = [[inputs.fasta(rng, n_records=2, max_len=350, shared=shared)] for _ in range(G)]
    genomes[G - 3] = []                                           # a row without input in the last block
    st = check(genomes, 19, keep_singletons=keep)
    assert st["n_rounds"] == (G + 255) // 256
    km, mat, _ = gpu_build(genomes, 19, 1, keep)
    monkeypatch.setenv("GRMKM_NO_ROW_BLOCKS", "1")
    km2, mat2, st2 = gpu_build(genomes, 19, 1, keep)
    assert st2["n_rounds"] == 0
    assert np.array_equal(km, km2) and np.array_equal(mat, mat2)


def test_row_blocks_in_partial_builds(gpu):
    """Two emulated ranks with more than 256 rows each: every rank merges its row blocks into partial columns again
    (hash keys, no filter) before the export; the owners' ranges are cut on the agreed grid inside the finer merge grid."""
    _emulated_ranks(2, 700, False)
    _emulated_ranks(3, 1000, True)


def test_parse_quirks_of_long_files(gpu):
    """Files of several tiles each, FASTA and FASTQ, with the quirks that change the parser state across tile borders
    (CR-LF, blank lines, a junk prefix, no final newline, a header longer than two tiles): every tile's incoming state
    and stream position come from the look-back over its file's earlier tiles."""
    rng = np.random.default_rng(99)
    shared = [inputs.rand_seq(rng, 90_000)]
    genomes = [[inputs.fasta(rng, n_records=4, min_len=30_000, max_len=70_000, shared=shared, crlf=(g == 1), blank=(g == 2),
                             junk_prefix=(g == 3), final_nl=(g != 4))] for g in range(6)]
    genomes[5] = [b">" + b"h" * 40_000 + b"\n" + inputs.rand_seq(rng, 50_000) + b"\n"]       # a header longer than two tiles
    check(genomes, 31, keep_singletons=True)
    check(genomes, 15, keep_singletons=False)
    fq = [[inputs.fastq(rng, shared[0], n_reads=1500, read_len=100, crlf=(g == 1), final_nl=(g != 2))] for g in range(4)]
    check(fq, 21, min_abundance=1, keep_singletons=True, kind=1)
    check(fq, 21, min_abundance=2, keep_singletons=True, kind=1)
