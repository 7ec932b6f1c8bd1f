"""CPU-only tests of the host-side logic (no kernel launches): loaders, storage, index tables, window maps."""
import os

import numpy as np
import pandas as pd
import pytest

from conftest import golden


def test_index_tables_match_reference_on_cpu():
    from digdriver_b200.sequence_model import sequence_tools as st
    z = golden("tables")
    assert st.mk_trans_idx() == list(z["trans_idx"])
    df = st.mk_mutation_context(return_df=True)
    assert list(df.MUT_TYPE) == list(z["mutctx_mut"]) and list(df.CONTEXT) == list(z["mutctx_ctx"])
    assert list(st.mk_context_sequences(2, 2)) == list(golden("scan")["columns_2_2"])
    assert len(st.mk_context_sequences(1, 1, collapse=True)) == 32
    assert st.reverse_complement("AACGN") == "NCGTT"
    assert st.seq_to_context("ANA") == "" and st.type_mutation("G", "A", collapse=True) == "C>T"


def test_get_ideal_overlaps_golden():
    from digdriver_b200.sequence_model.genic_driver_tools import get_ideal_overlaps, trip_to_str
    z = golden("overlaps")
    for i in range(8):
        for W in (10000, 1000):
            got = get_ideal_overlaps(3, z["case%d_w%d_in" % (i, W)], W)
            assert [list(t) for t in got] == z["case%d_w%d_out" % (i, W)].tolist()
    assert trip_to_str((1, 0, 10)) == "chr1:0-10"


def test_storage_roundtrip(tmp_path):
    from digdriver_b200 import storage
    st = storage.Store(str(tmp_path / "s"), "w")
    df = pd.DataFrame({"MUT_TYPE": ["A>C", "C>T"], "FREQ": [1e-6, 2.5e-7], "FLAG": [True, False]},
                      index=["chr1:0-10", "chr1:10-20"])
    st.write_table("window_10000/K/elements", df)
    got = storage.read_hdf(str(tmp_path / "s"), "window_10000/K/elements")
    assert list(got.columns) == list(df.columns) and list(got.index) == list(df.index)
    assert np.array_equal(got.FREQ.values, df.FREQ.values) and got.FLAG.dtype == bool
    s = pd.Series([3, 4], index=["AAA", "AAC"])
    st.write_table("genome_counts", s)
    assert st.read_table("genome_counts").to_dict() == {"AAA": 3, "AAC": 4}
    st.write_array("idx", np.arange(6).reshape(2, 3), dtype=np.int32)
    assert st.read_array("idx").dtype == np.int32 and st.has("idx") and not st.has("nope")
    st.set_attrs(n_up=1, n_down=np.int64(2))
    assert st.get_attrs() == {"n_up": 1, "n_down": 2}
    assert st.keys("window_10000") == ["K"]
    with pytest.raises(FileNotFoundError):
        storage.Store(str(tmp_path / "missing"), "r")


def test_read_mutation_file_schemas(tmp_path):
    from digdriver_b200.data_tools import mutation_tools as mt
    rows = [("1", 100, 101, "A", "C", "S1", "G1", "Missense", "A>C", "TAG"),
            ("1", 100, 101, "A", "C", "S1", "G1", "Missense", "A>C", "TAG"),
            ("X", 5, 6, "A", "C", "S1", ".", "Noncoding", "A>C", "TAG"),
            ("2", 7, 9, "AT", "A", "S2", "G2", "INDEL", "cds_INDEL", "."),
            ("2", 7, 9, "AT", "A", "S3", "G2", "INDEL", "cds_INDEL", ".")]
    f = tmp_path / "m.tsv"
    pd.DataFrame(rows).to_csv(f, sep="\t", header=False, index=False)
    df = mt.read_mutation_file(str(f))
    assert list(df.columns) == ['CHROM', 'START', 'END', 'REF', 'ALT', 'SAMPLE', 'GENE', 'ANNOT', 'MUT_TYPE', 'CONTEXT']
    assert df.CHROM.dtype.kind == "i" and set(df.CHROM) == {1, 2}         # sex chromosomes dropped
    assert (df.ANNOT == "INDEL").sum() == 1                               # indels unique on (..., GENE)
    assert len(mt.read_mutation_file(str(f), drop_duplicates=True)) == 2
    assert len(mt.read_mutation_file(str(f), drop_sex=False)) == 4
    pd.DataFrame([r[:6] for r in rows]).to_csv(f, sep="\t", header=False, index=False)
    assert list(mt.read_mutation_file(str(f), unique_indels=False).columns) == ['CHROM', 'START', 'END', 'REF', 'ALT', 'SAMPLE']
    wl, bl = mt.filter_hypermut_samples(df, 1, return_blacklist=True)
    assert bl == ["S1"] and set(wl.SAMPLE) == {"S2"}


def test_bed12_boundaries(tmp_path):
    from digdriver_b200.data_tools import mutation_tools as mt
    f = tmp_path / "e.bed"
    f.write_text("chr1\t100\t500\tE1\t0\t-\t100\t500\t0\t2\t50,20,\t0,380,\n"
                 "X\t1\t9\tEX\t0\t+\t1\t9\t0\t1\t8\t0\n"
                 "2\t10\t40\tE2\t0\t+\t10\t40\t0\t1\t30\t0\n")
    df = mt.bed12_boundaries(str(f))
    assert list(df.ELT) == ["E1", "E2"] and list(df.CHROM) == [1, 2]
    assert df.BLOCK_STARTS.iloc[0] == [100, 480] and df.BLOCK_ENDS.iloc[0] == [150, 500]
    blocks = mt._read_bed_blocks(str(f), bed12=True)
    assert len(blocks) == 4 and list(blocks.CHROM) == ["chr1", "chr1", "X", "2"]


def test_window_tiling_and_map():
    from digdriver_b200 import genome as G, kernels
    w = G.tile_windows([1, 2], [40123, 2000], 1000)
    assert len(w) == 40 + 1 and w[-1].tolist() == [2, 0, 1000] and w[39].tolist() == [1, 39000, 40000]
    off, wmap = kernels.build_window_map(w[:, 0], w[:, 1], 1000, 3)
    assert off.tolist() == [0, 0, 40, 41] and wmap[39] == 39 and wmap[40] == 40
    keep = np.r_[0:10, 12:41]
    off, wmap = kernels.build_window_map(w[keep, 0], w[keep, 1], 1000, 3)
    assert wmap[10] == -1 and wmap[11] == -1 and wmap[12] == 10
    assert kernels.element_max_span([0, 2, 3], [100, 25000, 7], [900, 25100, 9], 1000) == 26
    assert G.hg19_like_lengths().sum() == 3_100_000_000


def test_fasta_reader(tmp_path):
    from digdriver_b200.genome import Genome
    f = tmp_path / "g.fa"
    f.write_text(">chr1 desc\nACGT\nacgN\n>chr2\nTT\n")
    g = Genome.from_fasta(str(f))
    assert g.names == ["chr1", "chr2"] and g.fetch("chr1") == "ACGTacgN" and g.fetch("chr2", 1, 2) == "T"
    assert g.lengths.tolist() == [8, 2]


def test_qvals():
    from digdriver_b200.sequence_model.nb_model import get_q_vals
    q = get_q_vals([0.01, 0.04, 0.03, 0.5])
    np.testing.assert_allclose(q, [0.04, 0.04 * 4 / 3, 0.04 * 4 / 3, 0.5])


def test_cli_parsers_accept_the_reference_arguments():
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    mods = {}
    for name in ("DigPreprocess", "DigPretrain", "DigDriver"):
        spec = importlib.util.spec_from_file_location("cli_" + name, os.path.join(root, "scripts", name + ".py"))
        mods[name] = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mods[name])
    a = mods["DigPretrain"].parse_args("countMutations --outputFile m --mutation-file f.tsv")
    assert a.fmut == "f.tsv" and a.func.__name__ == "count_training_mutations"
    a = mods["DigPreprocess"].parse_args("preprocess_genic_model g.h5 g.fa out --window 1000")
    assert a.out_key == "cds/window_10kb" and a.window == 1000 and a.func.__name__ == "preprocess_cds_contexts"
    a = mods["DigPreprocess"].parse_args("countGenomeContext g.fa out --bed w.bed --up 2 --down 2 --n-procs 4")
    assert a.up == 2 and a.bed == "w.bed" and a.func.__name__ == "countGenomeContext"
    a = mods["DigPretrain"].parse_args("elementModel pre.h5 data.h5 KEY --n-procs 3")
    assert a.save_key == "KEY" and a.N_procs == 3
    a = mods["DigDriver"].parse_args("elementDriver m.txt model.h5 KEY --f-bed e.bed --outpfx x --outdir o --scale-type genome")
    assert a.f_bed == "e.bed" and a.scale_type == "genome" and a.max_muts_per_sample == 3e9
    a = mods["DigDriver"].parse_args("geneDriver m.txt model.h5 --outpfx x --outdir o --scale-by-mutations")
    assert a.scale_by_expectation is False
    a = mods["DigDriver"].parse_args("targetDriver m.txt model.h5 --panel MSK_341 --outpfx x --outdir o --scale-by-samples")
    assert a.panel == "MSK_341" and a.scale_by_samples and a.func.__name__ == "target_driver"
    a = mods["DigPreprocess"].parse_args("preprocess_tiled tiles.bed data.h5 g.fa 10000 TILES --n-procs 2")
    assert a.window == 10000 and a.save_key == "TILES" and a.func.__name__ == "preprocess_tiled"
    a = mods["DigPretrain"].parse_args("tiledModel pre.h5 data.h5 TILES --output_h5 out.h5")
    assert a.output_h5 == "out.h5" and a.func.__name__ == "pretrain_tiled"
    spec = importlib.util.spec_from_file_location("cli_DataExtractor", os.path.join(root, "scripts", "DataExtractor.py"))
    de = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(de)
    a = de.parse_args(["addObjectives", "d.h5", "m.txt", "--sample-filter-stdev", "2.5", "--max-muts-per-sample", "9"])
    assert a.sample_filter_stdev == 2.5 and a.max_muts_per_sample == 9 and a.cnv is False


def test_window_tiling_rule_and_tile_names():
    """extract_high_mappability's tiling (DataExtractor.py:70-77): from 0 while i + window < size; tiled-model names."""
    from digdriver_b200.data_tools import objectives
    from digdriver_b200.sequence_model.genic_driver_tools import _index_transform
    idx = objectives.tile_windows({1: 30_000, 2: 10_000, 3: 10_001}, 10_000)
    assert idx.tolist() == [[1, 0, 10_000], [1, 10_000, 20_000], [3, 0, 10_000]]      # the last partial window is dropped
    assert objectives.tile_windows({7: 100}, 30, overlap=10).tolist() == [[7, 0, 30], [7, 20, 50], [7, 40, 70], [7, 60, 90]]
    assert _index_transform("chr12:100-250") == "region_12_100_250"


def test_store_element_groups_round_trip(tmp_path):
    from digdriver_b200 import storage
    st = storage.Store(str(tmp_path / "s"), "w")
    names = ["e1", "e2", "e3"]
    L = np.arange(3 * 192, dtype=np.float64).reshape(3, 192)
    R = (np.arange(3 * 192, dtype=np.int64) * 7).reshape(3, 192)
    ov = [[(1, 0, 1000), (1, 1000, 2000)], [], [(2, 5000, 6000)]]
    st.write_element_groups("window_1000/K", names, L, R, ov)
    assert st.has("window_1000/K")
    n2, L2, R2, ov2 = storage.Store(str(tmp_path / "s"), "r").read_element_groups("window_1000/K")
    assert n2 == names and np.array_equal(L2, L) and np.array_equal(R2, R) and ov2 == ov
    n3, L3, R3, ov3 = st.read_element_groups("window_1000/K", ["e3", "e1"])
    assert n3 == ["e3", "e1"] and np.array_equal(L3, L[[2, 0]]) and ov3 == [ov[2], ov[0]]
    with pytest.raises(KeyError):
        st.read_element_groups("window_1000/K", ["nope"])


def test_fetch_sequence_and_host_helpers():
    from digdriver_b200.genome import Genome
    from digdriver_b200.sequence_model import sequence_tools as st
    from digdriver_b200.driver_model import transfer_tools as tt
    g = Genome.from_dict({"chr1": "acgtNNacgtACGT"})
    assert st.fetch_sequence(g, "chr1", 0, 4, n_up=2, n_down=2) == ("ACGTNN", 0, 6)        # START 0 -> n_up
    assert st.fetch_sequence(g, "chr1", 3, 5, n_up=1, n_down=1) == ("GTNN", 2, 6)
    assert st._parse_region_str("chr12:100-250") == ("chr12", 100, 250)
    assert tt._mle_t(3, 1, 0.5, 2.0) == max(0.5 * 2.0, (3 + 0.5 - 1) / (1 + 0.5))
    assert tt._mle_t(0, 1, 2.0, 0.1) == (0 + 2.0 - 1) / (1 + 10.0)
    assert tt._mrfold_factor(0.0, 5.0) == 1e-10 and tt._mrfold_factor(2.0, 4.0) == 0.5


def test_filter_hypermut_script(tmp_path):
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("cli_filter_hypermut", os.path.join(root, "scripts", "filter_hypermut.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    rows = []
    for i in range(30):                                            # sample H: 30 coding rows, sample L: 3
        rows.append((1, 100 + i, 101 + i, "A", "C", "H", "G%d" % i, "Missense", "A>C", "AAA"))
    for i in range(3):
        rows.append((2, 500 + i, 501 + i, "C", "T", "L", "G1", "Synonymous", "C>T", "ACA"))
    for i in range(50):                                            # non-coding rows never count
        rows.append((3, 900 + i, 901 + i, "G", "T", "L", ".", "Noncoding", "G>T", "AGA"))
    pd.DataFrame(rows).to_csv(tmp_path / "cohort.annot.txt", sep="\t", header=False, index=False)
    out = tmp_path / "out"
    mod.main("--input-dir %s --output-dir %s" % (tmp_path, out))               # reference behaviour: limit 3000
    assert len(pd.read_table(out / "cohort.no_hypermut.annot.txt", header=None)) == 83
    mod.main("--input-dir %s --output-dir %s --max-muts-per-sample 10 --honour-threshold" % (tmp_path, out))
    kept = pd.read_table(out / "cohort.no_hypermut.annot.txt", header=None)
    assert set(kept[5]) == {"L"} and len(kept) == 53


def test_nb_model_sequence_helpers(tmp_path):
    """nb_model.mutation_freq_conditional / _joint / tabix_to_dataframe (reference nb_model.py:13-77)."""
    from digdriver_b200.sequence_model import nb_model
    idx = pd.MultiIndex.from_tuples([("A>C", "AAA"), ("A>G", "AAA"), ("C>T", "ACG")])
    S_mut = pd.Series([4, 6, 9], index=idx)
    S_gen = pd.Series({"AAA": 100, "ACG": 30})
    got = nb_model.mutation_freq_conditional(S_mut, S_gen, 2)
    assert got.dtype == float and list(got.index) == list(idx)
    assert got.tolist() == [4 / (2 * 100), 6 / (2 * 100), 9 / (2 * 30)]
    assert nb_model.mutation_freq_joint(S_mut, S_gen, 2).equals(got)

    class Tbx:
        def fetch(self, chrom, start, end):
            return ["1\t5\t6\tA\tC\tS1\tMissense", "1\t9\t10\tG\tT\tS2\tNoncoding"]
    df = nb_model.tabix_to_dataframe(Tbx(), "1", 0, 100)
    assert list(df.columns) == ['CHROM', 'START', 'END', 'REF', 'ALT', 'ID', 'ANNOT'] and df.START.tolist() == [5, 9]

    class Empty:
        def fetch(self, *a):
            return []
    assert list(nb_model.tabix_to_dataframe(Empty(), "1", 0, 1).columns) == ['CHROM', 'START', 'END', 'REF', 'ALT', 'ID']


def test_nb_model_train_sequence_model_from_store(tmp_path):
    """nb_model.train_sequence_model / expected_mutations_by_context (reference nb_model.py:79-124) on a store that
    holds per-window mutation counts with (mutation, context) tuple columns."""
    from digdriver_b200 import storage
    from digdriver_b200.sequence_model import nb_model
    rows = ["chr1:0-1000", "chr1:1000-2000", "chr2:0-1000"]
    cols = pd.MultiIndex.from_tuples([("A>C", "AAA"), ("A>G", "AAA"), ("C>T", "ACG")])
    df_mut = pd.DataFrame([[1, 2, 3], [4, 0, 1], [7, 7, 7]], index=rows, columns=cols)
    df_gen = pd.DataFrame({"AAA": [100, 50, 10], "ACG": [30, 20, 5]}, index=rows)
    st = storage.Store(str(tmp_path / "m"), "w")
    st.write_table("mutation_counts", df_mut)
    st.write_table("genome_counts", df_gen)
    back = storage.Store(str(tmp_path / "m"), "r").read_table("mutation_counts")
    assert list(back.columns) == list(cols) and np.array_equal(back.values, df_mut.values)
    train = [(1, 0, 1000), (1, 1000, 2000)]
    Pr, d = nb_model.train_sequence_model(train, str(tmp_path / "m"), N=2)
    assert Pr.tolist() == [5 / (2 * 150), 2 / (2 * 150), 4 / (2 * 50)]
    assert d == {"AAA": 5 / 300 + 2 / 300, "ACG": 4 / 100}
    exp_train, exp_test = nb_model.expected_mutations_by_context(train, [(2, 0, 1000)], str(tmp_path / "m"), N=2)
    np.testing.assert_allclose(exp_train.values, [100 * d["AAA"] + 30 * d["ACG"], 50 * d["AAA"] + 20 * d["ACG"]], rtol=1e-15)
    np.testing.assert_allclose(exp_test.values, [10 * d["AAA"] + 5 * d["ACG"]], rtol=1e-15)


def test_mask_runs_round_trip():
    """Run-length form of the N mask (packed-genome cache, host_pipeline.mask_runs_of): lossless, split at chromosome
    boundaries, empty for an N-free genome."""
    from digdriver_b200.host_pipeline import mask_runs_of
    rng = np.random.default_rng(4)
    n_words = 3000
    bits = np.zeros(n_words * 32, dtype=np.uint8)
    for _ in range(40):
        a = int(rng.integers(0, n_words * 32 - 700))
        bits[a:a + int(rng.integers(1, 600))] = 1
    bits[32 * 1000 - 5:32 * 1000 + 70] = 1                 # crosses the boundary between the two chromosomes below
    words = np.packbits(bits).view(">u4").astype(np.uint32)
    runs = mask_runs_of(words.view(np.int32), np.array([0, 32_000]), n_words * 32)
    assert runs.dtype == np.int64 and runs.shape[1] == 3 and len(runs) < 400
    out = np.zeros(n_words, dtype=np.uint32)
    for first, cnt, val in runs:
        assert not np.any(out[first:first + cnt])          # disjoint
        out[first:first + cnt] = val
    assert np.array_equal(out, words)
    assert not any(f < 1000 < f + c for f, c, _ in runs)   # no run spans the chromosome boundary (word 1000)
    assert mask_runs_of(np.zeros(10, dtype=np.int32), np.array([0]), 320).shape == (0, 3)


def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs: a seeded, sorted sample of count-table rows with their window indices, whole small arrays,
    integer arrays as exact float32 and larger integers and floats as float64."""
    import torch
    import bench
    from types import SimpleNamespace
    n_win = 10_000
    c5 = torch.randint(0, 10_001, (n_win, 1024), dtype=torch.int32, generator=torch.Generator().manual_seed(0))
    di = SimpleNamespace(win_chrom=torch.zeros(n_win, dtype=torch.int32), counts5=c5, counts3=c5[:, :64].contiguous(),
                         totals5=c5.sum(0) * 1000, totals3=c5[:, :64].sum(0))
    res = {"PVAL_MUT_BURDEN": torch.linspace(0, 1, 7, dtype=torch.float64), "CTX": torch.tensor([-1, 0, 63], dtype=torch.int32)}
    bench.dump_outputs(str(tmp_path / "a"), di, res)
    bench.dump_outputs(str(tmp_path / "b"), di, res)
    got = {f[:-4]: np.load(str(tmp_path / "a" / f)) for f in os.listdir(tmp_path / "a")}
    assert sorted(got) == sorted(["sample_windows", "counts5_sample", "counts3_sample", "totals5", "totals3",
                                  "PVAL_MUT_BURDEN", "CTX"])
    assert sorted(os.listdir(tmp_path / "b")) == sorted(k + ".npy" for k in got)
    for k, v in got.items():
        assert np.array_equal(v, np.load(str(tmp_path / "b" / (k + ".npy"))))
    rows = got["sample_windows"].astype(np.int64)
    assert len(rows) == bench.DUMP_WINDOWS and np.all(np.diff(rows) > 0)
    assert got["counts5_sample"].dtype == np.float32 and np.array_equal(got["counts5_sample"], c5[rows].numpy())
    assert got["totals5"].dtype == np.float64 and np.array_equal(got["totals5"], di.totals5.numpy())
    assert got["CTX"].dtype == np.float32 and got["CTX"].tolist() == [-1, 0, 63]
    assert got["PVAL_MUT_BURDEN"].dtype == np.float64 and np.array_equal(got["PVAL_MUT_BURDEN"], res["PVAL_MUT_BURDEN"].numpy())
