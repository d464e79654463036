"""Regenerates tests/golden/ref_answers.npz: the unmodified reference's answers to every question the tests ask it.

Needs oracle/_ref/libracon_ref.so, the reference compiled from racon's sources (`make -C oracle REF=<racon checkout>`).
The CPU tests that compare with the reference run here against a recorder (oracle_lib.RefAnswers(Ref())) that passes
each question -- layer order, window consensus, spoa graph, MSA, edlib alignment, breaking points -- to the live
reference and keeps its answer; the GPU test's question (long-read alignments) is asked directly.  The tests then
replay the stored answers, keyed by a digest of the inputs, on machines without the reference.
"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests")); sys.path.insert(0, HERE)

if __name__ == "__main__":
    import test_abi, test_aligner, test_gpu_aligner, test_msa, test_oracle, test_real_data
    from emu_lib import EmuAligner
    from make_msa_golden import msa_groups
    from oracle_lib import REF_ANSWERS, Oracle, Ref, RefAnswers
    live = Ref(); assert live.available, "oracle/_ref/libracon_ref.so is missing"
    ref, oracle, emu = RefAnswers(live), Oracle(), EmuAligner()
    test_abi.test_layer_order_is_racons_sort(ref)
    for case, golden in [("fastq_500", 1312), ("fasta_500", 1566), ("fastq_1000", 1289)]:
        test_real_data.test_oracle_reproduces_racon_on_real_windows(oracle, ref, case, golden)
    test_oracle.test_oracle_matches_live_reference(oracle, ref)
    test_oracle.test_partial_span_layers_use_the_subgraph_path(oracle, ref)
    test_msa.test_oracle_msa_matches_live_reference(oracle, ref, msa_groups())
    test_aligner.test_restatement_matches_live_edlib(oracle, ref)
    test_aligner.test_emulated_aligner_on_long_reads_against_live_edlib(ref, emu)
    test_aligner.test_breaking_points_restatement_and_engine(oracle, ref, emu)
    test_aligner.test_banded_passes_with_guessed_and_exact_bounds(oracle, ref, emu)
    for q, t in test_gpu_aligner.unmodified_edlib_pairs():
        ref.align(q, t)
    ref.save()
    print("wrote", len(ref.store), "answers,", os.path.getsize(REF_ANSWERS), "bytes to", REF_ANSWERS)
