"""N2 (SURVEY.md 8f): the chunk builder against the reference's own output, `FinRag_knowledge_graph/chunks.json`,
committed as tests/golden/reference_chunks.json (inputs: tests/golden/fin_statements.json, both by scripts/make_chunk_golden.py)."""
import json
import os

import pytest

from ragfin_b200 import chunker

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def bundle():
    with open(os.path.join(GOLDEN, "fin_statements.json")) as f:
        return json.load(f)


@pytest.fixture(scope="module")
def reference_chunks():
    with open(os.path.join(GOLDEN, "reference_chunks.json")) as f:
        return {c["id"]: c for c in json.load(f)}


def test_all_sixteen_chunks_equal_the_reference_byte_for_byte(reference_chunks, bundle):
    built = chunker.build_corpus_from_bundle(bundle)
    assert len(built) == 16 == len(reference_chunks)
    for c in built:
        ref = reference_chunks[c["id"]]
        assert c["text"] == ref["text"], c["id"]
        assert c["period"] == ref["period"] and c["chunk_type"] == ref["type"]
        assert len(c["text"]) == ref["size"]
        assert c["statement_type"] == "consolidated"


def test_insertion_order_is_quarter_major_then_the_four_builders(bundle):
    built = chunker.build_corpus_from_bundle(bundle)
    want = [f"icici_q{q}_fy2024_{s}" for q in range(1, 5)
            for s in ("profitability_analysis", "balance_sheet_health", "key_ratios", "segment_performance")]
    assert [c["id"] for c in built] == want          # row ids of the collection: chunks.json is id-sorted, the insert is not
    assert all(c["primary_value"] > 0 for c in built)


def test_period_columns():
    assert chunker.period_columns("Q1_FY2024") == ("june2023", "june2022")
    assert chunker.period_columns("Q4_FY2024") == ("march2024", "march2023")
    assert chunker.period_columns("Q3_FY2023") == ("december2022", "december2021")
    assert chunker.period_columns("H1") == (None, None)


def test_missing_statements_drop_their_chunks(bundle):
    docs = list(bundle["icici_q2_2023"].values())
    assert chunker.build_chunks([d for d in docs if d.get("reportType") != "CONSOLIDATED FINANCIAL RESULTS"], "Q2_FY2024") == []
    no_bs = chunker.build_chunks([d for d in docs if "consolidatedBalanceSheet" not in d], "Q2_FY2024")
    assert [c["chunk_type"] for c in no_bs] == ["profitability_analysis", "financial_ratios", "segment_analysis"]
    no_seg = chunker.build_chunks([d for d in docs if "segmentalResults" not in d and "consolidatedSegmentalResults" not in d], "Q2_FY2024")
    assert [c["chunk_type"] for c in no_seg] == ["profitability_analysis", "balance_sheet_analysis", "financial_ratios"]


def test_directory_loader_matches_the_bundle(bundle, tmp_path):
    for quarter, docs in bundle.items():
        os.makedirs(tmp_path / quarter)
        for name, doc in docs.items():
            with open(tmp_path / quarter / name, "w") as f:
                json.dump(doc, f)
    assert chunker.build_corpus(str(tmp_path)) == chunker.build_corpus_from_bundle(bundle)
