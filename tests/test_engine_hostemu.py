"""CPU-only tests of the host logic (Rego lowering, flattening, C-ABI plumbing, result materialisation)
through tests/_hostemu/libgk_hostemu.so -- the engine linked against a TEST-ONLY backend that runs the very
same per-object core (csrc/vm_core.h) in a CPU loop.  The GPU path is covered by test_gpu.py (`-m gpu`)."""
import ctypes
import os

import pytest

import parity_cases as P
from conftest import HOSTEMU, ROOT, golden
from gatekeeper_b200 import driver as D


@pytest.mark.parametrize("case", golden("gator_cases.json"), ids=lambda c: c["name"])
def test_gator_cases(case):
    P.case_gator(HOSTEMU, case)


def test_psp_suite():
    P.case_psp(HOSTEMU)


def test_config2_small():
    resp, want = P.case_config2(HOSTEMU, 150)
    assert len(want) > 500


def test_config2_without_namespace_cache_errors_are_autorejects():
    """namespaceSelector constraints with no cached Namespace: the error plane + autoreject results."""
    resp, want = P.case_config2(HOSTEMU, 40, start=5000, with_namespaces=False)
    assert any(w[-1] for w in want)
    assert sum(resp.err_totals) == sum(1 for w in want if w[-1])


def test_mixed_kinds():
    P.case_mixed_kinds(HOSTEMU, 150)


def test_config5_wildcards():
    P.case_config5(HOSTEMU, 150)


def test_allowedrepos_comprehension_variant():
    P.case_allowedrepos_comprehension_variant(HOSTEMU, 100)


def test_match_vectors_through_kernel_core():
    P.case_match_vectors(HOSTEMU)


def test_admission_shapes():
    P.case_admission_shapes(HOSTEMU)


def test_review_errors():
    P.case_review_errors(HOSTEMU)


def test_edge_batches():
    P.case_edge_batches(HOSTEMU)


def test_unsupported_is_an_error():
    P.case_unsupported_is_an_error_not_a_fallback(HOSTEMU)


def test_resident_batch_and_stale_program():
    from gatekeeper_b200 import workloads as W
    tm, cons = W.config1()
    drv = D.Driver(lib_path=HOSTEMU)
    for k, r in tm:
        drv.add_template(k, r)
    drv.AddConstraint(cons[0])
    blob = W.synth_objects(0, 100)
    rb = drv.upload([D.Review(object=blob.get(i)) for i in range(100)])
    a = rb.eval()
    b = rb.eval()
    assert (a.viol_bits == b.viol_bits).all() and a.totals == b.totals and len(rb) == 100 and rb.alg_bytes > 0
    drv.AddConstraint(dict(cons[0], metadata={"name": "second"}))
    with pytest.raises(D.GkError, match="older constraint set"):
        rb.eval()
    rb.free()


# ---- the product library: loads, exports the whole C ABI, and refuses to run without a GPU ---------------
def test_product_library_exports_every_declared_symbol():
    import re
    hdr = open(os.path.join(ROOT, "include", "gk_engine.h")).read()
    declared = set(re.findall(r"\b(gk_[a-z_]+)\s*\(", hdr)) - {"gk_cfg"}
    lib = ctypes.CDLL(D.LIB_PATH)
    missing = [s for s in sorted(declared) if not hasattr(lib, s)]
    assert not missing, missing
    assert set(D.EXPORTS) <= declared


def test_product_library_has_no_cpu_fallback():
    """Driver() in a child process that sees no CUDA device (CUDA_VISIBLE_DEVICES=""), so that this also runs on a GPU machine."""
    import re
    import subprocess
    import sys
    code = ("from gatekeeper_b200 import driver as D\n"
            "try:\n    D.Driver()\nexcept D.GkError as e:\n    print(e)\n"
            "else:\n    raise SystemExit('Driver() started without a CUDA device')\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert re.search("no CPU fallback|CUDA", r.stdout), r.stdout


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_mutation_fuzz(seed):
    nres, nbad = P.case_fuzz(HOSTEMU, n=500, seed=seed, start=7000 + 1000 * seed)
    assert nres > 500


@pytest.mark.parametrize("seed", [5, 6, 7])
def test_match_fuzz(seed):
    assert P.case_match_fuzz(HOSTEMU, seed=seed) > 1000


@pytest.mark.parametrize("seed", [77, 78])
def test_fuzz_other_templates(seed):
    assert P.case_fuzz_other_templates(HOSTEMU, seed=seed) > 500


def test_template_libs():
    assert P.case_template_libs(HOSTEMU) > 10


def test_more_builtins():
    assert P.case_more_builtins(HOSTEMU) > 30


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
def test_rego_fuzz(seed):
    """Random policies assembled from ~80 statement shapes x random parameters x damaged Pods: whatever loads must agree."""
    accepted, n_results, _ = P.case_rego_fuzz(HOSTEMU, n_templates=30, seed=seed)
    assert accepted >= 20 and n_results > 500


def test_enforcement_action_vectors_through_review():
    """pkg/util/enforcement_action_test.go (TestGetEnforcementAction :113-165, TestScopedActionForEP :235-385): the action a
    result is stamped with, and whether a scoped constraint is enforced at all at the caller's enforcement point."""
    from test_oracle import EA_VECTORS, SCOPED_VECTORS
    rego_src = 'package k\nviolation[{"msg": "m"}] { true }\n'
    pod = {"apiVersion": "v1", "kind": "Pod", "metadata": {"name": "p", "namespace": "default"}}
    for item, want in EA_VECTORS:
        drv = D.Driver(lib_path=HOSTEMU)
        drv.add_template("K", rego_src)
        drv.AddConstraint(dict({"apiVersion": "constraints.gatekeeper.sh/v1beta1", "kind": "K", "metadata": {"name": "k"}}, **item))
        res = drv.ReviewBatch([D.Review(object=pod)], "audit.gatekeeper.sh").results
        assert [r.enforcement_action for r in res] == [want]
    for name, ep, item, want in SCOPED_VECTORS:
        drv = D.Driver(lib_path=HOSTEMU)
        drv.add_template("K", rego_src)
        spec = dict(item["spec"], enforcementAction="scoped")
        drv.AddConstraint({"apiVersion": "constraints.gatekeeper.sh/v1beta1", "kind": "K", "metadata": {"name": "k"}, "spec": spec})
        res = drv.ReviewBatch([D.Review(object=pod)], ep).results
        if want:
            assert len(res) == 1 and res[0].enforcement_action == "scoped" and list(res[0].scoped_enforcement_actions) == want, name
        else:
            assert res == [], name      # not enforced at this point: the constraint is not even evaluated


def test_namespace_cache_add_semantics():
    """nsCache.Add (pkg/target/ns_cache.go:22-44; TestNamespaceCache, pkg/target/target_test.go:983-1153): a Namespace is cached, a
    Namespace that does not convert (spec: 3.0 -- the reference's own vector) and a non-map are ErrCachingType, another kind is
    ignored; a removed namespace is gone.  Observed through a namespaceSelector constraint."""
    from oracle import k8s
    rego_src = 'package k\nviolation[{"msg": "m"}] { true }\n'
    con = {"apiVersion": "constraints.gatekeeper.sh/v1beta1", "kind": "K", "metadata": {"name": "k"},
           "spec": {"match": {"namespaceSelector": {"matchLabels": {"ns1": "label"}}}}}
    pod = {"apiVersion": "v1", "kind": "Pod", "metadata": {"name": "p", "namespace": "my-ns1"}}
    for make in (lambda: ("oracle", k8s.Client()), lambda: ("engine", D.Driver(lib_path=HOSTEMU))):
        who, x = make()
        add = (lambda o, n: x.add_namespace(o, n)) if who == "oracle" else (lambda o, n: x.AddData("t", ["cluster", "v1", "Namespace", n], o))
        err = k8s.MatchError if who == "oracle" else D.GkError
        x.add_template("K", rego_src)
        (x.add_constraint if who == "oracle" else x.AddConstraint)(con)

        def n_results():
            if who == "oracle":
                return len(x.review(k8s.Review(obj=pod), k8s.AUDIT_EP))
            return len(x.ReviewBatch([D.Review(object=pod)], k8s.AUDIT_EP).results)
        assert n_results() == 1                      # namespace unknown: the matcher errors ("missing Namespace") -> one autoreject result
        add({"apiVersion": "v1", "kind": "Namespace", "metadata": {"name": "my-ns1", "labels": {"ns1": "label"}}}, "my-ns1")
        assert n_results() == 1                      # cached and selected: the violation
        add({"apiVersion": "v1", "kind": "Namespace", "metadata": {"name": "my-ns1", "labels": {"ns1": "other"}}}, "my-ns1")
        assert n_results() == 0                      # replaced: no longer selected
        with pytest.raises(err, match="cannot cache non-namespace type"):
            add({"apiVersion": "v1", "kind": "Namespace", "spec": 3.0}, "my-ns1")
        with pytest.raises(err, match="cannot cache non-namespace type"):
            add(3, "my-ns1")
        add({"apiVersion": "apps/v1", "kind": "Deployment", "metadata": {"name": "my-ns1", "labels": {"ns1": "label"}}}, "my-ns1")
        assert n_results() == 0                      # ignored: the cache still holds the replaced namespace
        if who == "oracle":
            x.ns_cache.pop("my-ns1")
        else:
            x.RemoveData("t", ["cluster", "v1", "Namespace", "my-ns1"])
        assert n_results() == 1                      # gone again: missing Namespace


def test_validate_constraint_vectors():
    """pkg/target/target_test.go TestValidateConstraint: 11 vectors + error-text agreement on hand-made selectors."""
    assert P.case_validate_constraint(HOSTEMU) == 8


def test_every():
    assert P.case_every(HOSTEMU) > 800


def test_cross_scope_join():
    assert P.case_cross_scope_join(HOSTEMU) > 20


def test_target_enforcement_vectors():
    P.case_target_enforcement(HOSTEMU)


def test_target_matcher_vectors():
    P.case_target_matcher(HOSTEMU)


def test_gator_test_table():
    P.case_gator_test_table(HOSTEMU)


def test_verify_suite():
    P.case_verify_suite(HOSTEMU)


def test_reviews_concurrent_with_constraint_changes():
    """Reviews and AddConstraint / RemoveConstraint from several threads at once (the webhook serves while controllers
    reconcile): a review runs against ONE compiled snapshot from flatten to rendering, a review that needs another snapshot
    waits for the ones in flight, results name their own constraint columns, snapshots pin their constraints."""
    import json
    import random
    import threading
    import time
    from gatekeeper_b200 import workloads as W
    from oracle import k8s
    tm, cons = W.config2()
    drv = D.Driver(lib_path=HOSTEMU, threads=2)
    for k, r in tm:
        drv.add_template(k, r)
    for c in cons:
        drv.AddConstraint(c)
    blob = W.synth_objects(0, 200)
    revs = [D.Review(object=json.loads(blob.get(i))) for i in range(200)]
    names = {c["kind"] + "/" + c["metadata"]["name"] for c in cons}
    stop = time.time() + 3.0
    errs, counts = [], {"rev": 0, "mut": 0}

    def reviewer():
        try:
            while time.time() < stop:
                r = drv.ReviewBatch(revs, k8s.AUDIT_EP)
                counts["rev"] += 1
                assert set(r.constraints) <= names and len(r.totals) == len(r.constraints)
                for x in r.results:
                    assert x.constraint in names
        except Exception as e:      # noqa: BLE001
            errs.append(repr(e))

    def mutator(seed):
        rnd = random.Random(seed)
        try:
            while time.time() < stop:
                c = rnd.choice(cons)
                if rnd.random() < 0.5:
                    drv.RemoveConstraint(c)
                drv.AddConstraint(c)
                counts["mut"] += 1
        except Exception as e:      # noqa: BLE001
            errs.append(repr(e))

    ts = [threading.Thread(target=reviewer) for _ in range(3)] + [threading.Thread(target=mutator, args=(i,)) for i in range(2)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errs, errs[:3]
    assert counts["rev"] >= 3 and counts["mut"] >= 10


def test_inexact_numbers_are_compared_not_skipped():
    P.case_inexact_numbers(HOSTEMU)


# ---- device ingest: the ingest kernels' per-object code (csrc/ingest_core.h) run by the test backend's CPU loops
def test_blob_config2_device_ingest():
    resp, want = P.case_blob_config2(HOSTEMU, 1500)
    assert len(want) > 10000


def test_blob_fuzz_device_ingest():
    P.case_blob_fuzz(HOSTEMU)


def test_blob_json_oddities():
    P.case_blob_json_oddities(HOSTEMU)


def test_blob_other_templates():
    P.case_blob_other_templates(HOSTEMU)


def test_blob_rego_fuzz():
    accepted, n_results, rejected, n_device = P.case_rego_fuzz(HOSTEMU, n_templates=40, n_objects=100, seed=11, via_blob=True)
    assert n_device >= accepted // 2, (n_device, accepted)


def test_doc_pins():
    assert P.case_doc_pins(HOSTEMU) == 5


def test_wildcard_vectors_through_kernel_core():
    P.case_wildcard_vectors_through_kernel(HOSTEMU)


def test_aggregate_limits_fail_the_mutation_not_later_reviews():
    """Round-1 advisor finding: limits only the JOINT constraint set can hit (250 iteration scopes here) used to surface at the next
    review and break every review from then on.  Now the AddConstraint that crosses the limit fails, and reviews keep working."""
    rego = """package manyfields
violation[{"msg": "x"}] { v := input.review.object.spec[input.parameters.field][_]; v == "bad" }
"""
    drv = D.Driver(lib_path=HOSTEMU)
    drv.add_template("ManyFields", rego)
    ok = 0
    failed = None
    for i in range(300):
        try:
            drv.AddConstraint({"kind": "ManyFields", "metadata": {"name": "c%d" % i}, "spec": {"parameters": {"field": "f%d" % i}}})
            ok += 1
        except D.GkError as e:
            failed = str(e)
            break
    assert failed is not None and "rego_unsupported" in failed and 200 <= ok < 300, (ok, failed)
    resp = drv.ReviewBatch([D.Review(object={"apiVersion": "v1", "kind": "X", "metadata": {"name": "o"}, "spec": {"f3": ["bad"], "f7": ["ok"]}})], "audit.gatekeeper.sh")
    assert [r.constraint for r in resp.results] == ["ManyFields/c3"]
    assert len(drv.constraints()) == ok


def test_expansion_templates_through_the_batch():
    assert P.case_expansion(HOSTEMU) >= 6


def test_referential_constraints_data_inventory():
    assert P.case_referential(HOSTEMU) > 40


def test_audit_counts_single_result_pairs_and_evaluates_only_list_candidates():
    got = P.case_audit_lazy(HOSTEMU)
    assert got["pairsEvaluated"] < got["results"]


def test_pages_of_wide_objects_shrink_the_tile():
    assert P.case_wide_objects(HOSTEMU, pods=24, containers=60) > 100


def test_audit_concurrent_with_reviews():
    P.case_audit_concurrent_with_reviews(HOSTEMU)


@pytest.mark.parametrize("config", [2, 4, 5])
def test_generated_kernel_text_matches_the_interpreted_netlist(config):
    """spec_codegen.cpp: the CUDA C++ text generated for the constraint set, compiled for the host, object by object against the
    interpreter -- decision and ambiguity netlists, pages with objects too wide for the mask registers."""
    assert P.case_spec_kernel(HOSTEMU, 1500, config=config) > 100


@pytest.mark.parametrize("config", [2, 4, 5])
def test_generated_kernel_text_compiles_with_nvrtc_for_sm100a(config, tmp_path, monkeypatch):
    """The text NVRTC gets on the GPU box (kernels.cu: spec_compile, same options) must compile here too -- NVRTC needs no
    device -- and the spec.match blocks must be the written-out form (no block left on the generic gk_match())."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("spec_nvrtc", os.path.join(ROOT, "tools", "spec_nvrtc.py"))
    tool = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tool)
    from gatekeeper_b200 import driver as D, workloads as W
    out = tmp_path / "spec.cu"
    monkeypatch.setenv("GK_SPEC_DUMP", str(out))
    monkeypatch.setenv("GK_SPEC_CHECK", "1")
    tm, cons = {2: W.config2, 4: W.config4, 5: W.config5}[config]()
    drv = D.Driver(lib_path=HOSTEMU)
    for k, r in tm:
        drv.add_template(k, r)
    for c in cons:
        drv.AddConstraint(c)
    for ns in W.synth_namespaces():
        drv.AddData("admission.k8s.gatekeeper.sh", ["cluster", "v1", "Namespace", ns["metadata"]["name"]], ns)
    drv.ReviewBlob(W.synth_objects(7, 300, mode=1 if config == 4 else 0), with_results=False)
    drv.close()
    text = out.read_bytes()
    assert b"GK_SPEC_FN int gk_spec_mrow_" in text and b"return gk_match(B, pool, cbytes, M" not in text
    try:
        cubin, log, _ = tool.nvrtc_compile(text)
    except RuntimeError as e:
        if "libnvrtc not found" in str(e):
            pytest.skip("no NVRTC in this container")
        raise
    assert len(cubin) > 10000 and b"gk_spec_kernel" in cubin
    # static size of the kernel (a regression guard, not a timing): the text of config 2 was 8104 SASS instructions with the match
    # blocks on the shared gk_match() and compiler-unrolled range loops, 4090 written out (tools/spec_nvrtc.py)
    import shutil
    if config == 2 and shutil.which("cuobjdump") and shutil.which("nvdisasm"):
        cb = tmp_path / "spec.cubin"
        cb.write_bytes(cubin)
        usage, total, region = tool.static_report(str(cb), str(out))
        assert total < 5000, (total, dict(region))


def test_written_out_match_blocks_on_long_and_non_ascii_patterns(monkeypatch):
    """emit_match (spec_codegen.cpp) inlines the bytes of a wildcard pattern up to 24 bytes and calls the shared gk_wild() above that:
    both sides of the limit, bytes >= 0x80, and the generated text checked object by object against the interpreter and the oracle."""
    monkeypatch.setenv("GK_SPEC_CHECK", "1")
    extra = ["n\u00e4mespace-\u00fc", "team-\u65e5\u672c", "x" * 24, "y" * 25, "a-namespace-name-of-more-than-twenty-four-bytes"]
    for seed in (41, 42):
        assert P.case_match_fuzz(HOSTEMU, n_constraints=40, n_objects=300, seed=seed, extra_names=extra) > 0


def test_audit_expands_generators_like_the_audit_loop():
    got = P.case_audit_expansion(HOSTEMU)
    assert got["results"] > 50
