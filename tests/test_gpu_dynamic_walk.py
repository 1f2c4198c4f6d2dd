"""GPU parity of the multi-candidate ("dynamic") mode at the file sizes where its chain stitch runs: body, package
list and round trip against the oracle, and the walk launches against the model of test_cpu_dynamic_walk, so that
every branch the model says a case reaches is one the library actually took."""
import numpy as np
import pytest

import inputs
import oracle as O
import test_cpu_dynamic_walk as W

pytestmark = pytest.mark.gpu

SPAN_LAUNCHES = 5  # k_select_span_fast, k_sizes, k_scan_tiles, k_offsets, k_pack_span


@pytest.fixture(scope="module")
def eng():
    from adaptive_compression_b200 import engine
    engine.require_cuda()
    return engine


def test_dynamic_walk_matches_oracle_and_model(eng):
    from adaptive_compression_b200 import _lib as L
    lib = L.lib()
    bad, models = [], []
    for name, data, cands, methods, marker, pcr, M in W.case_models():
        t = eng.to_device(data)
        before = lib.ambc_launch_count()
        o = eng.compress_dynamic_device(t, cands, mask=eng.method_mask(methods), flags=L.F_PER_CHUNK_RAW if pcr else 0,
                                        marker=marker)
        launches = lib.ambc_launch_count() - before
        wbody, wpm = O.compress_body(data, cands, methods, marker, pcr)
        body = o.body.cpu().numpy().tobytes()
        if body != wbody or [tuple(p) for p in o.packages] != [tuple(p) for p in wpm]:
            bad.append((name, "body", len(body), len(wbody)))
            continue
        want_launches = M.walk_launches() + (SPAN_LAUNCHES if M.chain else 0)
        if launches != want_launches:
            bad.append((name, "launches", launches, want_launches, len(M.rounds)))
        out, status = eng.decompress_device(o.body, len(data), marker=marker)
        if status != [0, 0] or out.cpu().numpy().tobytes() != data:
            bad.append((name, "round trip", status))
        models.append((name, M))
    assert not bad, bad
    cov = W.coverage(models)
    assert W.WANT_COVERAGE <= cov, sorted(W.WANT_COVERAGE - cov)


def test_clamped_candidate_takes_the_last_bytes(eng):
    """16384 is clamped to the last 7000 bytes; no other candidate of the list can take them in one package"""
    name, data, cands, methods, marker, pcr, M = next(c for c in W.case_models() if c[0] == "clamp_16384")
    o = eng.compress_dynamic_device(eng.to_device(data), cands)
    assert o.packages[-1][1] == 7000 and M.chain[-1][0] == len(data) - 7000
    assert [tuple(p) for p in o.packages] == [tuple(p) for p in O.compress_body(data, cands)[1]]


def test_seventeen_distinct_clamped_sizes_are_rejected(eng):
    from adaptive_compression_b200 import _lib as L
    sixteen = next(c[2] for c in W.case_models() if c[0] == "sizes16")
    assert len({min(c, 8192) for c in sixteen}) == 16
    seventeen = tuple(sixteen) + (4096,)
    with pytest.raises(L.AmbcError, match="distinct candidate sizes"):
        eng.compress_dynamic_device(eng.to_device(inputs.text(100_000, 570)), seventeen)


def test_facade_default_arguments_write_the_oracle_file(tmp_path):
    """AdaptiveCompressor() selects the reference's candidate list; on a 4 MiB cascade its file is the oracle's"""
    from adaptive_compression_b200 import AdaptiveCompressor
    name, data, cands, methods, marker, pcr, M = next(c for c in W.case_models() if c[0] == "cascade_ref_4M")
    assert tuple(cands) == inputs.REF_DEFAULT_CANDIDATES and len(M.rounds) >= 60
    src, dst, back = tmp_path / "in.bin", tmp_path / "out.ambc", tmp_path / "back.bin"
    src.write_bytes(data)
    c = AdaptiveCompressor()
    c.compress(str(src), str(dst))
    want, raw, _ = O.compress_file(data, inputs.REF_DEFAULT_CANDIDATES)
    assert not raw and dst.read_bytes() == want
    c.decompress(str(dst), str(back))
    assert back.read_bytes() == data
