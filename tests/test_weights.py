"""Weight export (SURVEY §8 a12, f4): state_dict / `.pth.tar` / TorchScript `.pt` -> the flat file libuahn.so reads."""
import collections
import json
import os
import struct

import numpy as np
import pytest
import torch

from cuahn_vio_b200 import synthetic as S, weights
from oracle import uahn_oracle as O

REFERENCE_GRAPHS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_graphs.json")


def test_traced_stand_in_matches_the_record_of_the_reference_traces():
    """oracle.uahn_oracle.trace stands in for the reference's `.pt` files in the tests below and in
    test_gpu_bench_parity.py: for every graph recorded from the reference's own traces (tests/golden/reference_graphs.json)
    it must show the recorded op-kind counts and number of inputs, and hold the reference's state_dict names and shapes
    in the reference's order."""
    rec = json.load(open(REFERENCE_GRAPHS))
    sd = S.synthetic_state_dict(0)
    for name, want in rec["graphs"].items():
        traced = O.trace(sd, name.removesuffix("_showError"), name.endswith("_showError"))
        cnt = collections.Counter(n.kind() for n in traced.inlined_graph.nodes())
        assert {k: cnt[k] for k in want["ops"]} == want["ops"], name
        assert len(list(traced.graph.inputs())) - 1 == want["inputs"], name
        assert [[k, list(v.shape)] for k, v in traced.state_dict().items()] == rec["state_dict"], name


def read_flat(path):
    """Parse the flat file back: (ordered [(name, array)], raw bytes)."""
    raw = open(path, "rb").read()
    assert raw[:8] == b"UAHNWTS1"
    (count,) = struct.unpack_from("<I", raw, 8)
    pos, out = 12, []
    for _ in range(count):
        (nl,) = struct.unpack_from("<I", raw, pos); pos += 4
        name = raw[pos:pos + nl].decode(); pos += nl
        (nd,) = struct.unpack_from("<I", raw, pos); pos += 4
        dims = struct.unpack_from(f"<{nd}I", raw, pos); pos += 4 * nd
        n = int(np.prod(dims))
        out.append((name, np.frombuffer(raw, "<f4", n, pos).reshape(dims))); pos += 4 * n
    assert pos == len(raw)
    return out, raw


def test_state_dict_round_trip(tmp_path):
    sd = S.synthetic_state_dict(0)
    p = str(tmp_path / "w.bin")
    weights.export_state_dict(sd, p)
    tensors, _ = read_flat(p)
    assert [n for n, _ in tensors] == list(S.state_dict_schema())
    for n, a in tensors:
        assert np.array_equal(a, sd[n].numpy())
    # the reference's checkpoint format: torch.load(...)['state_dict'] (trace_model.py:14, model_to_trace.py:344)
    ck = str(tmp_path / "UAHN_fcdrop05_16.pth.tar")
    torch.save({"state_dict": sd, "epoch": 3}, ck)
    p2 = str(tmp_path / "w2.bin")
    weights.export_checkpoint(ck, p2)
    assert open(p, "rb").read() == open(p2, "rb").read()
    with pytest.raises(KeyError):
        weights.export_state_dict({k: v for k, v in sd.items() if "block_4_6" not in k}, p2)


def test_torchscript_export_is_the_state_dict_export(tmp_path):
    """A `.pt` like the one the reference's trace_model.py:41-46 writes — what HomographyNet.cpp:89 loads — converts to
    exactly the bytes the export of the state_dict it was traced from gives, plus the variant / showError records."""
    pt = str(tmp_path / "traced_model_3_blocks_using_prior.pt")
    O.trace(S.synthetic_state_dict(0), "prior3").save(pt)
    p_ts, p_sd = str(tmp_path / "from_pt.bin"), str(tmp_path / "from_sd.bin")
    info = weights.export_torchscript(pt, p_ts)
    assert info == {"variant": "prior3", "show_error": False}
    weights.export_state_dict(S.synthetic_state_dict(0), p_sd)
    t_ts, raw_ts = read_flat(p_ts)
    t_sd, raw_sd = read_flat(p_sd)
    meta = [(n, a) for n, a in t_ts if n.startswith("__meta__.")]
    assert [(n, float(a[0])) for n, a in meta] == [("__meta__.variant", 1.0), ("__meta__.show_error", 0.0)]
    meta_bytes = sum(4 + len(n.encode()) + 4 + 4 + 4 for n, _ in meta)
    assert raw_ts[12 + meta_bytes:] == raw_sd[12:]           # the 54 tensors, byte for byte


def test_inspect_torchscript_rejects_other_graphs():
    class Tiny(torch.nn.Module):
        def forward(self, a, b):
            return a + b
    with pytest.raises(ValueError):
        weights.inspect_torchscript(torch.jit.trace(Tiny(), (torch.ones(1), torch.ones(1))))


def test_inspect_torchscript_identifies_every_reference_variant():
    """Every graph the two model slots of HomographyNet.cpp:81-124 can hold, traced the way trace_model.py:36-39 traces
    the reference (oracle.uahn_oracle.trace), goes through the op-count detector of export_torchscript.  The full and
    3-block graphs are tied to the reference's traces by the test above; the 2-block and 1-block graphs were never
    recorded from the reference, so for them only the stand-in is checked."""
    sd = S.synthetic_state_dict(0)
    for show in (False, True):
        for variant in ("full", "prior3", "prior2", "prior1"):
            assert weights.inspect_torchscript(O.trace(sd, variant, show)) == {"variant": variant, "show_error": show}
