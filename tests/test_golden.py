"""Known-answer vectors (tests/golden, produced by tools/gen_golden.py from exact big-int
definitions): the CPU oracle must reproduce them (CPU run) and so must the CUDA library (GPU run)."""
import json
import os

import numpy as np
import pytest

from oracle import capi

HERE = os.path.dirname(os.path.abspath(__file__))
NTT = json.load(open(os.path.join(HERE, "golden", "ntt_vectors.json")))["vectors"]
MSM = json.load(open(os.path.join(HERE, "golden", "msm_vectors.json")))["vectors"]
CID = {"bls12_381": 0, "bn254": 1, "bw6_761": 2}
SW = {"bls12_381": 4, "bn254": 4, "bw6_761": 6}       # u64 words per Fr element / scalar


def _coord_words(curve, group):
    return capi.coord_words(CID[curve], group)


def _u64(hexstr, cols):
    a = np.frombuffer(bytes.fromhex(hexstr), dtype=np.uint64)
    return a.reshape(-1, cols).copy() if a.size else np.zeros((0, cols), dtype=np.uint64)


def test_golden_files_are_reproducible(tmp_path):
    """tools/gen_golden.py, pointed at a scratch directory, regenerates the committed files byte for byte
    (the committed files themselves are only read)."""
    import importlib.util
    root = os.path.dirname(HERE)
    spec = importlib.util.spec_from_file_location("gen_golden", os.path.join(root, "tools", "gen_golden.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    gen.OUT = str(tmp_path)
    gen.main()
    for f in ("ntt_vectors.json", "msm_vectors.json", "wmap_vectors.json"):
        assert open(os.path.join(tmp_path, f)).read() == open(os.path.join(HERE, "golden", f)).read(), f


@pytest.mark.parametrize("i", range(len(NTT)))
def test_oracle_ntt_golden(i):
    v = NTT[i]
    got = capi.ntt(CID[v["curve"]], _u64(v["input"], SW[v["curve"]]), v["inverse"], v["coset"])
    assert got.tobytes().hex() == v["output"]


@pytest.mark.parametrize("i", range(len(MSM)))
def test_oracle_msm_golden(i):
    v = MSM[i]
    W = _coord_words(v["curve"], v["group"])
    xy, inf = capi.msm(CID[v["curve"]], v["group"], _u64(v["bases"], 2 * W), _u64(v["scalars"], SW[v["curve"]]),
                       np.array(v["infinity"], dtype=np.uint8))
    assert int(inf) == v["result_infinity"] and xy.tobytes().hex() == v["result"]


def test_oracle_witness_map_golden():
    """The C++ restatement of witness_map (io/oi helpers, distribute_powers) against the exact-definition fixture."""
    for v in json.load(open(os.path.join(HERE, "golden", "wmap_vectors.json")))["vectors"]:
        S = SW[v["curve"]]
        h = capi.witness_map(CID[v["curve"]], _u64(v["a"], S), _u64(v["b"], S), _u64(v["c"], S))
        assert h.tobytes().hex() == v["h"], v["curve"]


@pytest.mark.gpu
def test_gpu_ntt_golden():
    import zkmember_b200 as zkm
    zkm.init(0)
    for v in NTT:
        dom = zkm.Radix2EvaluationDomain(v["curve"], v["log_n"])
        x = _u64(v["input"], SW[v["curve"]])
        fn = {(False, False): dom.fft, (True, False): dom.ifft, (False, True): dom.coset_fft, (True, True): dom.coset_ifft}
        assert fn[(v["inverse"], v["coset"])](x).tobytes().hex() == v["output"], v["log_n"]


@pytest.mark.gpu
def test_gpu_msm_golden():
    import zkmember_b200 as zkm
    zkm.init(0)
    for v in MSM:
        W = _coord_words(v["curve"], v["group"])
        got = zkm.VariableBaseMSM.multi_scalar_mul(_u64(v["bases"], 2 * W), _u64(v["scalars"], SW[v["curve"]]), curve=v["curve"],
                                                   group=v["group"], infinity=np.array(v["infinity"], dtype=np.uint8))
        assert int(got.infinity) == v["result_infinity"] and got.xy.tobytes().hex() == v["result"], (v["curve"], v["group"], v["n"])
