"""The CPU restatement on seeded inputs that the other fixtures do not hold (oracle/make_golden.py, case 8): self,
repeated, reversed, unknown and far pairs, hop 3, min / max descriptors, the KD node generator on a PPI-shaped graph.

Every test holds the oracle to the records stored in tests/golden/vs_reference_pins.npz (written by the oracle itself,
`python oracle/make_golden.py --vs-reference-pins`), so a change of the oracle on these inputs is caught anywhere.
Where a checkout of the REAL reference exists (oracle/_ref/ or $TLC_REFERENCE_ROOT, see oracle/ref_harness.py), each
test also imports it in place and compares it live on the same inputs: as-is batch output (images, counts) and the
canonical-order stage outputs (filtration values, PD0, Pos/Neg, PD1) must agree bit for bit / to 1e-11."""
import numpy as np
import pytest

import make_golden as mg
import oracle as orc
import ref_harness as rh
from helpers import rel_err, sorted_rows

LIVE = rh.available()
PINS = np.load(mg.VS_REF_FILE)


def _inputs(key):
    """-> (edges, kappa, targets in the graph's labels, oracle graph, label -> id)"""
    gk = str(PINS[key + "__graph"])
    edges, kappa = PINS[gk + "__edges"].astype(np.int64), PINS[gk + "__kappa"]
    og, lut = mg.vs_ref_graph(edges, kappa)
    return edges, kappa, PINS[key + "__targets"], og, lut


def _check_batch(r, pi_ref, cnt_ref):
    assert r["cnt_compute"] == cnt_ref
    assert np.array_equal(pi_ref.any(axis=1), r["pi"].any(axis=1))
    assert rel_err(r["pi"], pi_ref) < 1e-11


@pytest.mark.parametrize("name,scale,hop,cont,ext", mg.VS_REF_BATCH)
def test_batch_matches_reference(name, scale, hop, cont, ext):
    key = mg.vs_ref_key("batch", name, scale, hop, cont, ext)
    edges, kappa, tg, og, lut = _inputs(key)
    r = og.run_batch(mg.vs_ref_map(lut, tg), hop=hop, flags=orc.F_NORM | (orc.F_EXTENDED if ext else 0))
    _check_batch(r, PINS[key + "__pi"], int(PINS[key + "__cnt"]))
    if LIVE:
        pi_ref, cnt_ref, _ = rh.run_batch(edges, kappa, tg, hop, ext)
        _check_batch(r, pi_ref, cnt_ref)


def test_stages_match_canonical_reference():
    edges, kappa, tg, og, lut = _inputs("stages")
    pinned = 0
    for i, (a, b) in enumerate(tg):
        if int(a) not in lut or int(b) not in lut:
            assert "stages__%d__status" % i not in PINS.files
            continue
        o = og.run_one(lut[int(a)], lut[int(b)], hop=2, flags=orc.F_NORM | orc.F_EXTENDED)
        for f in mg.VS_REF_STAGE_FIELDS:
            assert np.array_equal(np.asarray(o[f]), PINS["stages__%d__%s" % (i, f)]), (i, f)
        pinned += 1
    assert pinned >= 3
    if not LIVE:
        return
    _, _, pi = rh.run_batch(edges, kappa, tg[:1], 2, True)
    checked = 0
    for a, b in tg:
        if int(a) not in lut or int(b) not in lut:
            continue
        st = rh.run_one_stages(pi, int(a), int(b), 2)
        if st["ncomp"] != 1 or st.get("PD1") is None:
            continue
        o = og.run_one(lut[int(a)], lut[int(b)], hop=2, flags=orc.F_NORM | orc.F_EXTENDED)
        assert list(o["vert"]) == st["nodes"]
        assert np.array_equal(o["fval"], np.array([st["fval"][x] for x in st["nodes"]]))
        k = o["pkind"]
        assert np.array_equal(np.stack([o["pbirth"], o["pdeath"]], 1)[k != orc.K_ONE], np.array(st["PD0"]).reshape(-1, 2))
        assert np.array_equal(np.stack([o["pbirth"], o["pdeath"]], 1)[k == orc.K_ONE], np.array(st["PD1"]).reshape(-1, 2))
        vert = o["vert"]
        assert np.stack([vert[o["elo"]][o["pos"]], vert[o["ehi"]][o["pos"]]], 1).tolist() == [list(e) for e in st["Pos"]]
        assert np.stack([vert[o["elo"]][o["neg"]], vert[o["ehi"]][o["neg"]]], 1).tolist() == [list(e) for e in st["Neg"]]
        checked += 1
    assert checked >= 3


def test_kd_generator_asis_vs_oracle():
    """SURVEY.md row A9: Knowledge_Distillation/data_utils_NC.compute_persistence_image (filt='ricci', mode='PI')
    imported AS-IS (oracle/ref_harness.load_kd) on a PPI-shaped graph vs the oracle's node mode + KD flags."""
    edges, kappa, nodes, og, lut = _inputs("kd")
    fl = orc.F_NORM | orc.F_EXTENDED | orc.F_KEEP_ZERO | orc.F_NORM_EPS
    for i, u_old in enumerate(nodes):
        for hop in (1, 2):
            o = og.run_one(lut[int(u_old)], lut[int(u_old)], hop=hop, mode=orc.MODE_NODE, flags=fl)
            for f in mg.VS_REF_KD_FIELDS:
                want = PINS["kd__%d_%d__%s" % (i, hop, f)]
                if f == "img":
                    assert rel_err(o[f], want) < 1e-10, (i, hop)
                else:
                    assert np.array_equal(np.asarray(o[f]), want), (i, hop, f)
    if not LIVE:
        return
    g = rh.build_nx_graph(edges)
    ricci = rh.ricci_list(edges, [float(k) for k in kappa])
    for u_old in nodes:
        for hop in (1, 2):
            r = rh.kd_run_node(g, ricci, int(u_old), hop)
            o = og.run_one(lut[int(u_old)], lut[int(u_old)], hop=hop, mode=orc.MODE_NODE, flags=fl)
            if r is None:
                assert o["status"] == 2
                continue
            newid = np.array([lut[int(x)] for x in r["old_label"]])
            order = np.argsort(newid)
            assert np.array_equal(newid[order], o["vert"])
            assert np.array_equal(r["filt"][order], o["fval"])
            up, one = o["pkind"] == 0, o["pkind"] == 4
            assert np.array_equal(sorted_rows(r["ord0"]), sorted_rows(np.stack([o["pbirth"][up], o["pdeath"][up]], 1)))
            assert np.array_equal(sorted_rows(r["ext1"]), sorted_rows(np.stack([o["pbirth"][one], o["pdeath"][one]], 1)))
            assert rel_err(r["pi"], o["img"]) < 1e-10


@pytest.mark.parametrize("hop,descriptor,ext", mg.VS_REF_EDGE)
def test_edge_cases_match_reference(hop, descriptor, ext):
    """targets the other fixtures do not hold: self pairs (u, u), repeated targets, reversed pairs, unknown labels,
    far-apart pairs; hop 3; min / max descriptors with the loops -- the oracle vs its record and, where a checkout
    exists, vs the as-is reference batch call."""
    edges, kappa, tg, og, lut = _inputs("edge")
    r = og.run_batch(mg.vs_ref_map(lut, tg), hop=hop, descriptor=descriptor, flags=orc.F_NORM | (orc.F_EXTENDED if ext else 0))
    key = mg.vs_ref_key("edge", hop, descriptor, ext)
    _check_batch(r, PINS[key + "__pi"], int(PINS[key + "__cnt"]))
    assert np.array_equal(r["pi"][:3], r["pi"][10:13])                       # repeated targets: identical rows
    if LIVE:
        pi_ref, cnt_ref, _ = rh.run_batch(edges, kappa, tg, hop, ext, descriptor=descriptor)
        _check_batch(r, pi_ref, cnt_ref)
