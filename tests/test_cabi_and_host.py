"""CPU tier: the C-ABI library loads and exports every symbol the header declares (no compute calls),
host-side packing / validation / topology logic, input readers, statistics table, world_size-2 gloo path."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pandas as pd
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------ C-ABI surface
def test_library_exports_every_declared_symbol():
    import ctypes
    from simplyp_b200 import _cabi
    header = open(os.path.join(ROOT, "include", "simplyp_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = sorted(set(re.findall(r"\b(simplyp_[a-z0-9_]+)\s*\(", header)))
    assert declared, "no declarations found"
    lib = ctypes.CDLL(_cabi.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert sorted(_cabi.EXPORTS) == declared
    lib2 = _cabi.load()
    assert lib2.simplyp_abi_version() == 4
    assert b"sm_100a" in lib2.simplyp_version()


def test_no_cpu_fallback_without_a_device():
    """Without a CUDA device the compute entry points must fail loudly (error code / exception)."""
    from simplyp_b200 import _cabi
    lib = _cabi.load()
    if lib.simplyp_device_count() > 0:
        pytest.skip("a GPU is visible here")
    with pytest.raises(_cabi.SimplypError):
        _cabi.run_host(np.zeros((3, 4)), np.zeros((1, 40)), np.zeros((1, 1, 16)), np.array([0, 0], dtype=np.int32),
                       np.zeros(0, dtype=np.int32), _cabi.default_options())
    with pytest.raises(_cabi.SimplypError):
        from simplyp_b200.engine import Engine
        Engine()


def test_product_never_imports_the_oracle():
    for dirpath, _dirs, files in os.walk(os.path.join(ROOT, "simplyp_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f
                assert "hostemu" not in src or f.endswith((".cuh",)), f


def test_topology_levels_and_errors():
    from simplyp_b200 import _cabi
    #   0 1 -> 2 ; 2 3 -> 4
    po = np.array([0, 0, 0, 2, 2, 4], dtype=np.int32)
    pid = np.array([0, 1, 2, 3], dtype=np.int32)
    n, lv = _cabi.topology_levels(po, pid)
    assert n == 3 and list(lv) == [0, 0, 1, 0, 2]
    with pytest.raises(_cabi.SimplypError):     # a parent that comes later in run order
        _cabi.topology_levels(np.array([0, 1, 1], dtype=np.int32), np.array([1], dtype=np.int32))
    d = _cabi.make_dims(10, 5, 100, 1, 2, 4)
    assert _cabi.workspace_bytes(d, True) >= 10 * 5 * 100 * 32
    assert _cabi.workspace_bytes(d, False) < 10 * 5 * 100 * 32


# ------------------------------------------------------------------------------------------ packing / validation
def test_packing_layout_matches_header():
    from simplyp_b200 import packing as pk
    header = open(os.path.join(ROOT, "include", "simplyp_b200.h")).read()
    body = header[header.index("SIMPLYP_P_F_QUICK = 0"):header.index("SIMPLYP_NP_MEMBER = ")]
    names = re.findall(r"SIMPLYP_P_([A-Z0-9_]+)", body)
    assert len(names) == len(pk.MEMBER_FIELDS) == 40
    assert int(re.search(r"SIMPLYP_NP_MEMBER = (\d+)", header).group(1)) == pk.NP_MEMBER
    assert int(re.search(r"SIMPLYP_NP_SC = (\d+)", header).group(1)) == pk.NP_SC
    assert int(re.search(r"SIMPLYP_NOUT = (\d+)", header).group(1)) == pk.NOUT == len(pk.RAW_COLS)


def test_validation_errors_match_reference(tarland_2004_static):
    """Same exception types as reference model.py:322-328 (ValueError), :357 (AssertionError), :524 (KeyError)."""
    from simplyp_b200 import model as spm, packing as pk
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = tarland_2004_static
    bad = p_SC.copy()
    bad.loc["f_S", 1] = 0.4
    with pytest.raises(ValueError, match="Land use proportions"):
        pk.validate_land_use(bad, p["SC_list"])
    bad = p_SC.copy()
    bad.loc["f_NC_Ar", 1] = 0.1
    bad.loc["f_NC_S", 1] = 0.1
    with pytest.raises(ValueError, match="2 kinds of newly-converted land"):
        pk.validate_land_use(bad, p["SC_list"])
    p2 = p.copy()
    p2["d_maxE_spr"] = 20
    with pytest.raises(AssertionError):
        pk.check_erosion_windows(p2)
    ps = p_struc.copy()
    ps.loc[1, "Upstream_SCs"] = 7.0
    with pytest.raises(KeyError):
        pk.build_topology(ps, p["SC_list"])
    assert pk.parse_upstream("1, 2") == [1, 2] and pk.parse_upstream(3.0) == [3] and pk.parse_upstream(np.nan) == []


def test_prepare_inputs_mutates_like_reference(tarland_2004_static):
    from simplyp_b200 import model as spm
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = tarland_2004_static
    p_LU, p_SC = p_LU.copy(), p_SC.copy()
    topo, nc = spm._prepare_inputs(p_struc, p_LU, p_SC, p)
    spm._finish_mutations(p_LU, p_SC, p, topo.sc_ids)
    assert p_SC.loc["f_A", 1] == 0.5 and p_SC.loc["NC_type", 1] == "None" and nc == {1: "None"}
    assert p_LU.loc["EPC0_0", "A"] == pytest.approx(5.17) and p_LU.loc["TDPs0", "A"] == pytest.approx(5.17 * 290)
    assert p_LU.loc["Plab0", "A"] == pytest.approx(2873227.5)


def test_ensemble_packing_and_sharding(tarland_2004_static):
    from simplyp_b200 import ensemble as ens, packing as pk
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = tarland_2004_static
    s = ens.latin_hypercube(100, seed=1)
    for name, (lo, hi) in ens.TARLAND_RANGES.items():
        v = np.sort(s[name])
        assert v.min() >= lo and v.max() <= hi
        assert np.all(np.diff(np.floor((v - lo) / (hi - lo) * 100)) >= 1 - 1e-9)     # one sample per stratum
    member, sc = ens.pack_members(pk.member_vector(p, p_LU), pk.sc_matrix(p_SC, [1]), s)
    assert member.shape == (100, 40) and sc.shape == (100, 1, 16)
    assert np.array_equal(member[:, pk.MEMBER_INDEX["fc"]], s["fc"])
    assert np.array_equal(sc[:, 0, pk.SC_INDEX["TDPeff"]], s["sc:TDPeff"])
    pi, pLUi, pSCi = ens.apply_member_to_pandas(s, 7, p, p_LU, p_SC)
    assert pi["fc"] == s["fc"][7] and pLUi.loc["T_s", "A"] == s["T_s:A"][7] and pSCi.loc["TDPeff", 1] == s["sc:TDPeff"][7]
    covered = []
    for r in range(3):
        lo, hi = ens.shard_bounds(100, 3, r)
        covered += list(range(lo, hi))
    assert covered == list(range(100))


# ------------------------------------------------------------------------------------------ inputs
def _write_xlsx(path, sheets):
    """Minimal .xlsx writer laid out as a spreadsheet application saves a workbook, used to round-trip the stdlib
    reader: strings in the shared-string table (every other one as two rich-text runs), a styles part, floats under a
    number format, datetimes as day serials (origin 1899-12-30) under a custom and a builtin date format, rows
    alternating, and the styles / shared strings listed among the workbook's relationships."""
    import datetime
    import zipfile
    from xml.sax.saxutils import escape

    def col(i):
        s = ""
        i += 1
        while i:
            i, r = divmod(i - 1, 26)
            s = chr(65 + r) + s
        return s

    ns = 'xmlns="http://schemas.openxmlformats.org/spreadsheetml/2006/main"'
    rel = "http://schemas.openxmlformats.org/officeDocument/2006/relationships/"
    strings = {}
    with zipfile.ZipFile(path, "w") as z:
        z.writestr("[Content_Types].xml", '<?xml version="1.0"?><Types xmlns="http://schemas.openxmlformats.org/package/2006/content-types"><Default Extension="rels" ContentType="application/vnd.openxmlformats-package.relationships+xml"/><Default Extension="xml" ContentType="application/xml"/></Types>')
        z.writestr("_rels/.rels", '<?xml version="1.0"?><Relationships xmlns="http://schemas.openxmlformats.org/package/2006/relationships"><Relationship Id="rId1" Type="%sofficeDocument" Target="xl/workbook.xml"/></Relationships>' % rel)
        wb = ['<?xml version="1.0"?><workbook %s xmlns:r="http://schemas.openxmlformats.org/officeDocument/2006/relationships"><sheets>' % ns]
        rels = ['<?xml version="1.0"?><Relationships xmlns="http://schemas.openxmlformats.org/package/2006/relationships">']
        for k, (name, rows) in enumerate(sheets.items(), 1):
            wb.append('<sheet name="%s" sheetId="%d" r:id="rId%d"/>' % (escape(name), k, k))
            rels.append('<Relationship Id="rId%d" Type="%sworksheet" Target="worksheets/sheet%d.xml"/>' % (k, rel, k))
            xml = ['<?xml version="1.0"?><worksheet %s><sheetData>' % ns]
            for r, row in enumerate(rows, 1):
                xml.append('<row r="%d">' % r)
                for c, v in enumerate(row):
                    if v is None:
                        continue
                    ref = "%s%d" % (col(c), r)
                    if isinstance(v, str):
                        xml.append('<c r="%s" t="s"><v>%d</v></c>' % (ref, strings.setdefault(v, len(strings))))
                    elif isinstance(v, datetime.datetime):
                        days = (v - datetime.datetime(1899, 12, 30)).days
                        xml.append('<c r="%s" s="%d"><v>%d</v></c>' % (ref, 2 + r % 2, days))
                    elif isinstance(v, float):
                        xml.append('<c r="%s" s="1"><v>%r</v></c>' % (ref, v))
                    else:
                        xml.append('<c r="%s"><v>%d</v></c>' % (ref, v))
                xml.append("</row>")
            xml.append("</sheetData></worksheet>")
            z.writestr("xl/worksheets/sheet%d.xml" % k, "".join(xml))
        wb.append("</sheets></workbook>")
        n = len(sheets)
        rels.append('<Relationship Id="rId%d" Type="%sstyles" Target="styles.xml"/>' % (n + 1, rel))
        rels.append('<Relationship Id="rId%d" Type="%ssharedStrings" Target="sharedStrings.xml"/>' % (n + 2, rel))
        rels.append("</Relationships>")
        z.writestr("xl/workbook.xml", "".join(wb))
        z.writestr("xl/_rels/workbook.xml.rels", "".join(rels))
        z.writestr("xl/styles.xml", '<?xml version="1.0"?><styleSheet %s><numFmts count="1"><numFmt numFmtId="164" formatCode="dd/mm/yyyy;@"/></numFmts><cellXfs count="4"><xf numFmtId="0"/><xf numFmtId="2" applyNumberFormat="1"/><xf numFmtId="164" applyNumberFormat="1"/><xf numFmtId="14" applyNumberFormat="1"/></cellXfs></styleSheet>' % ns)
        sst = ['<?xml version="1.0"?><sst %s count="%d" uniqueCount="%d">' % (ns, len(strings), len(strings))]
        for i, text in enumerate(sorted(strings, key=strings.get)):
            if i % 2 == 0 and len(text) > 1:
                h = len(text) // 2
                sst.append('<si><r><t xml:space="preserve">%s</t></r><r><rPr><b/></rPr><t xml:space="preserve">%s</t></r></si>'
                           % (escape(text[:h]), escape(text[h:])))
            else:
                sst.append('<si><t xml:space="preserve">%s</t></si>' % escape(text))
        sst.append("</sst>")
        z.writestr("xl/sharedStrings.xml", "".join(sst))


def test_read_input_data_roundtrip(tmp_path, monkeypatch):
    """Write the Tarland set-up in the original project's layout — the parameter workbook in Current_Release/v0-2A,
    naming the met CSV and the two observation workbooks by its own Windows-style relative paths — as workbooks saved
    the way a spreadsheet application saves them (_write_xlsx), read it back with read_input_data from the workbook's
    directory, and get the same objects as the fixture loader."""
    import datetime
    import simplyp_b200 as sp
    from simplyp_b200 import _xlsx, tarland
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = tarland.load(dynamic="n")
    wb_dir = tmp_path / "Current_Release" / "v0-2A"
    wb_dir.mkdir(parents=True)

    def place(rel_path):
        path = os.path.normpath(os.path.join(str(wb_dir), rel_path.replace("\\", "/")))
        os.makedirs(os.path.dirname(path), exist_ok=True)
        return path

    z = np.load(os.path.join(tarland.DATA_DIR, "tarland_met.npz"))
    idx = pd.date_range(str(z["day0"]), periods=int(z["n"]), freq="D")
    sel = (idx >= "2003-12-01") & (idx <= "2005-01-31")
    with open(place(p_SU["metdata_fpath"]), "w") as f:
        f.write("Date,T_air,PET,Precipitation\n")
        for d, t, e, pr in zip(idx[sel], z["T_air"][sel], z["PET"][sel], z["Precipitation"][sel]):
            f.write("%s,%r,%r,%r\n" % (d.strftime("%d/%m/%Y"), float(t), float(e), float(pr)))
    o = obs[1]
    # discharge dates as date-formatted cells, chemistry dates as plain day serials
    serial = [(d - pd.Timestamp("1899-12-30")).days for d in o.index]
    q_rows = [["Date", "Q"]] + [[d.to_pydatetime(), None if np.isnan(v) else float(v)] for d, v in zip(o.index, o["Q"])]
    chem_cols = ["SRP", "SS", "TDP", "TP", "PP"]
    c_rows = [["Date"] + chem_cols] + [[s] + [None if np.isnan(o[c].iloc[i]) else float(o[c].iloc[i]) for c in chem_cols]
                                      for i, s in enumerate(serial)]
    # the original workbook's two observation paths are swapped (Qobsdata_fpath names the chemistry workbook)
    _write_xlsx(place(p_SU["chemObsData_fpath"]), {"1": q_rows})
    q_cells = _xlsx.Workbook(place(p_SU["chemObsData_fpath"])).cells("1")
    assert all(isinstance(q_cells[(r, 0)], datetime.datetime) for r in (1, 2))     # both date formats recognised
    _write_xlsx(place(p_SU["Qobsdata_fpath"]), {"1": c_rows})
    sheets = {
        "Readme": [["nothing here"]],
        "Setup": [["Param", "Description", "Value"]] + [[k, "", (v if isinstance(v, str) else float(v))] for k, v in p_SU.items()],
        "Reach_structure": [["Reach", "Upstream", "Final"], [1, None, None]],
        "LU": [["", "Param", "", "", "A", "S", "IG", "NC"]] + [["", r, "", ""] + [None if np.isnan(p_LU.loc[r, c]) else float(p_LU.loc[r, c]) for c in ["A", "S", "IG", "NC"]] for r in p_LU.index],
        "SC_reach": [["", "Param", "", "", 1]] + [["", r, "", "", float(p_SC.loc[r, 1])] for r in p_SC.index],
        "Constant": [["", "Param", "", "", "Value"]] + [["", k, "", "", float(v)] for k, v in p.items() if k != "SC_list"],
    }
    _write_xlsx(str(wb_dir / "Parameters_v0-2A_Tarland.xlsx"), sheets)
    monkeypatch.chdir(wb_dir)
    got = sp.read_input_data("Parameters_v0-2A_Tarland.xlsx")
    g_SU, g_dyn, g_p, g_LU, g_SC, g_struc, g_met, g_obs = got
    for k, v in p_SU.items():
        assert g_SU[k] == v, k
    assert g_SU["st_dt"] == "2004-01-01" and g_SU["Dynamic_EPC0"] == "n" and g_struc.shape == (1, 2)
    for k in p.index:
        if k != "SC_list":
            assert float(g_p[k]) == float(p[k]), k
    assert list(g_p["SC_list"]) == [1]
    assert np.allclose(g_LU.loc[p_LU.index, ["A", "S", "IG", "NC"]].to_numpy(float), p_LU.to_numpy(float), equal_nan=True)
    assert np.array_equal(g_SC.loc[p_SC.index, 1].to_numpy(float), p_SC[1].to_numpy(float))
    assert len(g_met) == 366 and np.array_equal(g_met["P"].to_numpy(), met["P"].to_numpy())
    assert np.array_equal(g_met["D_snow_end"].to_numpy(), met["D_snow_end"].to_numpy())
    assert list(g_obs[1].columns) == list(o.columns) and g_obs[1].index.equals(o.index)
    for c in o.columns:
        assert np.array_equal(g_obs[1][c].to_numpy(), o[c].to_numpy(), equal_nan=True), c


def test_snow_module_vs_oracle_and_golden(golden_dir):
    import simplyp_b200 as sp
    from oracle import simplyp_oracle as orc
    from simplyp_b200 import tarland
    raw = tarland.load_met("1981-01-01", "2010-12-31", inc_snowmelt=False).rename(columns={"P": "Precipitation"})
    out = sp.snow_hydrol_inputs(3.0, 2.74, raw)
    P, D_end, melt = orc.snow_hydrol_inputs(3.0, 2.74, raw["Precipitation"].to_numpy(), raw["T_air"].to_numpy())
    assert np.array_equal(out["P"].to_numpy(), P) and np.array_equal(out["D_snow_end"].to_numpy(), D_end)
    assert list(out.columns[-6:]) == ["P_snow", "P_rain", "P_melt", "D_snow_start", "D_snow_end", "P"]
    assert "P" not in raw.columns      # the input frame is not modified


def test_daily_pet_matches_thornthwaite_by_hand():
    import simplyp_b200 as sp
    from simplyp_b200 import inputs
    idx = pd.date_range("2003-01-01", "2004-12-31", freq="D")
    t = 8 + 8 * np.sin(2 * np.pi * (idx.dayofyear.to_numpy() - 110) / 365.25)
    met = pd.DataFrame({"T_air": t}, index=idx)
    out = sp.daily_PET(57.1, met)
    assert "PET" in out.columns and out["PET"].notnull().all() and len(out) == len(met)
    lat = inputs.deg2rad(57.1)
    tm = met["T_air"].groupby([idx.year, idx.month]).mean()
    pet_2004 = inputs.annual_thornthwaite(tm.loc[2004].to_numpy(), inputs.monthly_mean_daylight_hours(lat, 2004), 2004)
    assert out.loc["2004-07-16", "PET"] == pytest.approx(pet_2004[6] / 31)       # monthly value sits on the 16th
    assert out.loc["2004-08-01", "PET"] == pytest.approx(
        pet_2004[6] / 31 + (pet_2004[7] / 31 - pet_2004[6] / 31) * 16 / 31)       # linear in between
    with pytest.raises(ValueError):
        sp.daily_PET(57.1, met.iloc[:400])                                         # incomplete calendar year
    # daylight helper against the closed form at the equinox (about 12 h everywhere)
    assert inputs.daylight_hours(inputs.sunset_hour_angle(lat, inputs.sol_dec(81))) == pytest.approx(12.0, abs=0.2)


# ------------------------------------------------------------------------------------------ statistics / post-processing
def test_goodness_of_fit_table_vs_reference(golden_dir):
    import simplyp_b200 as sp
    from simplyp_b200 import tarland
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = tarland.load(dynamic="y")
    z = np.load(os.path.join(golden_dir, "ref_tarland2004.npz"))
    gof = json.load(open(os.path.join(golden_dir, "ref_gof.json")))
    for key in ("dyny_tight", "dynn_reftol"):
        R = pd.DataFrame(z[key + "_r"], columns=list(z[key + "_r_cols"]), index=met.index)
        got = sp.goodness_of_fit_stats(p_SU, {1: R}, obs)
        assert list(got.columns) == gof[key]["columns"] and list(got.index) == gof[key]["index"]
        assert np.allclose(got.to_numpy(float), np.array(gof[key]["values"]), rtol=1e-9, atol=1e-12)
    # the shipped GoF_stats.csv (reference tolerance, older SciPy): agreement to the solver noise
    s = np.load(os.path.join(golden_dir, "shipped_golden.npz"))
    R = pd.DataFrame(z["dyny_reftol_r"], columns=list(z["dyny_reftol_r_cols"]), index=met.index)
    got = sp.goodness_of_fit_stats(p_SU, {1: R}, obs)
    rows = [i for i, (name, reach) in enumerate(zip(s["gof_index"], s["gof"][:, 7])) if reach == 1]
    for i in rows:
        var = str(s["gof_index"][i])
        assert got.loc[var, "N obs"] == s["gof"][i, 0]
        assert got.loc[var, "NSE"] == pytest.approx(s["gof"][i, 1], abs=2e-3)


def test_sum_to_waterbody():
    import simplyp_b200 as sp
    idx = pd.date_range("2004-01-01", periods=5)
    def frame(q, m, t, pp):
        return pd.DataFrame({"Q_cumecs": q, "Msus_kg/day": m, "TDP_kg/day": t, "PP_kg/day": pp}, index=idx)
    R = {1: frame(np.full(5, 1.0), np.full(5, 100.0), np.full(5, 2.0), np.full(5, 1.0)),
         2: frame(np.full(5, 3.0), np.full(5, 300.0), np.full(5, 2.0), np.full(5, 3.0)),
         3: frame(np.full(5, 9.0), np.full(5, 1.0), np.full(5, 1.0), np.full(5, 1.0))}
    ps = pd.DataFrame({"Upstream_SCs": [np.nan] * 3, "In_final_flux?": [1.0, 1.0, np.nan]}, index=[1, 2, 3])
    out = sp.sum_to_waterbody(ps, 3, R, 0.7)
    assert np.allclose(out["Q_cumecs"], 4.0) and np.allclose(out["SS_mgl"], 400.0 / 4.0 * 1000 / 86400)
    assert np.allclose(out["TP_kg/day"], 8.0) and np.allclose(out["SRP_mgl"], 0.7 * out["TDP_mgl"])
    ps1 = pd.DataFrame({"Upstream_SCs": [np.nan] * 3, "In_final_flux?": [1.0, np.nan, np.nan]}, index=[1, 2, 3])
    assert sp.sum_to_waterbody(ps1, 3, R, 0.7) is None
    with pytest.raises(ValueError):
        sp.sum_to_waterbody(ps, 1, R, 0.7)


# ------------------------------------------------------------------------------------------ multi-process (gloo)
def test_all_gather_of_statistics_world_size_2():
    """The N>1 path: contiguous member shards per rank, one all-gather of the per-member statistics."""
    script = r'''
import os, sys
sys.path.insert(0, %r)
import torch, torch.distributed as dist
from simplyp_b200 import ensemble as ens
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%%s" %% os.environ["PORT"], rank=int(os.environ["RANK"]), world_size=2)
M, V = 11, 2
full = torch.arange(M * V * 10, dtype=torch.float64).reshape(M, V, 10)
lo, hi = ens.shard_bounds(M, 2, dist.get_rank())
got = ens.all_gather_stats(full[lo:hi].clone(), M)
assert got.shape == full.shape and torch.equal(got, full), (got.shape, lo, hi)
# pre-allocated buffers (what bench.py holds): the producer writes into .local, gather() allocates nothing;
# ragged shards (11 = 6 + 5) are compacted, equal ones (12 = 6 + 6) come back as the buffer itself
for M2 in (11, 12):
    full2 = torch.arange(M2 * V * 10, dtype=torch.float64).reshape(M2, V, 10) + 0.5
    gb = ens.GatherBuffers(M2, (V, 10), "cpu")
    lo, hi = ens.shard_bounds(M2, 2, dist.get_rank())
    assert gb.local.shape[0] == hi - lo
    for rep in range(2):
        gb.local.copy_(full2[lo:hi] + rep)
        out = gb.gather()
        assert torch.equal(out, full2 + rep), (M2, rep)
    assert (out.data_ptr() == gb.buffer.data_ptr()) == (M2 == 12)
# the fused gather (peer memory) needs CUDA: without a device its constructor fails — on BOTH ranks together, after
# both have taken part in its handle exchange (nobody is left waiting in a collective), and there is no CPU fallback
from simplyp_b200 import _cabi
if _cabi.load().simplyp_device_count() <= 0:
    try:
        ens.PeerGather(12, (V, 10), "cuda:0")
        raise AssertionError("PeerGather must not work without a CUDA device")
    except _cabi.SimplypError:
        pass
    dist.barrier()
dist.destroy_process_group()
print("ok", dist.get_rank() if dist.is_initialized() else "")
''' % ROOT
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, "-c", script], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
    outs = [p.communicate(timeout=180)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), outs


def test_integration_md_stub_matches_the_header():
    """The ctypes structures printed in INTEGRATION.md (the binding a maintainer would paste into the reference) have
    the same fields, in the same order, as include/simplyp_b200.h and simplyp_b200/_cabi.py."""
    from simplyp_b200 import _cabi
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    block = text[text.index("class Options(C.Structure):"):text.index("_dp, _ip, _lp")]
    names = re.findall(r'\("([a-z_0-9]+)", C\.c_', block)
    assert names == [f[0] for f in _cabi.SimplypOptions._fields_]
    header = open(os.path.join(ROOT, "include", "simplyp_b200.h")).read()
    body = header[header.index("typedef struct SimplypOptions {"):header.index("} SimplypOptions;")]
    hnames = re.findall(r"^\s*(?:double|int32_t)\s+([a-z_0-9]+)", body, flags=re.M)
    assert hnames == names
