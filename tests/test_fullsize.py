"""Full-size parity: every BASELINE config at its real size, src/tgsfilter (C++ host over libtgsf_cuda)
against the UNMODIFIED reference CLI (oracle/_ref/tgsfilter) on the same FASTQ file.

Compared per run: the multiset of output records (order-independent digest, tests/cpp/fastx_digest.cpp:
the reference writes in worker-completion order with -t > 1), every `INFO:` line of stderr
(T.cpp:3071-3098, 3214-3235: all DropInfo integers, the resolved trims and adapters) and the
`var data` block + summary table of the HTML report.  Inputs come from bench.py's generator (the
workload the bench measures), written to tmpfs.  Without a reference build the host CLI is compared with
the reference's results recorded on the same inputs (tests/golden/fullsize_reference.json).

Sizes (SURVEY.md §8): C1 20 k HiFi reads, C2 200 k ONT reads (4.7 Gbases), C3 50 k ultra-long reads up
to 1 Mb with middle adapters (split and -D), C4 1 M CLR reads (9.7 Gbases), C5 200 k HiFi reads with
6-12 kb tandem repeats at -k 11 -p 5000, with and without -g/-d downsampling.  TGSF_FULLSIZE_SCALE
scales the read counts (debugging).  With TGSF_FULLSIZE_LOG=<path> the results of the runs against the
reference build are appended to that JSON file (profiles/parity_fullsize.json is such a file).
"""
import json
import os
import re
import shutil
import subprocess
import tempfile
import time

import numpy as np
import pytest

import ref_lib

pytestmark = [pytest.mark.gpu]

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST_CLI = os.path.join(ROOT, "src", "tgsfilter")
RECORDED_REFERENCE = os.path.join(ROOT, "tests", "golden", "fullsize_reference.json")
SCALE = float(os.environ.get("TGSF_FULLSIZE_SCALE", "1"))
READS = {1: 20_000, 2: 200_000, 3: 50_000, 4: 1_000_000, 5: 200_000}

RUNS = [
    ("C1_hifi", 1, ["-x", "hifi"]),
    ("C2_ont", 2, ["-x", "ont"]),
    ("C3_ultralong_split", 3, ["-x", "ont", "-M", "35", "-T", "50"]),
    ("C3_ultralong_discard", 3, ["-x", "ont", "-M", "35", "-T", "50", "-D"]),
    ("C4_clr_band_bias", 4, ["-x", "clr", "-q", "7", "-Q", "15", "-e", "150", "-b", "1"]),
    ("C5_hifi_repeat", 5, ["-x", "hifi", "-k", "11", "-p", "5000"]),
    ("C5_hifi_repeat_downsample", 5, ["-x", "hifi", "-g", "100m", "-d", "20", "-k", "11", "-p", "5000"]),
    # -p 5000 leaves ~30 % of the bases, fewer than -d 20 asks for: a smaller depth makes the length cut-off bite
    ("C5_hifi_repeat_downsample_d5", 5, ["-x", "hifi", "-g", "100m", "-d", "5", "-k", "11", "-p", "5000"]),
]


def _threads():
    return max(1, min(32, (os.cpu_count() or 2) - 1))  # the reference's own clamp (T.cpp:488-499)


def _info(stderr: str):
    return [l for l in stderr.splitlines()
            if l.startswith(("INFO", "Warning")) and "written to" not in l and "reset -t" not in l]


def _report_parts(html: str):
    m = re.search(r"var data = \{\n(.*?)\}\n</script>", html, re.S)
    assert m, "no `var data` block in the report"
    return m.group(1), re.findall(r"<td>(.*?)</td>", html)


def _data_sections(data: str):
    parts = re.split(r"((?:raw|clean)\w+): \{", data)
    return {parts[i]: parts[i + 1] for i in range(1, len(parts) - 1, 2)}


def _assert_report_data_equal(h_data: str, r_data: str):
    """Equal section by section.  The two *QualDis sections may be shorter in the reference when it ran with
    several threads: Get_qual_Dis (T.cpp:2586-2597) overwrites maxQual while it walks the per-thread histograms,
    so the plotted range ends at the highest quality seen by the LAST worker thread, not at the overall maximum
    (with -t 1, as in the small-size tests, both are the same).  The reference's x / y must then be a prefix."""
    h, r = _data_sections(h_data), _data_sections(r_data)
    assert list(h) == list(r)
    for key in r:
        if h[key] == r[key]:
            continue
        assert key.endswith("QualDis"), f"report section {key} differs"
        hx, hy = re.search(r"x: \[(.*?)\],\ny: \[(.*?)\]", h[key], re.S).groups()
        rx, ry = re.search(r"x: \[(.*?)\],\ny: \[(.*?)\]", r[key], re.S).groups()
        hx, hy, rx, ry = (v.split(",") for v in (hx, hy, rx, ry))
        assert len(rx) <= len(hx) and hx[:len(rx)] == rx and hy[:len(ry)] == ry, f"report section {key} differs"
        assert h[key].split("yTitleGap")[1] == r[key].split("yTitleGap")[1]


@pytest.fixture(scope="module")
def workdir():
    base = "/dev/shm" if os.path.isdir("/dev/shm") else None
    d = tempfile.mkdtemp(prefix="tgsf_fullsize_", dir=base)
    yield d
    shutil.rmtree(d, ignore_errors=True)


@pytest.fixture(scope="module")
def inputs(workdir):
    """config -> (path, n_reads, n_bases); the FASTQ of one config is generated once and deleted when
    the next config is asked for (tmpfs is RAM)."""
    import torch
    import bench
    from tgsfilter_b200 import synth
    state = {"cfg": None}

    def get(cfg):
        if state["cfg"] == cfg:
            return state["val"]
        if state["cfg"] is not None:
            os.unlink(state["val"][0])
        n = max(64, int(READS[cfg] * SCALE))
        dev = torch.device("cuda", 0)
        d_bases, d_quals, _, offsets, total = bench.gen_workload_gpu(cfg, n, 20261017 + cfg, dev)
        bases = d_bases[:total].cpu().numpy()
        quals = d_quals[:total].cpu().numpy()
        del d_bases, d_quals
        torch.cuda.empty_cache()
        path = os.path.join(workdir, f"in_c{cfg}.fq")
        synth.write_fastq(path, bases, quals, offsets)
        state["cfg"], state["val"] = cfg, (path, n, int(total), int(np.diff(offsets).max()))
        return state["val"]

    return get


def _run(exe, args, in_path, run_dir, extra_env=None):
    os.makedirs(run_dir, exist_ok=True)
    out = os.path.join(run_dir, "out.fq")
    env = dict(os.environ)
    env.update(extra_env or {})
    t0 = time.perf_counter()
    pr = subprocess.run([exe, "-i", in_path, "-o", out] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                        cwd=run_dir, env=env, timeout=1500)
    secs = time.perf_counter() - t0
    html = ""
    for fn in os.listdir(run_dir):
        if fn.endswith(".html"):
            with open(os.path.join(run_dir, fn), "r", errors="replace") as f:
                html = f.read()
    return pr.returncode, out, pr.stderr.decode("utf-8", "replace"), html, secs


def _digest(tool, path, run_dir):
    by_len = os.path.join(run_dir, "by_len.tsv")
    names = os.path.join(run_dir, "names.tsv")
    pr = subprocess.run([tool, path, "--by-length", by_len, "--names", names], stdout=subprocess.PIPE, check=True)
    d = json.loads(pr.stdout)
    with open(by_len) as f:
        d["by_len"] = {int(a): (int(b), c) for a, b, c in (l.split() for l in f)}
    d["names_path"] = names
    os.unlink(path)  # keep tmpfs small
    return d


def _name_diff(a_path, b_path, limit=8):
    def load(p):
        with open(p) as f:
            return set(f.read().splitlines())
    a, b = load(a_path), load(b_path)
    return sorted(a - b)[:limit], sorted(b - a)[:limit]


def _vs_recorded_reference(tag, args, path, n_reads, n_bases, max_len, workdir, tool):
    """Without a reference build: the reference CLI's results on these same inputs, recorded by this test on a B200
    (tests/golden/fullsize_reference.json, the reference side of profiles/parity_fullsize.json): record and base
    counts of its output, the order-independent digest of its records (runs without downsampling) and the number
    of its INFO lines."""
    if SCALE != 1:
        pytest.skip("the recorded reference results are for the full sizes")
    with open(RECORDED_REFERENCE) as f:
        ref = {r["run"]: r for r in json.load(f)}[tag]
    assert (n_reads, n_bases, max_len) == (ref["reads"], ref["bases"], ref["longest_read"]), "input differs from the recorded one"
    run_dir = os.path.join(workdir, tag + "_ours")
    h_rc, h_out, h_err, _, _ = _run(HOST_CLI, args, path, run_dir)
    assert h_rc == 0, h_err[-2000:]
    h_dig = _digest(tool, h_out, run_dir)
    shutil.rmtree(run_dir, ignore_errors=True)
    assert len(_info(h_err)) == ref["info_lines"]
    assert (h_dig["records"], h_dig["bases"]) == (ref["records_out"], ref["bases_out"])
    if "-g" not in args:  # with downsampling the records of the cut-off length are not defined, only their count
        assert (h_dig["sum"], h_dig["xor"]) == (ref["digest_sum"], ref["digest_xor"])


@pytest.mark.parametrize("tag,cfg,args", RUNS, ids=[r[0] for r in RUNS])
def test_fullsize_host_cli_vs_reference_cli(tag, cfg, args, workdir, inputs, cpp_tool):
    tool = cpp_tool("fastx_digest")
    path, n_reads, n_bases, max_len = inputs(cfg)
    if not ref_lib.available():
        _vs_recorded_reference(tag, args, path, n_reads, n_bases, max_len, workdir, tool)
        return
    t = _threads()
    r_rc, r_out, r_err, r_html, r_secs = _run(ref_lib.CLI, args + ["-t", str(t)], path, os.path.join(workdir, tag + "_ref"))
    assert r_rc == 0, r_err[-2000:]
    r_dig = _digest(tool, r_out, os.path.join(workdir, tag + "_ref"))
    h_rc, h_out, h_err, h_html, h_secs = _run(HOST_CLI, args, path, os.path.join(workdir, tag + "_ours"))
    assert h_rc == 0, h_err[-2000:]
    h_dig = _digest(tool, h_out, os.path.join(workdir, tag + "_ours"))

    downsample = "-g" in args
    result = {"run": tag, "config": cfg, "cli": " ".join(args), "reads": n_reads, "bases": n_bases,
              "longest_read": max_len, "reference_threads": t, "reference_seconds": round(r_secs, 2),
              "host_cli_seconds": round(h_secs, 2), "reference_gbases_per_s": round(n_bases / r_secs / 1e9, 4),
              "records_out": r_dig["records"], "bases_out": r_dig["bases"], "digest_sum": r_dig["sum"],
              "digest_xor": r_dig["xor"], "info_lines": len(_info(r_err))}
    try:
        assert _info(h_err) == _info(r_err)
        assert (h_dig["records"], h_dig["bases"]) == (r_dig["records"], r_dig["bases"])
        if not downsample:
            if (h_dig["sum"], h_dig["xor"]) != (r_dig["sum"], r_dig["xor"]):
                only_h, only_r = _name_diff(h_dig["names_path"], r_dig["names_path"])
                raise AssertionError(f"record multisets differ; only ours: {only_h}; only reference: {only_r}")
            h_data, h_cells = _report_parts(h_html)
            r_data, r_cells = _report_parts(r_html)
            assert h_cells == r_cells
            _assert_report_data_equal(h_data, r_data)
        else:
            # equal lengths at the cut-off are picked in unordered_map order by the reference (T.cpp:2297-2301):
            # every length class must agree except the shortest selected one, where only the count is defined
            assert set(h_dig["by_len"]) == set(r_dig["by_len"])
            cut = min(r_dig["by_len"])
            for ln, (cnt, hs) in r_dig["by_len"].items():
                assert h_dig["by_len"][ln][0] == cnt, f"count of length {ln}"
                if ln != cut:
                    assert h_dig["by_len"][ln][1] == hs, f"records of length {ln} differ"
            result["cut_off_length"] = cut
        result["equal"] = True
    finally:
        result.setdefault("equal", False)
        log = os.environ.get("TGSF_FULLSIZE_LOG")
        rows = []
        if log and os.path.exists(log):
            try:
                with open(log) as f:
                    rows = json.load(f)
            except Exception:
                rows = []
        rows = [r for r in rows if r.get("run") != tag] + [result]
        if log:
            with open(log, "w") as f:
                json.dump(rows, f, indent=1)
        for sub in (tag + "_ref", tag + "_ours"):
            shutil.rmtree(os.path.join(workdir, sub), ignore_errors=True)
