"""Static check on the wide product pass (no GPU): every instantiation of wide_round_kernel fits the two 128-thread blocks
per SM it is launched at, with at most a few spilled words. Reads the ptxas log `make -C jolt_b200/csrc` leaves
in-tree; skipped before a build."""
import pathlib
import re

import pytest

CSRC = pathlib.Path(__file__).resolve().parents[1] / "jolt_b200" / "csrc"


def ptxas_entries(log: pathlib.Path) -> dict:
    """mangled kernel name -> (registers, spill_store_bytes, spill_load_bytes)"""
    out, cur, spills = {}, None, (0, 0)
    for line in log.read_text().splitlines():
        m = re.search(r"Compiling entry function '([^']+)'", line)
        if m:
            cur = m.group(1)
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            spills = (int(m.group(1)), int(m.group(2)))
        m = re.search(r"Used (\d+) registers", line)
        if m and cur:
            out[cur] = (int(m.group(1)),) + spills
            cur = None
    return out


@pytest.fixture(scope="module")
def wide_log():
    log = CSRC / "wide_product.ptxas.log"
    if not log.exists():
        pytest.skip("no build in this tree yet (python -c 'import __graft_entry__ as g; g.build()')")
    return ptxas_entries(log)


def test_wide_round_kernels_fit_two_blocks_of_128_without_real_spills(wide_log):
    ents = {k: v for k, v in wide_log.items() if "wide_round_kernel" in k}
    # plain D = 5..8 x 2 orders x {eval-only, bind, 125-bit bind} x SKIP1 on/off, split-eq D = 4..8 x 2 x 3 (SKIP1 only)
    assert len(ents) == 4 * 2 * 3 * 2 + 5 * 2 * 3, sorted(ents)
    for name, (regs, st, ld) in ents.items():
        assert regs <= 255, (name, regs)  # 2 blocks x 128 threads x 255 registers fill the register file
        assert st <= 32 and ld <= 32, (name, st, ld)  # a few words, touched once per pair index next to ~30 products
    # the shapes used most, products of 5..8 tables under SKIP1 with a 125-bit challenge, do not spill at all below D = 8
    for name, (regs, st, ld) in ents.items():
        if re.search(r"wide_round_kernelILi[567]ELi[01]ELb1ELb1ELb1ELb0E", name):
            assert (st, ld) == (0, 0), (name, st, ld)
