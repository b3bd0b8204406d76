"""CPU checks of the embedding-width limit of the tensor-core candidate pass: the one exported
eligibility rule, and the workspace it sizes for rows up to 512 wide.  No compute calls."""
import ctypes

import pytest

from mclstexp_b200 import _lib, build, retrieval


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def _documented_rule(n_bank, dim, k, flags):
    return not (flags & _lib.FM_EXACT_ONLY) and dim <= 512 and k <= 896 and n_bank >= k


def test_tc_eligible_matches_documented_rule(lib):
    checked = 0
    for flags in (_lib.FM_DEFAULT, _lib.FM_EXACT_ONLY, _lib.FM_BANK_PACKED, _lib.FM_NO_SPECULATION):
        for k in (1, 192, 193, 896, 897):
            for n_bank in (k - 1, k, k + 1, 1_000_000):
                for dim in range(1, 601):
                    want = _documented_rule(n_bank, dim, k, flags)
                    got = lib.mclst_find_matches_tc_eligible(n_bank, dim, k, flags)
                    assert got == int(want), (n_bank, dim, k, flags, got)
                    checked += 1
    assert checked == 4 * 5 * 4 * 600
    for dim, want in ((256, 1), (257, 1), (511, 1), (512, 1), (513, 0)):
        assert lib.mclst_find_matches_tc_eligible(10_000, dim, 50, 0) == want, dim
        assert retrieval.tc_eligible(10_000, dim, 50) == bool(want)
        assert not retrieval.tc_eligible(10_000, dim, 50, _lib.FM_EXACT_ONLY)


@pytest.mark.parametrize("N,Q,k", [(1_000_000, 65536, 50), (9000, 600, 50), (30011, 4000, 200), (777, 1, 1)])
def test_wide_workspace_only_adds_wider_packed_images(lib, N, Q, k):
    """D = 512 keeps everything of D = 256 but the fp16 operand images, which are twice as wide:
    (n_pad + q_pad) * 256 more halves."""
    def ws(dim, flags=0):
        n = ctypes.c_size_t()
        _lib.check(lib.mclst_find_matches_workspace_bytes(N, Q, dim, k, flags, ctypes.byref(n)), "workspace")
        return n.value
    n_pad = -(-N // 256) * 256
    q_pad = -(-Q // 128) * 128
    extra = (n_pad + q_pad) * 256 * 2
    diff = ws(512) - ws(256)
    assert abs(diff - extra) < 2 * 256, (diff, extra)
    # the images are padded to whole 64-wide K blocks
    assert ws(449) == ws(512) and ws(257) == ws(320) < ws(321)
    # the exact path keeps no packed image: its workspace does not depend on the width
    assert ws(512, _lib.FM_EXACT_ONLY) == ws(256, _lib.FM_EXACT_ONLY)
    assert ws(513) == ws(512, _lib.FM_EXACT_ONLY)
