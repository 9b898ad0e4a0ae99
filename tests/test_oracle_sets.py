"""The reference model of the set export (tests/sets_model.py) against the CPU oracle, and the ctypes mirrors of the new
ABI structs against the header.  No GPU needed."""
import ctypes as C
import subprocess

import numpy as np

from conftest import NOW_NS, NOW_SEC, README_FILTER, ROOT
from sets_model import SetsModel, issuer_digests


def _corpus(ora, n=6000):
    cfg = ora.synth_cfg(n, dup_mode=1)
    blob, offs, idx = ora.synth_corpus(cfg, 0, n)
    iblob, ioffs = ora.synth_issuers(cfg)
    return blob, offs, idx, iblob, ioffs


def _two_batches(ora):
    blob, offs, idx, iblob, ioffs = _corpus(ora)
    m = SetsModel(ora, README_FILTER)
    h = (len(offs) - 1) // 2
    ra, na = m.process(blob, offs[:h + 1], iblob, ioffs, idx[:h], NOW_NS)
    rb, nb = m.process(blob, offs[h:], iblob, ioffs, idx[h:], NOW_NS)
    return m, (ra, rb), (na, nb)


def test_model_sets_agree_with_oracle_cardinalities(ora):
    m, (ra, rb), _ = _two_batches(ora)
    sets = m.list_sets()
    assert len(sets) > 10 and sum(c for _, _, c in sets) < m.next_index       # the corpus has duplicates
    for d, h, c in sets:
        assert m.db.set_cardinality(h, d) == c
    ex = m.export()
    assert ex.sets.size == len(sets) and ex.n_members == sum(c for _, _, c in sets)
    keys = [(bytes(s["issuer_digest"]), int(s["exp_hour"])) for s in ex.sets]
    assert keys == sorted(keys)
    for j in range(ex.sets.size):
        fi = [f for _, f in ex.members(j)]
        assert fi == sorted(fi) and len(set(fi)) == len(fi)


def test_model_members_equal_the_oracle_cache_sets(ora):
    """Every set's members, replayed through the oracle's own KnownCertificates over its MockRemoteCache
    (ora_was_unknown / ora_cache_set_list), are exactly the model's members; the new-entry bits agree too."""
    blob, offs, idx, iblob, ioffs = _corpus(ora, 4000)
    m = SetsModel(ora, README_FILTER)
    r, new = m.process(blob, offs, iblob, ioffs, idx, NOW_NS)
    ids = []
    for k in range(len(ioffs) - 1):
        der = iblob[int(ioffs[k]):int(ioffs[k + 1])].tobytes()
        rc, c = ora.parse_cert(der)
        ids.append(ora.issuer_id(der[c.spki_off:c.spki_off + c.spki_len]))
    cache = ora.Cache()
    for i in np.nonzero(r.status == ora.ST_OK)[0]:
        a = int(offs[i]) + int(r.serial_off[i])
        was = cache.was_unknown(int(r.exp_hour[i]), ids[int(idx[i])][1], blob[a:a + int(r.serial_len[i])].tobytes())
        assert was == bool(new[i])
    id_of = {d: s for d, s in ids}
    for d, h, c in m.list_sets():
        got = cache.set_list(ora.serials_key(h, id_of[d]))
        assert sorted(got) == sorted(s for s, _ in m.members(h, d)) and len(got) == c


def test_first_indices_are_the_positions_of_the_new_entries(ora):
    m, (ra, rb), (na, nb) = _two_batches(ora)
    was_unknown = np.concatenate([ra.was_unknown, rb.was_unknown])
    assert np.array_equal(np.concatenate([na, nb]), was_unknown)            # no long serials in this corpus
    ex = m.export()
    assert sorted(ex.first_index.tolist()) == np.nonzero(was_unknown)[0].tolist()
    assert ex.next_index == was_unknown.size


def test_eviction_drops_exactly_the_expired_sets(ora):
    m, _, _ = _two_batches(ora)
    before = m.list_sets()
    hours = sorted({h for _, h, _ in before})
    cut = hours[len(hours) // 2] * 3600
    m.evict_expired(cut)
    after = m.list_sets()
    assert after == [s for s in before if s[1] * 3600 > cut] and len(after) < len(before)
    for d, h, c in before:
        assert m.db.set_cardinality(h, d) == (c if h * 3600 > cut else 0)


def test_list_sets_hour_range_and_preload(ora):
    blob, offs, idx, iblob, ioffs = _corpus(ora, 2000)
    m = SetsModel(ora, README_FILTER)
    dig = issuer_digests(ora, iblob, ioffs)[0]
    m.preload(NOW_SEC // 3600 + 5, dig, [b"\x01\x02", b"\x03", b"\x01\x02"])
    assert m.next_index == 3 and m.members(NOW_SEC // 3600 + 5, dig) == [(b"\x01\x02", 0), (b"\x03", 1)]
    m.process(blob, offs, iblob, ioffs, idx, NOW_NS)
    all_ = m.list_sets()
    hours = sorted({h for _, h, _ in all_})
    lo, hi = hours[1], hours[-2]
    assert m.list_sets(lo, hi) == [s for s in all_ if lo <= s[1] <= hi]


def test_set_struct_layouts_match_header(tmp_path):
    """ctmr_set_info / ctmr_set_export: sizes and offsets of the ctypes mirrors, measured with a gcc probe."""
    from ct_mapreduce_b200 import capi
    src = tmp_path / "probe.c"
    src.write_text('#include "include/ctmr.h"\n#include <stdio.h>\n#include <stddef.h>\n'
                   'int main(){printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\\n",'
                   'sizeof(ctmr_set_info), offsetof(ctmr_set_info, exp_hour), offsetof(ctmr_set_info, count),'
                   'offsetof(ctmr_set_info, member_off), sizeof(ctmr_set_export), offsetof(ctmr_set_export, next_index),'
                   'offsetof(ctmr_set_export, n_sets), offsetof(ctmr_set_export, n_members), offsetof(ctmr_set_export, serial_bytes),'
                   'offsetof(ctmr_set_export, sets), offsetof(ctmr_set_export, sets_cap), offsetof(ctmr_set_export, serials),'
                   'offsetof(ctmr_set_export, serial_off), offsetof(ctmr_set_export, first_index),'
                   'offsetof(ctmr_set_export, members_cap));return 0;}\n')
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-I", ROOT, str(src), "-o", str(exe)], check=True, cwd=ROOT)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    S, X, D = capi.SetInfo, capi.SetExport, capi.SET_INFO_DTYPE
    assert got == [C.sizeof(S), S.exp_hour.offset, S.count.offset, S.member_off.offset, C.sizeof(X), X.next_index.offset,
                   X.n_sets.offset, X.n_members.offset, X.serial_bytes.offset, X.sets.offset, X.sets_cap.offset, X.serials.offset,
                   X.serial_off.offset, X.first_index.offset, X.members_cap.offset]
    assert got[:4] == [D.itemsize, D.fields["exp_hour"][1], D.fields["count"][1], D.fields["member_off"][1]]
