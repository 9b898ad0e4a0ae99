"""Reference model of the set read-back (include/ctmr.h, "the sets read back") on top of the CPU oracle.

The oracle decides every entry (parse, filter, expDate, serial); this model keeps what Redis would hold afterwards --
"serials::<expDate>::<issuer>" sets -- together with each member's first-seen global entry index, counted like the
product's next_index (every entry of every batch, every preloaded serial), and produces the canonical export: sets by
(issuer digest, exp_hour), members by first index, evicted sets absent, serials longer than 39 octets never stored
(the product's documented divergence: it declines them with CTMR_ST_SERIAL_TOO_LONG).
"""
from __future__ import annotations

import numpy as np

MAX_SERIAL = 39


def issuer_digests(ora, iblob, ioffs):
    """Issuer.ID() digest of every issuer certificate of a batch (None where it does not parse)."""
    out = []
    for k in range(len(ioffs) - 1):
        der = np.asarray(iblob)[int(ioffs[k]):int(ioffs[k + 1])].tobytes()
        rc, c = ora.parse_cert(der)
        out.append(None if rc else ora.issuer_id(der[c.spki_off:c.spki_off + c.spki_len])[0])
    return out


class SetsModel:
    def __init__(self, ora, issuer_cn_filter: bytes = b"", log_expired: bool = False):
        self.ora = ora
        self.db = ora.DB(issuer_cn_filter, log_expired)
        self.next_index = 0
        self.sets: dict = {}          # (digest, hour) -> {serial: first index}

    def process(self, blob, offsets, iblob, ioffs, issuer_idx, now_ns):
        """One batch through the oracle; returns the oracle's per-entry result and the model's own was_unknown."""
        r = self.db.process(blob, offsets, iblob, ioffs, issuer_idx, now_ns)
        digests = issuer_digests(self.ora, iblob, ioffs)
        blob = np.asarray(blob)
        n = len(offsets) - 1
        new = np.zeros(n, np.uint8)
        for i in range(n):
            if r.status[i] != self.ora.ST_OK or r.serial_len[i] > MAX_SERIAL:
                continue
            a = int(offsets[i]) + int(r.serial_off[i])
            serial = blob[a:a + int(r.serial_len[i])].tobytes()
            s = self.sets.setdefault((digests[int(issuer_idx[i])], int(r.exp_hour[i])), {})
            if serial not in s:
                s[serial] = self.next_index + i
                new[i] = 1
        self.next_index += n
        return r, new

    def preload(self, hour: int, digest: bytes, serials):
        s = self.sets.setdefault((bytes(digest), int(hour)), {})
        for k, ser in enumerate(serials):
            s.setdefault(bytes(ser), self.next_index + k)
        self.next_index += len(serials)

    def evict_expired(self, now_sec: int):
        self.db.evict_expired(now_sec)
        for key in [k for k in self.sets if k[1] * 3600 <= now_sec]:
            del self.sets[key]

    def live(self):
        return sorted((k, v) for k, v in self.sets.items() if v)

    def list_sets(self, lo=None, hi=None):
        """[(digest, hour, count)] of the live sets in canonical order, lo <= hour <= hi."""
        return [(d, h, len(v)) for (d, h), v in self.live() if (lo is None or h >= lo) and (hi is None or h <= hi)]

    def members(self, hour: int, digest: bytes):
        """[(serial, first index)] of one set, by first index."""
        return sorted(self.sets.get((bytes(digest), int(hour)), {}).items(), key=lambda kv: kv[1])

    def export(self):
        """The canonical export as engine.SetExport."""
        from ct_mapreduce_b200 import capi
        from ct_mapreduce_b200.engine import SetExport
        live = self.live()
        sets = np.zeros(len(live), capi.SET_INFO_DTYPE)
        serials, first, lens, run = [], [], [], 0
        for j, ((d, h), mem) in enumerate(live):
            sets[j]["issuer_digest"] = np.frombuffer(d, np.uint8)
            sets[j]["exp_hour"], sets[j]["count"], sets[j]["member_off"] = h, len(mem), run
            for ser, fi in sorted(mem.items(), key=lambda kv: kv[1]):
                serials.append(ser)
                first.append(fi)
                lens.append(len(ser))
            run += len(mem)
        off = np.zeros(len(lens) + 1, np.uint64)
        off[1:] = np.cumsum(lens, dtype=np.uint64)
        return SetExport(self.next_index, sets, np.frombuffer(b"".join(serials), np.uint8).copy(), off, np.array(first, np.uint64))
