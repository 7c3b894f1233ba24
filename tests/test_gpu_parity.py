"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on identical packed
batches.  Bit-exact: every comparison is byte equality."""
import random

import numpy as np
import pytest

from distributed_crawler_b200 import abi
from distributed_crawler_b200.corpus import Corpus
from distributed_crawler_b200.engine import Engine, names_to_keys32
from distributed_crawler_b200.pack import Channel, Comment, FormattedText, Message, pack_telegram
from helpers import ALL, TANDEM, assert_results_equal, msg, names, no_page, vector_message
from oracle.pyoracle import Oracle

pytestmark = pytest.mark.gpu


def both(batch, flags=ALL, **cfg):
    o, e = Oracle(**cfg), Engine(**cfg)
    ro, rg = o.telegram(batch, flags), e.telegram(batch, flags)
    assert_results_equal(ro, rg, flags)
    if flags & abi.RUN_FRONTIER:
        assert np.array_equal(o.frontier_export(), e.frontier_export())
    assert rg.gpu_launches > 0
    if rg.gpu_launches == 1 and batch.n:  # a page-sized batch took the one-launch path: the ordinary pipeline as well
        with no_page():
            e2 = Engine(**cfg)
            r2 = e2.telegram(batch, flags)
            assert r2.gpu_launches > 1
            assert_results_equal(ro, r2, flags, "ordinary pipeline")
            if flags & abi.RUN_FRONTIER:
                assert np.array_equal(o.frontier_export(), e2.frontier_export())
            e2.close()
    e.close()
    return ro, rg


def test_reference_link_vectors_on_gpu(vectors, engine):
    msgs = [vector_message(v) for v in vectors["channel_links"]]
    r = engine.telegram(pack_telegram(msgs), abi.RUN_LINKS)
    for i, v in enumerate(vectors["channel_links"]):
        assert names(r, i) == sorted(v["expected"]), f'{v["name"]} ({v["go_file"]}:{v["go_line"]})'


def test_reference_filter_vectors_on_gpu(vectors, engine):
    got = engine.filter_usernames([v["username"].encode() for v in vectors["filter_username"]])
    for v, reason in zip(vectors["filter_username"], got):
        assert (reason == "") == v["valid"], v["name"]
        if not v["valid"]:
            assert reason == v["reason"], v["name"]


def test_tandem_vector_on_gpu(vectors, engine):
    t = vectors["tandem"]["with_edges"]
    m = msg("messageText", t["text"], [tuple(e) for e in t["entities"]])
    r = engine.telegram(pack_telegram([m], [Channel(name=t["owner_url"], username=t["owner_url"])]), TANDEM)
    edges = [l["name"][: l["len"]].tobytes().decode() for l in r.links if l["flags"] & abi.LF_NEW]
    assert edges == t["expected_edges"]


@pytest.mark.parametrize("n,profile", [(1, 2), (7, 1), (3000, 2), (60000, 2), (60000, 3), (20000, 1)])
def test_corpus_parity(n, profile):
    c = Corpus(n, profile=profile, first=12345)
    both(c.batch, ALL)


def test_corpus_parity_configs():
    c = Corpus(30000, profile=2)
    both(c.batch, ALL, tz_offset_sec=19800, crawl_label=b'lab"<el>\xff', min_post_date=1_720_000_000,
         capture_nsec=0, created_at_sec=1_760_000_000)
    both(c.batch, TANDEM, tz_offset_sec=-18000)
    both(c.batch, abi.RUN_JSONL)


def test_empty_and_ragged():
    both(pack_telegram([]))
    ms = [msg("messageText", ""), msg("messageText", None), msg("none"), msg("messagePhoto", "", media="x"),
          msg("messageText", "a"), msg("messageVideo", None, media="VID"), msg("messageText", "t.me/", handle=""),
          msg("messageText", "t.me/abcd"), msg("messageText", "t.me/abcde"), msg("messageText", "xt.me/abcdefghijklmnopqrstuvwxyz0123456789x")]
    both(pack_telegram(ms, [Channel("", "", "")]))


def test_status_edge_cases():
    ms = [msg(date=1_600_000_000, text="t.me/skipped1"), msg(date=1_800_000_000, text="t.me/kept12"),
          msg(text="x", panics=True, date=1_800_000_000),
          msg("messageText", "😀 @testchan", [(1, 5, "mention", "")], date=1_800_000_000),
          msg("messageText", "abc @testchan", [(4, -3, "mention", "")], date=1_800_000_000),
          msg("messageText", "abc @testchan", [(2 ** 31 - 1, 2, "url", "")], date=1_800_000_000)]
    ro, rg = both(pack_telegram(ms), ALL, min_post_date=1_700_000_000)
    assert list(rg.status[:4]) == [abi.ST_SKIPPED, abi.ST_EMITTED, abi.ST_FAILED, abi.ST_FAILED]


def test_regex_adversarial():
    chain = "t.me/abcdt.me/efght.me/ijklmt.me/nopqr xt.me/chain_end " * 40
    longname = "t.me/" + "a" * 31 + "t.me/bcdefg " + "t.me/" + "b" * 32 + "t.me/cdefgh " + "t.me/" + "c" * 40
    many = " ".join(f"t.me/name{i:05d}" for i in range(1500))
    dup = " ".join("t.me/SameName https://t.me/samename/1" for _ in range(300))
    reserved = "t.me/joinchat/x t.me/JoinChat t.me/sharefoo t.me/share t.me/proxy?x t.me/addstickers t.me/setlanguagex"
    ents = [(0, 4, "url", ""), (5, 600, "url", ""), (3, 9, "mention", ""), (0, 5000, "mention", ""), (7, 1, "text_url", "http://t.me/share"),
            (7, 1, "text_url", "https://t.me/share/url?url=https://t.me/realchan"), (9, 2, "text_url", "t.me/ok_chan_1"), (0, 0, "bold", "")]
    ms = [msg("messageText", chain), msg("messageText", longname), msg("messageText", many), msg("messageText", dup),
          msg("messageText", reserved), msg("messagePhoto", many[:9000], ents), msg("messageText", "@ab @abcd @abcde_ @1abcde", [(0, 25, "mention", "")]),
          msg("messageText", "é" * 70 + "t.me/after_two_byte " + "😀" * 33 + "t.me/after_emoji", [(70, 20, "url", ""), (70 + 20 + 66, 16, "url", "")])]
    both(pack_telegram(ms))


def test_utf8_escape_fuzz_around_strip_boundaries():
    rng = random.Random(99)
    frag = [b"a", b" ", b"\"", b"\\", b"<", b"&", b"\n", b"\x01", b"\x7f", "é".encode(), "Я".encode(), "中".encode(),
            "😀".encode(), " ".encode(), " ".encode(), "‧".encode(), b"\xe2\x80", b"\xe2", b"\x80", b"\xbf",
            b"\xff", b"\xc0\x80", b"\xc1", b"\xed\xa0\x80", b"\xed\x9f\xbf", b"\xf0\x9f", b"\xf0\x9f\x98", b"\xf4\x90\x80\x80",
            b"\xf4\x8f\xbf\xbf", b"\xe0\x9f\x80", b"\xe0\xa0\x80", b"\xf0\x8f\x80\x80", b"\xf0\x90\x80\x80", b"\xf5\x80\x80\x80"]
    ms = []
    for t in range(3000):
        n = rng.choice([120, 124, 126, 127, 128, 129, 130, 132, 250, 256, 260, 384, 5, 0, 1, 3,
                        496, 507, 508, 509, 510, 511, 512, 513, 514, 516, 1020, 1023, 1024, 1025, 1536])
        body = bytearray()
        while len(body) < n:
            body += rng.choice(frag) if rng.random() < 0.5 else b"xyz "[: rng.randrange(1, 5)]
        body = bytes(body[: n + rng.randrange(0, 4)])
        ents = [(rng.randrange(0, 140), rng.randrange(0, 12), rng.choice(["mention", "url"]), "")] if t % 3 == 0 else []
        ms.append(msg("messageText", body, ents, handle=body[:40], reactions=[(body[:7], 3), (body[3:9], 1)] if t % 5 == 0 else []))
    ro, rg = both(pack_telegram(ms))
    assert (ro.status == abi.ST_FAILED).sum() > 0  # the fuzz does hit the surrogate-offset panic path


def test_reactions_and_comments():
    rs = [("👍", 3), ("❤", 2), ("👍", 9), ("❤️", 1), ("", 5), ("zz", -4), ("a\"b", 2 ** 31 - 1)]
    cm = [Comment("c1 <x>", [("🔥", 1), ("🔥", 2), ("a", 0)], 5, 0, "bob"), Comment("", None, 0, 1, ""), Comment("t.me/notalink", [], -1, -2, "h\n")]
    ms = [msg("messageText", "x", reactions=rs, comments=cm), msg("messageText", "y", reactions=rs[:1], comments=None),
          msg("messageText", "z", reactions=[(f"k{i:02d}", i) for i in range(31, -1, -1)])]
    both(pack_telegram(ms))


def test_big_maps_and_many_links_are_per_record_slow_paths():
    """No format limits: a reactions map with more than 32 entries (also inside a comment, also with repeated and dirty
    keys) and a text with thousands of link candidates are processed like any other record."""
    rs = [(f"k{i % 47:02d}", i) for i in range(100)] + [('q"%d' % i, -i) for i in range(40)] + [("👍", 1), ("", 2), ("👍", 3)]
    cm = [Comment("big map inside", [(f"c{i:03d}", i) for i in range(70, -1, -1)], 1, 2, "h")]
    many = " ".join(f"t.me/chan_{i:05d}" for i in range(6000))
    ms = [msg("messageText", "a", reactions=rs), msg("messageText", "b", reactions=rs[:33], comments=cm),
          msg("messageText", many), msg("messageText", "t.me/after_many x" * 3, reactions=[("z", 1)] * 40)]
    ro, rg = both(pack_telegram(ms))
    assert len(rg.links) >= 6001


def test_frontier_across_batches_and_slots():
    c = Corpus(90000, profile=3)
    o, e = Oracle(), Engine()
    parts = [c.batch.slice(a, a + 30000) for a in (0, 30000, 60000)]
    for p in parts:
        ro = o.telegram(p, TANDEM)
        rg = e.telegram(p, TANDEM)
        assert_results_equal(ro, rg, TANDEM)
    assert np.array_equal(o.frontier_export(), e.frontier_export())
    # pipelined submission over the three slots gives the same set (membership; order is per batch)
    e2 = Engine()
    for s, p in enumerate(parts):
        e2.telegram_submit(s, p, TANDEM)
    tot = 0
    for s in range(3):
        tot += e2.telegram_wait(s).n_new
        e2.release(s)
    assert tot == e.frontier_size()
    a = {bytes(x) for x in e2.frontier_export()}
    assert a == {bytes(x) for x in e.frontier_export()}


def test_frontier_insert_api(engine):
    o = Oracle()
    rng = random.Random(5)
    names_ = [b"name%05d" % rng.randrange(3000) for _ in range(20000)]
    k = names_to_keys32(names_)
    assert np.array_equal(o.frontier_insert(k), engine.frontier_insert(k))
    assert np.array_equal(o.frontier_export(), engine.frontier_export())
    k2 = names_to_keys32([b"name%05d" % i for i in range(2990, 3010)])
    assert np.array_equal(o.frontier_insert(k2), engine.frontier_insert(k2))
    engine.frontier_clear()
    assert engine.frontier_size() == 0


def test_resident_run_matches_batch_call(engine):
    c = Corpus(20000, profile=2)
    r1 = engine.telegram(c.batch, abi.RUN_JSONL | abi.RUN_LINKS)
    engine.telegram_upload(1, c.batch)
    r2 = engine.telegram_run_resident(1, abi.RUN_JSONL | abi.RUN_LINKS, copy=True)
    assert np.array_equal(r1.jsonl, r2.jsonl) and np.array_equal(r1.links, r2.links)
    r3 = engine.telegram_run_resident(1, abi.RUN_JSONL | abi.RUN_NO_D2H)
    assert r3.jsonl_len == r1.jsonl_len
    assert engine.read_jsonl(1, 0, 4096) == r1.jsonl[:4096].tobytes()


def test_full_size_config2_properties():
    """BASELINE config 2 at full size (10 M messages): too big for a full oracle pass in a test, so
    check size-independent properties + byte parity on random windows."""
    n = 10_000_000
    c = Corpus(n, profile=2)
    e = Engine()
    e.telegram_upload(0, c.batch)
    r = e.telegram_run_resident(0, abi.RUN_JSONL | abi.RUN_LINKS | abi.RUN_NO_D2H)
    assert r.n == n and r.jsonl_len > 2000 * n * 0.9
    o = Oracle()
    # the big run's first and last windows are byte-identical to the oracle on those windows
    head = o.telegram(c.batch.slice(0, 3000), abi.RUN_JSONL)
    assert e.read_jsonl(0, 0, len(head.jsonl)) == head.jsonl.tobytes()
    tail = o.telegram(c.batch.slice(n - 3000, n), abi.RUN_JSONL)
    assert e.read_jsonl(0, r.jsonl_len - len(tail.jsonl), len(tail.jsonl)) == tail.jsonl.tobytes()
    # random interior windows: locate each window in the big blob by its oracle bytes
    rng = random.Random(3)
    e2 = Engine()
    for _ in range(12):
        a = rng.randrange(0, n - 4000)
        sub = c.batch.slice(a, a + 4000)
        ro = o.telegram(sub, abi.RUN_JSONL)
        rg = e2.telegram(sub, abi.RUN_JSONL)
        assert np.array_equal(ro.jsonl, rg.jsonl)
    assert e.read_jsonl(0, r.jsonl_len - 1, 1) == b"\n"


def test_emitter_hand_over_boundaries():
    """The lane emitter writes the simple cases itself and leaves the rest to the esc / maps kernels: the rules sit at
    LANE_TEXT_MAX (512 bytes), LANE_LINKS_MAX (4 outlinks), LANE_MAP_MAX (6 entries), 8-byte keys, repeated keys,
    strings that need escaping.  Messages on both sides of every boundary (and, since the round-2 tile experiments, lines
    between 2 and 20 KB, with and without maps, comment lists longer than 4 KB) in one warp and spread over several, in
    shuffled orders so that lines start at every alignment."""
    from distributed_crawler_b200.pack import Comment
    msgs = []
    for k, n in enumerate([0, 1, 15, 16, 17, 127, 128, 129, 511, 512, 513, 1024, 3000, 1900, 2000, 2100, 3900, 4000, 4100, 4150, 4200,
                           4250, 4300, 4400, 4700, 6000, 6200, 9000, 20000]):
        body = ("x" * n)
        msgs.append(Message(id=(k + 1) << 20, text=FormattedText(body)))                       # clean, around the text limit
        msgs.append(Message(id=(k + 100) << 20, text=FormattedText(body[: max(n - 1, 0)] + "\n")))   # needs escaping
        msgs.append(Message(id=(k + 200) << 20, text=FormattedText(body[: max(n - 2, 0)] + "é")))    # non-ASCII, clean
    for nl in range(0, 8):  # outlinks around LANE_LINKS_MAX
        text = " ".join("t.me/channel_%02d_%d" % (nl, j) for j in range(nl))
        msgs.append(Message(id=(300 + nl) << 20, text=FormattedText(text)))
    emoji = ["👍", "❤️", "🔥", "😀", "🎉", "🤔", "👎", "😢", "abcdefgh", "abcdefghi", 'q"k', "a"]
    for nr in range(0, 9):  # reactions around LANE_MAP_MAX
        msgs.append(Message(id=(400 + nr) << 20, text=FormattedText("r"), reactions=[(emoji[j], j + 1) for j in range(nr)]))
    msgs.append(Message(id=500 << 20, reactions=[("👍", 1), ("🔥", 2), ("👍", 3)]))                 # repeated key: last wins
    msgs.append(Message(id=501 << 20, reactions=[("abcdefgh", 1), ("abcdefghi", 2)]))            # 8- and 9-byte keys
    msgs.append(Message(id=502 << 20, reactions=[('q"k', 5), ("a", -7)]))                        # key that needs escaping
    msgs.append(Message(id=503 << 20, reactions=[("", 1), ("b", 2)]))                            # empty key
    msgs.append(Message(id=504 << 20, comments=None))
    msgs.append(Message(id=505 << 20, comments=[Comment("c1", [("👍", 1)], 3, 4, "h"), Comment("c\n2", None, 0, 0, "unknown")]))
    msgs.append(Message(id=506 << 20, handle='ha"ndle', media="m<edia", content_type="messageVideo", text=FormattedText("cap")))
    for k, n in enumerate(range(1950, 2250, 12)):  # lines with reactions on both sides of the buffer-minus-scratch limit
        msgs.append(Message(id=(600 + k) << 20, text=FormattedText("y" * n), reactions=[("👍", 2), ("zz", 1)]))
    for k, n in enumerate(range(4050, 4330, 8)):   # lines without scratch on both sides of the buffer limit
        msgs.append(Message(id=(700 + k) << 20, text=FormattedText("w" * (n - 1) + "\t")))
    big = [Comment("comment %d " % j + "z" * 300, [("🔥", j)], j, 0, "h%d" % j) for j in range(12)]
    msgs.append(Message(id=800 << 20, comments=big))                                               # comment list longer than the buffer
    msgs.append(Message(id=801 << 20, comments=big[:3], reactions=[("👍", 1)], text=FormattedText("t.me/with_comments " * 20)))
    rnd = random.Random(5)
    for order in range(3):
        rnd.shuffle(msgs)
        both(pack_telegram(msgs), ALL)
        both(pack_telegram(msgs[:31]), ALL)


def test_malformed_batches_are_rejected(engine):
    """A batch whose offsets point outside its arrays comes back as TGI_E_ARG with the mask of the broken check (host
    check for small batches, device check for big ones) instead of an illegal address; the context stays usable.  One
    case per check: record strings / channel / content type, entity, reaction and comment offsets, entity URL, reaction
    emoji, comment strings, comment reactions, channel strings."""
    from distributed_crawler_b200.engine import EngineError

    def rejected(b, array, idx, value, mask, field=None):
        a = getattr(b, array).copy()
        if field:
            a[field][idx] = value
        else:
            a[idx] = value
        bad = type(b)(**{k: (a if k == array else getattr(b, k)) for k in b.FIELDS})
        with pytest.raises(EngineError) as ei:
            engine.telegram(bad, ALL)
        assert ei.value.code == abi.E_ARG and f"(mask {mask:#x})" in str(ei.value), (b.n, array, field, str(ei.value))

    for n in (500, 200_000):  # host-side and device-side validation
        b = Corpus(n, profile=2).batch
        for field, value, mask in (("str_off", 1 << 40, 1), ("chan_idx", 1 << 30, 2), ("text_len", 0xFFFFFFF0, 1), ("content_type", 200, 2)):
            rejected(b, "recs", n // 2, value, mask, field)
        rejected(b, "ent_off", n // 3, b.ent_off[-1] + 5, 4)  # not monotonic / past the entity array
        rejected(b, "react_off", n // 3, len(b.reacts) + 5, 8)
        rejected(b, "comment_off", n // 3, len(b.comments) + 5, 16)
        rejected(b, "ents", int(np.flatnonzero(b.ents["type"] == abi.ENT_TEXT_URL)[0]), 0xFFFFFFF0, 32, "url_off")
        rejected(b, "reacts", len(b.reacts) // 2, 0xFFFFFFF0, 64, "emoji_off")
        rejected(b, "comments", len(b.comments) // 2, 0xFFFFFFF0, 128, "text_off")
        rejected(b, "comments", int(np.flatnonzero(b.comments["flags"] & 1)[0]), 0xFFFFFFF0, 256, "react_start")
        rejected(b, "chans", len(b.chans) - 1, 0xFFFFFFF0, 512, "str_off")
    ok = Corpus(1000, profile=2)
    assert engine.telegram(ok.batch, ALL).n == 1000  # still alive


def test_random_messages_of_every_shape():
    """The random messages of tests/test_oracle_golden.py (every content type, nil / empty / filled lists and maps, invalid
    UTF-8, negative ids ...; there the oracle is compared with the independent restatement of tests/go_rules.py) through
    the CUDA path: page kernel and bulk pipeline."""
    from test_oracle_golden import _random_messages
    chans = [Channel("T<itle>  ", "nm", "usr", 10, 20, 30), Channel(b"\xff\"t", "name_2", "", 0, 0, 0), Channel("", "", "u3", 2 ** 31 - 1, 7, 2 ** 40)]
    for trial, cfg in enumerate([dict(), dict(tz_offset_sec=19800, crawl_label=b'lab"<el>\xff', capture_nsec=0, created_at_sec=1_760_000_000),
                                 dict(tz_offset_sec=-12600, min_post_date=1_650_000_000, created_at_nsec=999, capture_nsec=120_000_000)]):
        ms = _random_messages(random.Random(100 + trial), 800)
        both(pack_telegram(ms, chans), ALL, **cfg)
        both(pack_telegram(ms, chans), TANDEM, **cfg)
