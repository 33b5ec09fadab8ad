"""GPU DAG replay: the windowed (pre-verified scripts) schedule must give exactly the per-transaction verdicts and
the final UTXO set of the blockwise schedule, which in turn must match the oracle's composed-view replay."""
import numpy as np
import pytest

import oracle_tx
from rusty_kaspa_b200 import Params
from rusty_kaspa_b200.replay import DagReplayer
from rusty_kaspa_b200.simgen import SimDag
from rusty_kaspa_b200.txbatch import build_batch

pytestmark = pytest.mark.gpu


def _blocks(seed, n_blocks, tpb, mix, frac_invalid):
    dag = SimDag(seed=seed, n_keys=64, n_nonces=128, mix=mix, frac_invalid=frac_invalid, coinbase_maturity=2, coinbase_outputs=6)
    return dag, [dag.make_block(tpb) for _ in range(n_blocks)]


@pytest.mark.parametrize("mix", [(1, 0, 0, 0), (0.4, 0.2, 0.2, 0.2)])
def test_windowed_equals_blockwise_equals_oracle(gpu_ctx, oracle, mix):
    dag, blocks = _blocks(31, 36, 20, mix, 0.12)
    prm = Params(coinbase_maturity=2, storage_mass_parameter=dag.C)
    # oracle
    ost = oracle_tx.State(oracle)
    op = oracle_tx.params(coinbase_maturity=2, storage_mass_parameter=dag.C)
    exp = []
    for txs, pov in blocks:
        b = build_batch(txs)
        r = ost.validate(b, pov, 0, op, threads=2)
        exp.append(r)
        ost.accept(b, ((r["status"] == 0) | (r["status"] == 12)).astype(np.uint8), pov)
        ost.commit()
    # blockwise on the GPU
    r1 = DagReplayer(gpu_ctx, prm, 1 << 14)
    got1 = r1.replay_blockwise(blocks)
    # windowed on the GPU: three windows of 12 blocks
    r2 = DagReplayer(gpu_ctx, prm, 1 << 14)
    got2 = []
    for w in range(0, len(blocks), 12):
        got2 += r2.replay_windowed(blocks[w:w + 12])
    for e, a, c in zip(exp, got1, got2):
        for f in ("status", "script_err"):
            assert (a[f] == e[f]).all() and (c[f] == e[f]).all(), f
        ok = e["status"] == 0
        assert (a["fee"][ok] == e["fee"][ok]).all() and (c["fee"][ok] == e["fee"][ok]).all()
    assert r1.us.count() == r2.us.count() == ost.count()
    assert r1.us.digest() == r2.us.digest() == ost.digest()
    assert len({int(s) for e in exp for s in e["status"]}) >= 4
    r1.close(); r2.close(); ost.close()


def test_multiset_hash_follows_the_utxo_set(gpu_ctx):
    """utxo_validation.rs:120,144,189: the running multiset hash (coinbase + accepted txs of every block, K8) stays equal to
    the MuHash of the whole UTXO set (kgv_utxo_muhash) — checked after every few blocks of a replay with rejected txs."""
    from rusty_kaspa_b200 import MuHash
    dag, blocks = _blocks(17, 24, 16, (0.6, 0.2, 0.1, 0.1), 0.15)
    prm = Params(coinbase_maturity=2, storage_mass_parameter=dag.C)
    r = DagReplayer(gpu_ctx, prm, 1 << 13)
    ms = MuHash.of_utxo_set(gpu_ctx, r.us)
    assert ms.finalize() == MuHash(gpu_ctx).finalize()  # empty set
    seen_reject = False
    for w in range(0, len(blocks), 6):
        res = r.replay_blockwise(blocks[w:w + 6], multiset=ms)
        seen_reject = seen_reject or any(((x["status"] != 0) & (x["status"] != 12)).any() for x in res)
        whole = MuHash.of_utxo_set(gpu_ctx, r.us)
        assert ms.finalize() == whole.finalize(), w
    assert seen_reject and r.us.count() > 0
    r.close()


@pytest.mark.parametrize("fixture,check_every", [("simpa_goref_1060.json.gz", 1), ("simpa_goref_pruning_5000.json.xz", 64)])
def test_virtual_chain_of_the_simpa_dag_reproduces_the_reference_headers(gpu_ctx, fixture, check_every):
    """The reference's simpa DAG fixture replayed on the GPU along its virtual selected-parent chain, mergeset by mergeset in consensus
    order (golden_util.simpa_dag_replay_plan): kgv_validate_txs against the GPU UTXO table (selected parent: SkipScriptChecks, the
    rest Full, utxo_validation.rs:132-137), kgv_muhash_txs, kgv_utxo_apply_accepted.  After every chain block the running multiset
    hash must finalize to the utxoCommitment the REFERENCE wrote into that header, and the accepted tx ids to its acceptedIdMerkleRoot."""
    import pyref
    from golden_util import simpa_dag_replay_plan
    from rusty_kaspa_b200 import MuHash, GpuUtxoSet, TransactionValidator
    from rusty_kaspa_b200.validator import FLAGS_FULL, FLAGS_SKIP_SCRIPT_CHECKS
    fx, by, order, sp, ordered_mergeset, chain = simpa_dag_replay_plan(fixture)
    tip = chain[-1]
    tv = TransactionValidator(gpu_ctx, Params(coinbase_maturity=fx["coinbase_maturity"], storage_mass_parameter=fx["storage_mass_parameter"]))
    us = GpuUtxoSet(gpu_ctx, 1 << 16)
    running = MuHash(gpu_ctx)
    n_txs = n_blocks_merged = 0
    for pos, b in enumerate(chain[1:]):
        pov, s = by[b]["daa_score"], sp(b)
        cbb = build_batch([by[s]["txs"][0]])
        one = np.ones(1, dtype=np.uint8)
        running.combine(MuHash.from_transactions(gpu_ctx, cbb, one, pov, utxo_set=us))
        us.add_transactions(cbb, one, pov)
        accepted_ids = [gpu_ctx.tx_ids(cbb)[0].tobytes()]
        for k, mb in enumerate(ordered_mergeset(b)):
            n_blocks_merged += 1
            txs = by[mb]["txs"][1:]
            if not txs:
                continue
            batch = build_batch(txs)
            res = tv.validate_transactions_in_parallel(us, batch, pov, FLAGS_SKIP_SCRIPT_CHECKS if k == 0 else FLAGS_FULL)
            acc = (res["status"] == 0).astype(np.uint8)
            running.combine(MuHash.from_transactions(gpu_ctx, batch, acc, pov, utxo_set=us))
            us.add_transactions(batch, acc, pov)
            ids = gpu_ctx.tx_ids(batch)
            accepted_ids += [ids[i].tobytes() for i in range(len(txs)) if acc[i]]
            n_txs += int(acc.sum())
        if pos % check_every == 0 or b == tip:  # every finalize is one 3072-bit inversion (~25 ms)
            assert running.finalize().hex() == by[b]["utxo_commitment"], (b, pov)
        inner = gpu_ctx.merkle_roots(np.frombuffer(b"".join(accepted_ids), dtype=np.uint8).reshape(-1, 32), [0, len(accepted_ids)])[0].tobytes()
        assert pyref.blake2b_keyed(b"MerkleBranchHash", bytes.fromhex(by[s]["accepted_id_merkle_root"]) + inner).hex() == by[b]["accepted_id_merkle_root"], b
    assert MuHash.of_utxo_set(gpu_ctx, us).finalize().hex() == by[tip]["utxo_commitment"]
    assert len(chain) > 30 and n_txs > 150 and n_blocks_merged > 200, (len(chain), n_txs, n_blocks_merged)
    if "5000" in fixture:
        assert len(chain) > 1500 and n_txs > 4500
    us.close()


def _fast_windows(n_blocks, tpb, window, **kw):
    from rusty_kaspa_b200 import simgen
    g = simgen.FastDag(**kw)
    out, done = [], 0
    while done < n_blocks:
        k = min(window, n_blocks - done)
        g.generate(k, tpb)
        out.append(g.take())
        done += k
    return g, out


def test_replay_of_150k_generated_transactions_matches_the_cpu_path(gpu_ctx, oracle):
    """BASELINE's "bit-exact on a 100k-tx simpa DAG" at its stated size: a generated simpa-shaped chain (C++ generator, 1000 blocks, mixed
    1-/2-input P2PK Schnorr transactions, ~2 % invalid of every class) is replayed in order by kgv_replay_window (128-block windows) and by
    the oracle's restated CPU path (ok_state_replay); every per-transaction verdict, the accepted set and the final UTXO-set digest agree."""
    from rusty_kaspa_b200.replay import DagReplayer, REPLAY_BLOCK_DTYPE
    g, wins = _fast_windows(1000, 170, 128, seed=99, n_keys=512, n_nonces=2048, coinbase_maturity=30, frac_invalid=0.02, coinbase_outputs=16)
    prm = Params(coinbase_maturity=30, storage_mass_parameter=g.C)
    op = oracle_tx.params(coinbase_maturity=30, storage_mass_parameter=g.C)
    r = DagReplayer(gpu_ctx, prm, 1 << 20)
    ost = oracle_tx.State(oracle)
    n_tx = n_acc = 0
    seen = set()
    for wi, (b, first, pov) in enumerate(wins):
        arr = np.zeros(len(pov), dtype=REPLAY_BLOCK_DTYPE)
        arr["first_tx"], arr["n_txs"], arr["pov_daa_score"], arr["flags"] = first[:-1], np.diff(first), pov, 1
        # kgv_batch_prefetch: the next window's upload overlaps this window's compute (every second window; once with a batch that is then NOT the
        # one replayed next: the prefetched copy must simply be ignored)
        if wi + 1 < len(wins) and wi % 2 == 0:
            r.prefetch(wins[wi + 1][0])
        elif wi + 2 < len(wins) and wi == 3:
            r.prefetch(wins[wi + 2][0])
        got, acc = r.replay_window(b, arr, want_accept=True)
        exp, eacc = oracle_tx.state_replay(ost, b, first, pov, op, threads=16)
        for f in ("status", "script_err"):
            assert (got[f] == exp[f]).all(), f
        ok = exp["status"] == 0
        assert (got["fee"][ok] == exp["fee"][ok]).all() and (acc == eacc).all()
        n_tx += len(b.txs) - len(pov); n_acc += int(acc.sum()) - len(pov)
        seen |= {(int(s), int(e)) for s, e in zip(got["status"], got["script_err"])}
    c = g.counts()
    assert n_tx >= 100_000 and n_acc == n_tx - c["n_invalid"], (n_tx, n_acc, c)
    assert r.us.count() == ost.count() == c["n_utxos"] and r.us.digest() == ost.digest()
    assert len(seen) >= 6, seen
    r.close(); ost.close(); g.close()


def test_replay_block_flags_follow_the_reference_semantics(gpu_ctx, oracle):
    """Per-block flags of kgv_replay_window against the oracle: merged blocks whose coinbase is NOT accepted (only the selected parent's is,
    utxo_validation.rs:116-121), SkipScriptChecks blocks (:138-140: a bad signature is accepted there), validate-only blocks (:219-225: verdicts
    but no state change), on a mixed-class chain whose later blocks then miss the outputs that were never created."""
    from rusty_kaspa_b200.replay import DagReplayer, REPLAY_BLOCK_DTYPE
    g, wins = _fast_windows(160, 40, 40, seed=7, n_keys=64, n_nonces=256, coinbase_maturity=3, mix=(0.4, 0.2, 0.2, 0.2), frac_invalid=0.1, coinbase_outputs=12)
    prm = Params(coinbase_maturity=3, storage_mass_parameter=g.C)
    op = oracle_tx.params(coinbase_maturity=3, storage_mass_parameter=g.C)
    r = DagReplayer(gpu_ctx, prm, 1 << 16)
    ost = oracle_tx.State(oracle)
    rng = np.random.default_rng(5)
    seen_flags, skipped_bad_sig = set(), 0
    for b, first, pov in wins:
        flags = rng.choice([1, 1, 1, 0, 3, 4, 5, 2], size=len(pov)).astype(np.uint32)
        arr = np.zeros(len(pov), dtype=REPLAY_BLOCK_DTYPE)
        arr["first_tx"], arr["n_txs"], arr["pov_daa_score"], arr["flags"] = first[:-1], np.diff(first), pov, flags
        got, acc = r.replay_window(b, arr, want_accept=True)
        exp, eacc = oracle_tx.state_replay(ost, b, first, pov, op, block_flags=flags, threads=8)
        assert (got["status"] == exp["status"]).all() and (got["script_err"] == exp["script_err"]).all() and (acc == eacc).all()
        seen_flags |= set(int(f) for f in flags)
        assert r.us.count() == ost.count()
    assert r.us.digest() == ost.digest() and seen_flags >= {0, 1, 2, 3, 4, 5}
    r.close(); ost.close(); g.close()


def test_window_with_sibling_duplicates_double_spends_and_rejected_creators(gpu_ctx, oracle):
    """What a DAG window can hold and a chain cannot, against the oracle's block-by-block composed view: the SAME transaction in several sibling
    blocks (only its first instance is accepted, the others find their inputs spent), a different transaction double-spending an outpoint an
    earlier block of the window consumed, a transaction placed BEFORE the block that creates what it spends, and creators whose signature is
    broken after their descendants were built (txids do not cover signature scripts: the whole subtree must come out MissingTxOutpoints).
    One window, so every dependency is resolved inside kgv_replay_window's walk; then the window is replayed again in 7-block pieces."""
    import copy
    from rusty_kaspa_b200.simgen import tx_id
    dag = SimDag(seed=77, n_keys=64, n_nonces=128, mix=(0.6, 0.2, 0.1, 0.1), frac_invalid=0.0, coinbase_maturity=2, coinbase_outputs=6)
    rng = np.random.default_rng(3)
    blocks, n_respent = [], 0
    for bi in range(42):
        before = {(u["txid"], u["index"]): u for u in dag.utxos}
        txs, pov = dag.make_block(14)
        blocks.append((list(txs), pov))
        if bi in (10, 20, 30):
            # a double spend by a DIFFERENT transaction: the generator is handed back an outpoint this block just spent
            left = {(u["txid"], u["index"]) for u in dag.utxos}
            gone = [u for k, u in before.items() if k not in left]
            cand = [u for u in gone if not u["coinbase"] and u["amount"] >= 4]
            assert cand
            saved, dag.utxos = dag.utxos, [cand[0]]
            txs2, pov2 = dag.make_block(1)  # coinbase + ONE transaction, which can only pick the outpoint that is already spent
            assert len(txs2) == 2 and (txs2[1]["inputs"][0]["txid"], txs2[1]["inputs"][0]["index"]) == (cand[0]["txid"], cand[0]["index"])
            blocks.append((list(txs2), pov2))
            dag.utxos = saved + dag.utxos
            n_respent += 1
    # sibling duplicates: copies of earlier transactions in later blocks (and one copy EARLIER than its original)
    n_dup = 0
    for src_b, dst_b, k in ((5, 6, 2), (5, 9, 2), (12, 13, 4), (17, 25, 1), (31, 28, 3), (34, 35, 5), (34, 36, 5)):
        blocks[dst_b][0].append(copy.deepcopy(blocks[src_b][0][k]))
        n_dup += 1
    # rejected creators: break the signature of a transaction some later transaction depends on
    ids = {}
    for bi, (txs, _) in enumerate(blocks):
        for ti, t in enumerate(txs):
            ids.setdefault(tx_id(t), (bi, ti))
    broken = 0
    for bi in range(len(blocks) - 1, 0, -1):
        for t in blocks[bi][0][1:]:
            src = ids.get(t["inputs"][0]["txid"])
            if src and src[1] > 0 and broken < 5 and rng.random() < 0.5:
                c = blocks[src[0]][0][src[1]]
                ss = bytearray(c["inputs"][0]["sigscript"])
                if len(ss) > 20 and ss[10] == c["inputs"][0]["sigscript"][10]:
                    ss[10] ^= 0x40
                    c["inputs"][0]["sigscript"] = bytes(ss)
                    broken += 1
    assert broken >= 3 and n_dup == 7 and n_respent == 3
    prm = Params(coinbase_maturity=2, storage_mass_parameter=dag.C)
    op = oracle_tx.params(coinbase_maturity=2, storage_mass_parameter=dag.C)
    ost = oracle_tx.State(oracle)
    exp = []
    for txs, pov in blocks:
        b = build_batch(txs)
        r = ost.validate(b, pov, 0, op, threads=2)
        exp.append(r)
        ost.accept(b, ((r["status"] == 0) | (r["status"] == 12)).astype(np.uint8), pov)
        ost.commit()
    statuses = np.concatenate([e["status"] for e in exp])
    assert (statuses == 1).sum() >= n_dup + broken and (statuses == 9).sum() + (statuses == 10).sum() >= 3, np.bincount(statuses)
    for piece in (len(blocks), 7):
        r2 = DagReplayer(gpu_ctx, prm, 1 << 14)
        got = []
        for w in range(0, len(blocks), piece):
            got += r2.replay_windowed(blocks[w:w + piece])
        for bi, (e, c) in enumerate(zip(exp, got)):
            assert (c["status"] == e["status"]).all() and (c["script_err"] == e["script_err"]).all(), (piece, bi, c["status"], e["status"])
        assert r2.us.count() == ost.count() and r2.us.digest() == ost.digest()
        r2.close()
    ost.close()


@pytest.mark.parametrize("fixture", ["simpa_goref_1060.json.gz", "simpa_goref_pruning_5000.json.xz"])
def test_whole_virtual_chain_as_one_replay_window_reproduces_every_header_commitment(gpu_ctx, fixture):
    """The reference's simpa DAG fixtures, their whole virtual chain as ONE kgv_replay_window call: per chain block the merged blocks in consensus
    order with the chain block's daa score, the selected parent flagged ACCEPT_COINBASE | SKIP_SCRIPTS (utxo_validation.rs:116-140).  Then
    kgv_replay_muhash (one multiset per chain block), kgv_muhash_prefix_combine (the running multiset hash) and kgv_muhash_finalize_batch
    (ONE inversion for all chain blocks): EVERY header's utxoCommitment is reproduced (check_every = 1), and the final table's MuHash equals the tip's."""
    from golden_util import simpa_dag_replay_plan
    from rusty_kaspa_b200 import MuHash
    from rusty_kaspa_b200.muhash import finalize_batch, prefix_combine
    from rusty_kaspa_b200.replay import (DagReplayer, REPLAY_ACCEPT_COINBASE, REPLAY_SKIP_SCRIPTS, replay_blocks_array)
    fx, by, order, sp, ordered_mergeset, chain = simpa_dag_replay_plan(fixture)
    txs, ranges, group_first = [], [], [0]
    for b in chain[1:]:
        pov = by[b]["daa_score"]
        for k, mb in enumerate(ordered_mergeset(b)):
            t = by[mb]["txs"]
            ranges.append((len(txs), len(t), pov, (REPLAY_ACCEPT_COINBASE | REPLAY_SKIP_SCRIPTS) if k == 0 else 0))
            txs.extend(t)
        group_first.append(len(ranges))
    r = DagReplayer(gpu_ctx, Params(coinbase_maturity=fx["coinbase_maturity"], storage_mass_parameter=fx["storage_mass_parameter"]), 1 << 16)
    res, acc = r.replay_window(build_batch(txs), replay_blocks_array(ranges), want_accept=True)
    per_group = r.replay_muhash(group_first)
    running = prefix_combine(gpu_ctx, per_group)
    hashes = finalize_batch(gpu_ctx, running)
    want = [by[b]["utxo_commitment"] for b in chain[1:]]
    got = [h.tobytes().hex() for h in hashes]
    bad = [i for i, (g, w) in enumerate(zip(got, want)) if g != w]
    assert not bad, (len(bad), bad[:5])
    assert MuHash.of_utxo_set(gpu_ctx, r.us).finalize().hex() == want[-1]
    n_acc = int(acc.sum()) - (len(chain) - 1)
    assert len(want) > 30 and n_acc > 150
    if "5000" in fixture:
        assert len(want) > 1500 and n_acc > 4500
    r.close()
