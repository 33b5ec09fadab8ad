"""Replay of the reference's simpa-generated DAG fixture with the CPU oracle, checked against what the reference itself wrote into
every header: utxoCommitment (MuHash of the UTXO set in the block's past) and acceptedIdMerkleRoot (KIP-15).  This pins, with real
reference data, the whole path at once: mergeset order, coinbase handling, populate, UTXO-context rules incl. coinbase maturity and
storage mass, script checks, acceptance, UtxoDiff::add_transaction, MuHash::add_transaction, finalize, calc_merkle_root."""
import ctypes
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "oracle"))
sys.path.insert(0, HERE)
import oracle_tx  # noqa: E402
import pyref  # noqa: E402
from golden_util import simpa_dag_replay_plan  # noqa: E402
from rusty_kaspa_b200.txbatch import build_batch  # noqa: E402


class OkMuHash(ctypes.Structure):
    _fields_ = [("num", ctypes.c_uint64 * 48), ("den", ctypes.c_uint64 * 48)]


def _replay(oracle, fixture, blocks_of, chain_only):
    """blocks_of(plan) -> hashes to process in order; chain_only: one evolving state (the virtual chain) instead of one state per block"""
    fx, by, order, sp, ordered_mergeset, chain = simpa_dag_replay_plan(fixture)
    prm = oracle_tx.params(coinbase_maturity=fx["coinbase_maturity"], storage_mass_parameter=fx["storage_mass_parameter"])
    todo = chain if chain_only else order
    state, mh = {}, {}
    accepted_total = 0
    for h in todo:
        b, s = by[h], sp(h)
        m = OkMuHash()
        if s is None:
            oracle.ok_muhash_init(ctypes.byref(m))
            st, accepted_ids = {}, None
        else:
            ctypes.memmove(ctypes.byref(m), ctypes.byref(mh[s]), ctypes.sizeof(m))
            st = state[s] if chain_only else dict(state[s])
            pov = b["daa_score"]

            def add(txid, i, o, coinbase):
                st[(txid, i)] = {"amount": o["value"], "spk_version": o["spk_version"], "script": o["script"], "block_daa_score": pov, "is_coinbase": coinbase}
                d = pyref.utxo_element_bytes(txid, i, pov, o["value"], coinbase, o["spk_version"], o["script"])
                oracle.ok_muhash_add_element(ctypes.byref(m), d, len(d))

            cb = by[s]["txs"][0]
            cid = pyref.tx_id(cb)
            for i, o in enumerate(cb["outputs"]):
                add(cid, i, o, True)
            accepted_ids = [cid]
            for k, mb in enumerate(ordered_mergeset(h)):
                for tx in by[mb]["txs"][1:]:
                    ents = [st.get((i["txid"], i["index"])) for i in tx["inputs"]]
                    if any(e is None for e in ents):
                        continue  # MissingTxOutpoints
                    r = oracle_tx.validate_populated(oracle, build_batch([tx], [ents]), 0, pov, 1 if k == 0 else 0, prm)  # selected parent: SkipScriptChecks
                    if int(r["status"]) != 0:
                        continue
                    for i, e in zip(tx["inputs"], ents):
                        del st[(i["txid"], i["index"])]
                        d = pyref.utxo_element_bytes(i["txid"], i["index"], e["block_daa_score"], e["amount"], e["is_coinbase"], e["spk_version"], e["script"])
                        oracle.ok_muhash_remove_element(ctypes.byref(m), d, len(d))
                    tid = pyref.tx_id(tx)
                    for i, o in enumerate(tx["outputs"]):
                        add(tid, i, o, False)
                    accepted_ids.append(tid)
                    accepted_total += 1
        state[h], mh[h] = st, m
        if chain_only and s is not None:
            del state[s], mh[s]
        mm = OkMuHash()
        ctypes.memmove(ctypes.byref(mm), ctypes.byref(m), ctypes.sizeof(m))
        out = ctypes.create_string_buffer(32)
        oracle.ok_muhash_finalize(ctypes.byref(mm), out)
        assert out.raw.hex() == b["utxo_commitment"], (h, b["daa_score"])
        if accepted_ids is not None:
            root = ctypes.create_string_buffer(32)
            oracle.ok_merkle_root(b"".join(accepted_ids), ctypes.c_size_t(len(accepted_ids)), root)
            assert pyref.blake2b_keyed(b"MerkleBranchHash", bytes.fromhex(by[s]["accepted_id_merkle_root"]) + root.raw).hex() == b["accepted_id_merkle_root"], h
    return len(todo), accepted_total


def test_every_header_commitment_of_the_simpa_dag(oracle):
    """goref-1060-tx-265-blocks: every one of the 266 blocks from its own point of view (one UTXO state per block)"""
    n, accepted = _replay(oracle, "simpa_goref_1060.json.gz", None, chain_only=False)
    assert n == 266 and accepted > 500


def test_virtual_chain_of_the_5000_block_dag(oracle):
    """goref_custom_pruning_depth (5 001 blocks, 4 790 signed transactions): the 1 665 blocks of the virtual selected-parent chain"""
    n, accepted = _replay(oracle, "simpa_goref_pruning_5000.json.xz", None, chain_only=True)
    assert n > 1500 and accepted > 4500
