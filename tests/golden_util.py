"""Helpers shared by the golden-vector tests: fixture loading and the tx dict <-> bytes conventions."""
import gzip
import json
import lzma
import os

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    path = os.path.join(GOLDEN, name)
    if name.endswith(".gz") or name.endswith(".xz"):
        with (gzip.open if name.endswith(".gz") else lzma.open)(path, "rt") as f:
            return json.load(f)
    with open(path) as f:
        return json.load(f)


def tx_from_json(t):
    """hex strings -> bytes, in the dict layout oracle/pyref.py uses"""
    return {"version": t["version"],
            "inputs": [{"txid": bytes.fromhex(i["txid"]), "index": i["index"], "sigscript": bytes.fromhex(i["sigscript"]),
                        "sequence": i["sequence"], "sig_op_count": i["sig_op_count"]} for i in t["inputs"]],
            "outputs": [{"value": o["value"], "spk_version": o["spk_version"], "script": bytes.fromhex(o["script"])} for o in t["outputs"]],
            "lock_time": t["lock_time"], "subnetwork_id": bytes.fromhex(t["subnetwork_id"]), "gas": t["gas"],
            "payload": bytes.fromhex(t["payload"]), "mass": t.get("mass", 0)}


def entry_from_json(e):
    return {"amount": e["amount"], "spk_version": e["spk_version"], "script": bytes.fromhex(e["script"]),
            "block_daa_score": e.get("block_daa_score", 0), "is_coinbase": e.get("is_coinbase", False)}


def apply_sighash_action(tx, entries, action, arg):
    """consensus/core/src/hashing/sighash.rs:655-679"""
    if action == "Output":
        tx["outputs"][arg]["value"] = 100
    elif action == "Input":
        tx["inputs"][arg]["index"] = 2
    elif action == "AmountSpent":
        entries[arg]["amount"] = 666
    elif action == "PrevScriptPublicKey":
        entries[arg]["script"] = entries[arg]["script"] + bytes([1, 2, 3])
    elif action == "Sequence":
        tx["inputs"][arg]["sequence"] = 12345
    elif action == "Payload":
        tx["payload"] = bytes([6, 6, 6, 4, 2, 0, 1, 3, 3, 7])
    elif action == "Gas":
        tx["gas"] = 1234
    elif action == "SubnetworkId":
        tx["subnetwork_id"] = bytes([6, 6, 6, 4, 2, 0, 1, 3, 3, 7]) + bytes(10)
    else:
        assert action == "NoAction"


def simpa_dag_coinbase_only_chain_info():
    """From the simpa DAG fixture: for every block whose PAST contains only coinbase transactions, the data that determines its
    header commitments without running GHOSTDAG (selected parent = max (blue_work, hash) among the level-0 parents,
    consensus/src/processes/ghostdag/ordering.rs:38-42):
      utxo_commitment(B)          = MuHash of { outputs of coinbase(C) with block_daa_score = daa_score(child of C on B's selected chain),
                                    is_coinbase = true : C on the selected chain of B, C != B }   (utxo_validation.rs:117-121,189)
      accepted_id_merkle_root(B)  = merkle_hash(accepted_id_merkle_root(SP(B)), calc_merkle_root([id(coinbase(SP(B)))]))  (KIP-15, :401-410)
    Returns (blocks_by_hash, eligible hashes in file order, selected_parent function)."""
    import functools
    import sys
    fx = load("simpa_goref_1060.json.gz")
    by = {}
    for b in fx["blocks"]:
        by[b["hash"]] = dict(b, blue_work_int=int(b["blue_work"], 16), txs=[tx_from_json(t) for t in b["transactions"]])

    def sp(h):
        ps = by[h]["parents"]
        return max(ps, key=lambda p: (by[p]["blue_work_int"], bytes.fromhex(p))) if ps else None

    sys.setrecursionlimit(10000)

    @functools.lru_cache(None)
    def past_has_spends(h):
        return any(len(by[p]["txs"]) > 1 or past_has_spends(p) for p in by[h]["parents"])

    eligible = [b["hash"] for b in fx["blocks"] if not past_has_spends(b["hash"])]
    return by, eligible, sp


def simpa_dag_replay_plan(fixture="simpa_goref_1060.json.gz"):
    """The reference's own acceptance order for a simpa DAG fixture, derived from header data only (no GHOSTDAG run):
    selected parent = max (blue_work, hash) among the level-0 parents; mergeset(B) = past(B) - past(SP) - {SP}; consensus order =
    SP first, then the rest ascending by (blue_work, hash) (processes/ghostdag/ordering.rs:38-42, utxo_validation.rs:110-160).
    Returns (fixture, by_hash, file_order, sp(h), ordered_mergeset(h), virtual_chain)."""
    fx = load(fixture)
    by, order, idx = {}, [], {}
    for n, b in enumerate(fx["blocks"]):
        by[b["hash"]] = dict(b, bw=int(b["blue_work"], 16), txs=[tx_from_json(t) for t in b["transactions"]])
        order.append(b["hash"])
        idx[b["hash"]] = n
    key = lambda h: (by[h]["bw"], bytes.fromhex(h))
    past = {}  # ancestor sets as integer bitsets over the file (topological) order
    for h in order:
        s = 0
        for p in by[h]["parents"]:
            s |= past[p] | (1 << idx[p])
        past[h] = s

    def sp(h):
        return max(by[h]["parents"], key=key) if by[h]["parents"] else None

    def ordered_mergeset(h):
        s = sp(h)
        if s is None:
            return []
        bits = past[h] & ~past[s] & ~(1 << idx[s])
        rest = []
        while bits:
            low = bits & -bits
            rest.append(order[low.bit_length() - 1])
            bits ^= low
        return [s] + sorted(rest, key=key)

    tip = max(order, key=key)
    chain = [tip]
    while sp(chain[-1]) is not None:
        chain.append(sp(chain[-1]))
    chain.reverse()
    return fx, by, order, sp, ordered_mergeset, chain


def bip340_vectors():
    """tests/golden/bip340_vectors.csv (rows 0-14 of BIP-340's test-vectors.csv, provenance and self-validation in make_bip340.py):
    returns (pk (n,32), msg (n,32), sig (n,64) uint8 arrays, expected KGV_SIG_* status list, comments)"""
    import csv
    import os
    import numpy as np
    rows = list(csv.DictReader(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "bip340_vectors.csv"))))
    hexarr = lambda k, n: np.frombuffer(b"".join(bytes.fromhex(r[k]) for r in rows), dtype=np.uint8).reshape(-1, n).copy()
    exp = [int(r["kgv_status"]) for r in rows]
    assert all((e == 1) == (r["verification result"] == "TRUE") for e, r in zip(exp, rows))
    return hexarr("public key", 32), hexarr("message", 32), hexarr("signature", 64), exp, [r["comment"] for r in rows]


def storage_mass_cases():
    """tests/golden/storage_mass.json -> list of (name, tx dict, entries, storage_mass_parameter, expected mass or None, group) ; transactions of one
    plurality `group` must have equal non-zero mass (consensus/core/src/mass/mod.rs:516-729)"""
    d = load("storage_mass.json")

    def tx_of(ins, outs, in_scripts=None, out_scripts=None):
        n_i, n_o = len(ins), len(outs)
        in_scripts, out_scripts = in_scripts or [b""] * n_i, out_scripts or [b""] * n_o
        tx = {"version": 0, "inputs": [{"txid": bytes.fromhex("880eb9819a31821d9d2399e2f35e2433b72637e393d71ecc9b8d0250f49153c3"), "index": i, "sigscript": b"", "sequence": 0,
                                        "sig_op_count": 0} for i in range(n_i)],
              "outputs": [{"value": v, "spk_version": 0, "script": s} for v, s in zip(outs, out_scripts)], "lock_time": 1615462089000,
              "subnetwork_id": bytes(range(1, 11)) + bytes(10), "gas": 0, "payload": b"", "mass": 0}
        ents = [{"amount": a, "spk_version": 0, "script": s, "block_daa_score": 0, "is_coinbase": False} for a, s in zip(ins, in_scripts)]
        return tx, ents
    out = []
    for k, c in enumerate(d["cases"]):
        tx, ents = tx_of(c["ins"], c["outs"])
        out.append((f"case{k}", tx, ents, c["storage_mass_parameter"], c["expected"], None))
    for g, c in enumerate(d["plurality_cases"]):
        tx1, e1 = tx_of(c["inputs_tx1"], c["outputs_tx1"])
        big = bytes([1]) * c["script_len_for_plurality"]
        isc, osc = [b""] * len(c["inputs_tx2"]), [b""] * len(c["outputs_tx2"])
        (osc if c["override_output"] else isc)[c["plurality_index"]] = big
        tx2, e2 = tx_of(c["inputs_tx2"], c["outputs_tx2"], isc, osc)
        out.append((c["name"] + " /tx1", tx1, e1, c["storage_mass_parameter"], None, g))
        out.append((c["name"] + " /tx2", tx2, e2, c["storage_mass_parameter"], None, g))
    return out


def body_validation_blocks():
    """tests/golden/body_validation_block.json -> (hash_merkle_root hex, [(name, txs, expected status name)]): the reference's example block and the three
    set-check mutations of validate_body_in_isolation_test (body_validation_in_isolation.rs:423-460)"""
    import copy
    import pyref
    d = load("body_validation_block.json")
    base = [tx_from_json(t) for t in d["txs"]]
    dup = copy.deepcopy(base); dup.append(copy.deepcopy(dup[1]))
    dbl = copy.deepcopy(base); dbl[2]["inputs"][0]["txid"], dbl[2]["inputs"][0]["index"] = dbl[1]["inputs"][0]["txid"], dbl[1]["inputs"][0]["index"]
    chn = copy.deepcopy(base); chn[3]["inputs"][0]["txid"], chn[3]["inputs"][0]["index"] = pyref.tx_id(chn[2]), 0
    assert [m["error"] for m in d["mutations"]] == ["DuplicateTransactions", "DoubleSpendInSameBlock", "ChainedTransaction"]
    return d["hash_merkle_root"], [("example block", base, 0), ("duplicate", dup, 1), ("double spend", dbl, 2), ("chained", chn, 3)]
