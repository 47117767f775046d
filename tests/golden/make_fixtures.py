#!/usr/bin/env python3
"""Convert the reference's c-kzg-4844 YAML vectors into compact in-repo goldens.

Run in the build container (needs /root/reference, which does not exist on the GPU box):
    python tests/golden/make_fixtures.py

Sources (all read-only):
  /root/reference/tests/verify_kzg_proof/*/data.yaml            (122 cases, used by kzg_proof.rs:604-631)
  /root/reference/tests/verify_blob_kzg_proof/*/data.yaml       (29 cases,  used by kzg_proof.rs:654-680)
  /root/reference/tests/verify_blob_kzg_proof_batch/*/data.yaml (24 cases,  shipped but unused by the
                                                                 reference's own tests; the only n>=2 verdicts)
  /root/reference/src/trusted_setup.txt                         (mainnet ceremony output)
Outputs:
  tests/golden/ckzg_vectors.json   cases; blobs are referenced by index into the blob store
  tests/golden/ckzg_blobs.bin.gz   the distinct blobs, concatenated (lengths in the json), gzip-compressed
  kzg_rs_b200/data/mainnet_setup.bin   "KZGS" | u32 n1 | u32 n2 | n1*48 B G1 Lagrange (file order) | n2*96 B G2 monomial
Also records the two known-answer tests of kzg_proof.rs:739-778.
"""
import glob, gzip, hashlib, json, os, struct, sys
import yaml

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))

blob_store, blob_index = [], {}


def blob_ref(hexstr):
    raw = bytes.fromhex(hexstr[2:] if hexstr.startswith("0x") else hexstr)
    key = hashlib.sha256(raw).hexdigest()
    if key not in blob_index:
        blob_index[key] = len(blob_store)
        blob_store.append(raw)
    return blob_index[key]


def case_name(path):
    return os.path.basename(os.path.dirname(path))


out = {"verify_kzg_proof": [], "verify_blob_kzg_proof": [], "verify_blob_kzg_proof_batch": []}
for f in sorted(glob.glob(REF + "/tests/verify_kzg_proof/*/data.yaml")):
    d = yaml.safe_load(open(f))
    i = d["input"]
    out["verify_kzg_proof"].append({"name": case_name(f), "commitment": i["commitment"], "z": i["z"],
                                    "y": i["y"], "proof": i["proof"], "output": d["output"]})
for f in sorted(glob.glob(REF + "/tests/verify_blob_kzg_proof/*/data.yaml")):
    d = yaml.safe_load(open(f))
    i = d["input"]
    out["verify_blob_kzg_proof"].append({"name": case_name(f), "blob": blob_ref(i["blob"]),
                                         "commitment": i["commitment"], "proof": i["proof"],
                                         "output": d["output"]})
for f in sorted(glob.glob(REF + "/tests/verify_blob_kzg_proof_batch/*/data.yaml")):
    d = yaml.safe_load(open(f))
    i = d["input"]
    out["verify_blob_kzg_proof_batch"].append({"name": case_name(f), "blobs": [blob_ref(b) for b in i["blobs"]],
                                               "commitments": i["commitments"], "proofs": i["proofs"],
                                               "output": d["output"]})

# known-answer tests embedded in the reference's unit tests
kat_c = yaml.safe_load(open(REF + "/tests/verify_blob_kzg_proof/verify_blob_kzg_proof_case_correct_proof_fb324bc819407148/data.yaml"))
kat_e = yaml.safe_load(open(REF + "/tests/verify_blob_kzg_proof/verify_blob_kzg_proof_case_correct_proof_19b3f3f8c98ea31e/data.yaml"))
out["kat_compute_challenge"] = {  # kzg_proof.rs:739-753
    "blob": blob_ref(kat_c["input"]["blob"]), "commitment": kat_c["input"]["commitment"],
    "z": "0x4f00eef944a21cb9f3ac3390702621e4bbf1198767c43c0fb9c8e9923bfbb31a"}
out["kat_evaluate_polynomial"] = {  # kzg_proof.rs:755-778
    "blob": blob_ref(kat_e["input"]["blob"]),
    "z": "0x637c904d316955b7282f980433d5cd9f40d0533c45d0a233c009bc7fe28b92e3",
    "y": "0x1bdfc5da40334b9c51220e8cbea1679c20a7f32dd3d7f3c463149bb4b41a7d18"}
out["blob_lengths"] = [len(b) for b in blob_store]
out["blob_sha256"] = [hashlib.sha256(b).hexdigest() for b in blob_store]

with open(os.path.join(HERE, "ckzg_vectors.json"), "w") as fh:
    json.dump(out, fh, indent=0, separators=(",", ":"))
with open(os.path.join(HERE, "ckzg_blobs.bin.gz"), "wb") as fh:
    fh.write(gzip.compress(b"".join(blob_store), 9, mtime=0))

lines = open(REF + "/src/trusted_setup.txt").read().split()
n1, n2 = int(lines[0]), int(lines[1])
g1 = b"".join(bytes.fromhex(x) for x in lines[2:2 + n1])
g2 = b"".join(bytes.fromhex(x) for x in lines[2 + n1:2 + n1 + n2])
assert len(g1) == n1 * 48 and len(g2) == n2 * 96
os.makedirs(os.path.join(ROOT, "kzg_rs_b200", "data"), exist_ok=True)
with open(os.path.join(ROOT, "kzg_rs_b200", "data", "mainnet_setup.bin"), "wb") as fh:
    fh.write(b"KZGS" + struct.pack("<II", n1, n2) + g1 + g2)
print("cases:", {k: len(v) for k, v in out.items() if isinstance(v, list) and k.startswith("verify")},
      "distinct blobs:", len(blob_store), "bytes:", sum(map(len, blob_store)))
