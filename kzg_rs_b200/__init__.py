"""kzg_rs_b200 -- B200-native (sm_100a) drop-in for the EIP-4844 verification hot path of succinctlabs/kzg-rs.

Host-side mirror of the reference's public interface (src/lib.rs:12-18) over the C ABI of
include/kzgb200.h, plus the EIP-4844 publisher calls (blob_to_kzg_commitment, compute_kzg_proof,
compute_blob_kzg_proof) and EIP-7594 cells (compute_cells, compute_cells_and_kzg_proofs,
recover_cells_and_kzg_proofs, recover_cells_and_kzg_proofs_many -- many blobs, each from its own cells, one result per blob --,
compute_commitments_and_cell_proofs -- a publisher's commitments and cell proofs in one FK20 pass -- and
KzgProof.verify_cell_kzg_proof_batch).  The product is libkzgb200.so (hand-written CUDA); this package only marshals bytes.
"""
from .api import (BatchPipeline, DeviceGroup, compute_challenge, evaluate_polynomial_in_evaluation_form, Blob, Bytes32, Bytes48, KzgError, KzgProof, KzgSettings, Library, lib_path,  # noqa: F401
                  BYTES_PER_BLOB, BYTES_PER_COMMITMENT, BYTES_PER_PROOF, BYTES_PER_FIELD_ELEMENT,
                  blob_to_kzg_commitment, compute_kzg_proof, compute_blob_kzg_proof,
                  Cell, compute_cells, compute_cells_and_kzg_proofs, recover_cells_and_kzg_proofs, recover_cells_and_kzg_proofs_many,
                  compute_commitments_and_cell_proofs, BYTES_PER_CELL, CELLS_PER_EXT_BLOB)
