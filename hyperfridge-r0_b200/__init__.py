"""hyperfridge-r0_b200: B200-native STARK segment prover behind hyperfridge's `prover.prove(env, ELF)`.

The directory name is not a Python identifier; import it through `hfb200_loader.load()` (repo root) which
registers it as `hyperfridge_r0_b200`.
"""
from .binding import (Context, Hfb200Error, load_library, LIB_PATH, EXPORTS, CircuitDesc, Stats, N_GLOBAL, P,  # noqa: F401
                      CHECKPOINT_NAMES, Pool, SegmentJob, ir_source, verify_segment, verify_segments, digest_bytes, digest_pair, claim_encode,
                      claim_decode, claim_next_state, verify_claims, Claim, EXIT_HALTED, EXIT_SYSTEM_SPLIT,
                      BLIND_OS_ENTROPY, BLIND_DETERMINISTIC, SegmentDev, SegmentHandle, ACCUM_FN, DEV_INPUTS, SCAN_PRODUCT, SCAN_SUM,
                      device_count, WitnessDev, WitnessHandle, WITGEN_FN, scratch_view, Hal)
from .receipt import Receipt, CompositeReceipt, SegmentReceipt, Journal, encode_journal, decode_journal  # noqa: F401,E402
from .host import B200Prover, ProverOpts, Segment, Session, ProveInfo, default_prover, default_image_id, bind_claims  # noqa: F401,E402
