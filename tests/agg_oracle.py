"""The CPU oracle's view of aggregation proofs (TEST INFRASTRUCTURE ONLY): the KZG accumulator (lhs, rhs) an aggregation circuit
carries in its public instances, snark-verifier's LimbsEncoding<LIMBS, BITS>, and the deferred decider lhs = s * rhs folded into
the oracle's DualMSM.  Built on oracle/verifier.py without changing it: verify_proof stops before the pairing check, the two
carried terms join the proof's MSMs, and the check runs as DualMSM::check does (msm.rs:185-203)."""
import bn254 as bn
import verifier as orc


def encode_accumulator(lhs, rhs, limbs, bits):
    """Instance limbs of a KZG accumulator as an aggregation circuit exposes it: lhs.x, lhs.y, rhs.x, rhs.y, each split into
    `limbs` values of `bits` bits, least significant first (None = the identity, encoded as (0, 0))."""
    out = []
    for pt in (lhs, rhs):
        for v in ((0, 0) if pt is None else pt):
            out += [(v >> (bits * i)) & ((1 << bits) - 1) for i in range(limbs)]
    return out


def decode_accumulator(instances, spec):
    """(lhs, rhs) from a proof's instances ([circuit][column][row]; columns flattened instance-major) at spec.cells, or None
    when a cell is missing, a limb is >= 2^bits, a coordinate is >= q or a point is off the curve.  (0, 0) is the identity."""
    cols = [col for inst in instances for col in inst]
    vals = []
    for c, r in spec.cells:
        if c >= len(cols) or r >= len(cols[c]):
            return None
        vals.append(int(cols[c][r]))
    L = spec.limbs
    coords = []
    for q in range(4):
        v = 0
        for i, limb in enumerate(vals[q * L:(q + 1) * L]):
            if limb >= 1 << spec.bits:
                return None
            v += limb << (spec.bits * i)
        if v >= bn.P:
            return None
        coords.append(v)
    pts = []
    for x, y in (coords[0:2], coords[2:4]):
        if x == 0 and y == 0:
            pts.append(None)
        elif not bn.g1_is_on_curve((x, y)):
            return None
        else:
            pts.append((x, y))
    return pts[0], pts[1]


def verify_proof(params, vk, instances, proof, multiopen="shplonk", hash_kind="blake2b", accumulator=None, rho=None):
    """orc.verify_proof (SingleStrategy) of an aggregation proof.  accumulator: an object with .limbs, .bits, .cells; the carried
    pair is decoded first (failure = INVALID_INSTANCES, the precedence of the instance check, lib.rs:51-55); then rho * rhs joins
    the left MSM and rho * lhs the right one (DualMSM orientation e(L, [s]G2) e(R, -G2) = 1), so res.L / res.R, and
    orc.accumulate over such results, include the decider.  accumulator=None: orc.verify_proof unchanged."""
    if accumulator is None:
        return orc.verify_proof(params, vk, instances, proof, multiopen, hash_kind)
    if rho is None:
        raise ValueError("a carried accumulator needs its fold scalar rho")
    vk_cols = vk.cs.num_instance_columns
    carried = None
    if all(len(inst) == vk_cols for inst in instances):  # (otherwise orc.verify_proof reports InvalidInstances itself)
        carried = decode_accumulator(instances, accumulator)
        if carried is None:
            return orc.Result(status=orc.INVALID_INSTANCES, error="InvalidInstances (carried accumulator)")
    res = orc.verify_proof(params, vk, instances, proof, multiopen, hash_kind, check_pairing=False, eval_msm=False)
    if res.status != orc.OK:
        return res
    lhs, rhs = carried
    if rhs is not None:
        res.left.append_term(rho, rhs, ("carried", "rhs"))
    if lhs is not None:
        res.right.append_term(rho, lhs, ("carried", "lhs"))
    res.L, res.R = res.left.eval(), res.right.eval()
    if not bn.pairing_check([(res.L, params.s_g2), (res.R, bn.g2_neg(params.g2))]):
        res.status, res.error = orc.CONSTRAINT_SYSTEM_FAILURE, "ConstraintSystemFailure"
    return res
