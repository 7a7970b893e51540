"""Readers for tests/golden/*.npz (vectors produced by the reference itself, see gen_golden.py)."""
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def bytecode_vectors():
    """yield (case, vector idx, cols, push, keccak, r, expected_row, expected_exc)"""
    z = np.load(os.path.join(GOLDEN, "bytecode.npz"))
    r = z["r"]
    for name in z["names"]:
        name = str(name)
        base, push, kec = z[f"{name}/cols"], z[f"{name}/push"], z[f"{name}/keccak"]
        for k in range(len(z[f"{name}/mut_row"])):
            i, c = int(z[f"{name}/mut_row"][k]), int(z[f"{name}/mut_col"][k])
            cols, kk = base, kec
            if i >= 1000:
                kk = kec.copy()
                kk[c - 100, i - 1000, :] = z[f"{name}/mut_val"][k]
            elif i >= 0:
                cols = base.copy()
                cols[c, i, :] = z[f"{name}/mut_val"][k]
            yield name, k, cols, push, kk, r, int(z[f"{name}/exp_row"][k]), str(z[f"{name}/exp_exc"][k])


def evm_vectors():
    """yield (case, k, steps, bytecode, rw, flags, expected_row, expected_exc)"""
    z = np.load(os.path.join(GOLDEN, "evm.npz"))
    for name in z["names"]:
        name = str(name)
        S, B, R = z[f"{name}/steps"], z[f"{name}/bytecode"], z[f"{name}/rw"]
        for k in range(len(z[f"{name}/mut_kind"])):
            kind, i, c = int(z[f"{name}/mut_kind"][k]), int(z[f"{name}/mut_row"][k]), int(z[f"{name}/mut_col"][k])
            val = z[f"{name}/mut_val"][k]
            s, b, r, flags = S, B, R, 0
            if kind == 0 and i >= 0:
                s = S.copy(); s[c, i, :] = val
            elif kind == 1:
                r = R.copy(); r[c, i, :] = val
            elif kind == 2:
                b = B.copy(); b[c, i, :] = val
            elif kind == 3:  # duplicated rw row with one cell changed (lookup ambiguity)
                extra = R[:, i : i + 1, :].copy(); extra[c, 0, :] = val
                r = np.ascontiguousarray(np.concatenate([R, extra], axis=1))
            elif kind == 4:
                extra = B[:, i : i + 1, :].copy(); extra[c, 0, :] = val
                b = np.ascontiguousarray(np.concatenate([B, extra], axis=1))
            elif kind == 5:
                flags = 2  # ZK_FLAG_EVM_FIRST_STEP
            yield name, k, s, b, r, flags, int(z[f"{name}/exp_row"][k]), str(z[f"{name}/exp_exc"][k])


def copy_vectors():
    """yield (case, k, dict(copy, copy_flags, rw, rw_flags, tx, tx_flags, bytecode), r, exp_row, exp_exc)"""
    z = np.load(os.path.join(GOLDEN, "copy.npz"))
    r = z["r"]
    for name in z["names"]:
        name = str(name)
        base = {k: z[f"{name}/{k}"] for k in ("copy", "copy_flags", "rw", "rw_flags", "tx", "tx_flags", "bytecode")}
        for k in range(len(z[f"{name}/mut_kind"])):
            kind, i, c = int(z[f"{name}/mut_kind"][k]), int(z[f"{name}/mut_row"][k]), int(z[f"{name}/mut_col"][k])
            val = z[f"{name}/mut_val"][k]
            w = dict(base)
            if kind == 0:
                w["copy"] = base["copy"].copy(); w["copy"][c, i, :] = val
            elif kind == 1:
                w["rw"] = base["rw"].copy(); w["rw"][c, i, :] = val
            elif kind == 2:
                w["tx"] = base["tx"].copy(); w["tx"][c, i, :] = val
            elif kind == 3:
                w["bytecode"] = base["bytecode"].copy(); w["bytecode"][c, i, :] = val
            elif kind == 4:
                w["copy_flags"] = base["copy_flags"].copy(); w["copy_flags"][i] ^= 1
                if not w["copy_flags"][i]:  # Word -> value: the hi half disappears with the type
                    w["copy"] = base["copy"].copy(); w["copy"][4, i, :] = 0
            elif kind == 5 and c == 101:
                w["rw_flags"] = base["rw_flags"].copy(); w["rw_flags"][i] ^= 1
            elif kind == 5 and c == 102:
                extra = base["rw"][:, i : i + 1, :].copy(); extra[8, 0, :] = val
                w["rw"] = np.ascontiguousarray(np.concatenate([base["rw"], extra], axis=1))
                w["rw_flags"] = np.concatenate([base["rw_flags"], base["rw_flags"][i : i + 1]])
            yield name, k, w, r, int(z[f"{name}/exp_row"][k]), str(z[f"{name}/exp_exc"][k])


def state_vectors():
    """yield (case, k, rows, flags, mpt, exp_row, exp_exc)"""
    z = np.load(os.path.join(GOLDEN, "state.npz"))
    for name in z["names"]:
        name = str(name)
        S, F, M = z[f"{name}/rows"], z[f"{name}/flags"], z[f"{name}/mpt"]
        for k in range(len(z[f"{name}/mut_kind"])):
            kind, i, c = int(z[f"{name}/mut_kind"][k]), int(z[f"{name}/mut_row"][k]), int(z[f"{name}/mut_col"][k])
            val = z[f"{name}/mut_val"][k]
            s, f, m = S, F, M
            if kind == 0:
                s = S.copy(); s[c, i, :] = val
            elif kind == 1:
                f = F.copy(); f[i] ^= 1 << (c - 100)
                if not (f[i] >> (c - 100)) & 1:
                    s = S.copy(); s[51 if c == 100 else 53, i, :] = 0
            elif kind == 2:
                m = M.copy(); m[c, i, :] = val
            elif kind == 3:
                s = S.copy(); s[:, [i, i + 1], :] = S[:, [i + 1, i], :]
                f = F.copy(); f[[i, i + 1]] = F[[i + 1, i]]
            yield name, k, s, f, m, int(z[f"{name}/exp_row"][k]), str(z[f"{name}/exp_exc"][k])


def evm2_vectors(part="evm2"):
    """SHA3 / CALLDATACOPY steps: yield (case, k, dict(steps, bytecode, rw, rw_flags, copy, keccak), exp_row, exp_exc)"""
    z = np.load(os.path.join(GOLDEN, part + ".npz"))
    for name in z["names"]:
        name = str(name)
        base = {k: z[f"{name}/{k}"] for k in ("steps", "bytecode", "rw", "rw_flags", "copy", "keccak")}
        for extra in ("tx", "block", "tx_flags", "block_flags", "exp", "aux"):  # ORIGIN / GASPRICE / BlockCtx scenarios carry their context tables
            if f"{name}/{extra}" in z.files:
                base[extra] = z[f"{name}/{extra}"]
        for k in range(len(z[f"{name}/mut_kind"])):
            kind, i, c = int(z[f"{name}/mut_kind"][k]), int(z[f"{name}/mut_row"][k]), int(z[f"{name}/mut_col"][k])
            val = z[f"{name}/mut_val"][k]
            w = dict(base)
            if kind == 0:
                w["steps"] = base["steps"].copy(); w["steps"][c, i, :] = val
            elif kind == 1:
                w["rw"] = base["rw"].copy(); w["rw"][c, i, :] = val
            elif kind == 2:
                w["rw_flags"] = base["rw_flags"].copy(); w["rw_flags"][i] ^= 1
                if not w["rw_flags"][i] & 1:
                    w["rw"] = base["rw"].copy(); w["rw"][9, i, :] = 0
            elif kind == 5:  # duplicate rw row i with another value
                extra = base["rw"][:, i:i + 1, :].copy(); extra[c, 0, :] = val
                w["rw"] = np.ascontiguousarray(np.concatenate([base["rw"], extra], axis=1))
                w["rw_flags"] = np.concatenate([base["rw_flags"], base["rw_flags"][i:i + 1]])
            elif kind == 6:
                w["tx"] = base["tx"].copy(); w["tx"][c, i, :] = val
            elif kind == 7:
                w["block"] = base["block"].copy(); w["block"][c, i, :] = val
            elif kind == 12:
                w["tx_flags"] = base["tx_flags"].copy(); w["tx_flags"][i] ^= 1
            elif kind == 14:
                w["exp"] = base["exp"].copy(); w["exp"][c, i, :] = val
            elif kind == 15:
                w["aux"] = base["aux"].copy(); w["aux"][c, i, :] = val
            elif kind == 13:
                w["block_flags"] = base["block_flags"].copy(); w["block_flags"][i] ^= 1
            elif kind == 3:
                w["copy"] = base["copy"].copy(); w["copy"][c, i, :] = val
            elif kind == 4:
                w["keccak"] = base["keccak"].copy(); w["keccak"][c, i, :] = val
            yield name, k, w, int(z[f"{name}/exp_row"][k]), str(z[f"{name}/exp_exc"][k])


def evm3_vectors():
    """STOP steps (root -> EndTx, internal -> restored caller context); same layout as evm2"""
    return evm2_vectors("evm3")


def exp_vectors():
    """yield (case, k, rows, exp_row, exp_exc)"""
    z = np.load(os.path.join(GOLDEN, "exp.npz"))
    for name in z["names"]:
        name = str(name)
        R = z[f"{name}/rows"]
        for k in range(len(z[f"{name}/mut_row"])):
            i, c = int(z[f"{name}/mut_row"][k]), int(z[f"{name}/mut_col"][k])
            r = R
            if i >= 0:
                r = R.copy(); r[c, i, :] = z[f"{name}/mut_val"][k]
            yield name, k, r, int(z[f"{name}/exp_row"][k]), str(z[f"{name}/exp_exc"][k])


def evm4_vectors():
    """MEMORY steps (MLOAD / MSTORE / MSTORE8, tests/evm/test_memory.py); same layout as evm2"""
    return evm2_vectors("evm4")


def tx_vectors(part="tx"):
    """tx (sig) circuit Fr parts: yield (k, rows[14 (21)][n][4], flags[n], keccak[5][m][4], r limbs, exp_row, exp_exc)"""
    z = np.load(os.path.join(GOLDEN, part + ".npz"))
    R, F, K, r = z["rows"], z["flags"], z["keccak"], z["r"]
    for k in range(len(z["mut_kind"])):
        kind, i, c, val = int(z["mut_kind"][k]), int(z["mut_row"][k]), int(z["mut_col"][k]), z["mut_val"][k]
        rows, flags, kec = R, F, K
        if kind == 0:
            rows = R.copy(); rows[c, i, :] = val
        elif kind == 1:
            flags = F.copy(); flags[i] ^= 1
        elif kind == 2:
            flags = F.copy(); flags[i] ^= 2
        elif kind == 3:
            kec = K.copy(); kec[c, i, :] = val
        yield k, rows, flags, kec, r, int(z["exp_row"][k]), str(z["exp_exc"][k])


def sig_vectors():
    return tx_vectors("sig")


def evm5_vectors():
    """MSIZE / GAS / ISZERO / CMP / JUMP / JUMPI steps; same layout as evm2"""
    return evm2_vectors("evm5")


def evm6_vectors():
    """CALLER / CALLVALUE / CALLDATASIZE / ADDRESS / RETURNDATASIZE / CODESIZE steps; same layout as evm2"""
    return evm2_vectors("evm6")


def evm7_vectors():
    """BITWISE (AND / OR / XOR) / NOT / BYTE steps; same layout as evm2"""
    return evm2_vectors("evm7")


def evm8_vectors():
    """SCMP (SLT / SGT) / SIGNEXTEND steps; same layout as evm2"""
    return evm2_vectors("evm8")


def evm9_vectors():
    """BlockCtx (7 opcodes) / ORIGIN / GASPRICE steps with their block / tx tables; evm2 layout + tx, block"""
    return evm2_vectors("evm9")


def evm10_vectors():
    """SHL / SHR steps; same layout as evm2"""
    return evm2_vectors("evm10")


def evm28_vectors():
    """ErrorGasUintOverflow"""
    return evm2_vectors("evm28")


def evm27_vectors():
    """ErrorOutOfGasPrecompile"""
    return evm2_vectors("evm27")


def evm26_vectors():
    """ErrorOutOfGasCREATE"""
    return evm2_vectors("evm26")


def evm25_vectors():
    """ErrorOutOfGasSloadSstore"""
    return evm2_vectors("evm25")


def evm24_vectors():
    """CREATE / CREATE2"""
    return evm2_vectors("evm24")


def evm23_vectors():
    """CALL_OP"""
    return evm2_vectors("evm23")


def evm22_vectors():
    """ErrorOutOfGasCall"""
    return evm2_vectors("evm22")


def evm21_vectors():
    """RETURN / REVERT"""
    return evm2_vectors("evm21")


def evm20_vectors():
    """ErrorMaxCodeSizeExceeded / ErrorOutOfGasCodeStore / ErrorInvalidCreationCode"""
    return evm2_vectors("evm20")


def evm19_vectors():
    """EXP"""
    return evm2_vectors("evm19")


def evm18_vectors():
    """LOG / ErrorWriteProtection / BLOCKHASH"""
    return evm2_vectors("evm18")


def evm17_vectors():
    """SLOAD / SSTORE / CALLDATALOAD"""
    return evm2_vectors("evm17")


def evm16_vectors():
    """ADDMOD / MULMOD / SDIV_SMOD / SAR"""
    return evm2_vectors("evm16")


def evm15_vectors():
    """CODECOPY / RETURNDATACOPY / EXTCODECOPY and ErrorOutOfGasMemoryCopy"""
    return evm2_vectors("evm15")


def evm14_vectors():
    """BALANCE / EXTCODEHASH / EXTCODESIZE and ErrorOutOfGasAccountAccess"""
    return evm2_vectors("evm14")


def evm13_vectors():
    """out-of-gas / out-of-bound error states (ErrorOutOfGasSHA3 / StaticMemoryExpansion / DynamicMemoryExpansion / LOG / EXP,
    ErrorReturnDataOutOfBound)"""
    return evm2_vectors("evm13")


def evm12_vectors():
    """error states (ErrorStack / ErrorInvalidOpcode / ErrorOutOfGasConstant / ErrorInvalidJump) and SELFBALANCE"""
    return evm2_vectors("evm12")


def evm11_vectors():
    """BeginTx / EndTx / EndBlock steps: yield (case, k, dict(steps, bytecode, rw, rw_flags, copy, keccak, tx, tx_flags,
    block, block_flags, wd, flags = ZK_FLAG_EVM_* of the scenario), exp_row, exp_exc)"""
    z = np.load(os.path.join(GOLDEN, "evm11.npz"))
    for name in z["names"]:
        name = str(name)
        base = {k: z[f"{name}/{k}"] for k in ("steps", "bytecode", "rw", "rw_flags", "copy", "keccak", "tx", "tx_flags", "block",
                                            "block_flags", "wd")}
        first, last = [int(x) for x in z[f"{name}/first_last"]]
        base["flags"] = (2 if first else 0) | (4 if last else 0)
        if last:  # verify_steps(end_with_last_step=True) appends DUMMY_STEP_STATE = StepState(EndBlock, rw_counter=-1)
            dummy = np.zeros((13, 1, 4), dtype=np.uint64)
            dummy[0, 0, 0] = 3
            P = 21888242871839275222246405745257275088548364400416034343698204186575808495617
            dummy[1, 0, :] = [((P - 1) >> (64 * q)) & 0xFFFFFFFFFFFFFFFF for q in range(4)]
            dummy[5, 0, :] = 0
            dummy[8, 0, 0] = 1024
            base["steps"] = np.ascontiguousarray(np.concatenate([base["steps"], dummy], axis=1))
        for k in range(len(z[f"{name}/mut_kind"])):
            kind, i, c = int(z[f"{name}/mut_kind"][k]), int(z[f"{name}/mut_row"][k]), int(z[f"{name}/mut_col"][k])
            val = z[f"{name}/mut_val"][k]
            w = dict(base)
            if kind == 0:
                w["steps"] = base["steps"].copy(); w["steps"][c, i, :] = val
            elif kind == 1:
                w["rw"] = base["rw"].copy(); w["rw"][c, i, :] = val
            elif kind == 2:
                bit = 1 << (c - 100)
                w["rw_flags"] = base["rw_flags"].copy(); w["rw_flags"][i] ^= bit
                if not w["rw_flags"][i] & bit:
                    w["rw"] = base["rw"].copy(); w["rw"][9 if bit == 1 else 11, i, :] = 0
            elif kind == 5:
                extra = base["rw"][:, i:i + 1, :].copy(); extra[c, 0, :] = val
                w["rw"] = np.ascontiguousarray(np.concatenate([base["rw"], extra], axis=1))
                w["rw_flags"] = np.concatenate([base["rw_flags"], base["rw_flags"][i:i + 1]])
            elif kind == 6:
                w["tx"] = base["tx"].copy(); w["tx"][c, i, :] = val
            elif kind == 8:
                w["tx_flags"] = base["tx_flags"].copy(); w["tx_flags"][i] ^= 1
                if not w["tx_flags"][i]:
                    w["tx"] = base["tx"].copy(); w["tx"][4, i, :] = 0
            elif kind == 7:
                if c == 100:
                    w["block_flags"] = base["block_flags"].copy(); w["block_flags"][i] ^= 1
                    if not w["block_flags"][i]:
                        w["block"] = base["block"].copy(); w["block"][3, i, :] = 0
                else:
                    w["block"] = base["block"].copy(); w["block"][c, i, :] = val
            elif kind == 9:
                w["wd"] = base["wd"].copy(); w["wd"][c, i, :] = val
            elif kind == 3:
                w["copy"] = base["copy"].copy(); w["copy"][c, i, :] = val
            elif kind == 4:
                w["keccak"] = base["keccak"].copy(); w["keccak"][c, i, :] = val
            elif kind == 10:
                keep = [q for q in range(base["rw"].shape[1]) if q != i]
                w["rw"] = np.ascontiguousarray(base["rw"][:, keep, :]); w["rw_flags"] = base["rw_flags"][keep]
            yield name, k, w, int(z[f"{name}/exp_row"][k]), str(z[f"{name}/exp_exc"][k])


PI_CASES = ("basic", "full", "one_empty")


def load_pi():
    """public-inputs circuit: pi_<case>.npz merged into one mapping with keys "names" and "<case>/<array>" (one file per
    case keeps each file under 1 MB; the witness rows hold a running RLC that does not compress)"""
    out = {"names": np.array(PI_CASES)}
    for name in PI_CASES:
        z = np.load(os.path.join(GOLDEN, f"pi_{name}.npz"))
        out.update({f"{name}/{k}": z[k] for k in z.files})
    return out


def pi_vectors():
    """public-inputs circuit: yield (case, k, rows[28][n][4], keccak[5][m][4], gas[3][g][4], circuit_len, exp_row, exp_exc);
    the yielded matrices are only valid until the next iteration (corruptions are applied in place and undone)"""
    z = load_pi()
    for name in z["names"]:
        name = str(name)
        R, K, G = z[f"{name}/rows"].copy(), z[f"{name}/keccak"].copy(), z[f"{name}/gas"].copy()
        clen = int(z[f"{name}/circuit_len"][0])
        for k in range(len(z[f"{name}/mut_row"])):
            kind, i, c = int(z[f"{name}/mut_kind"][k]), int(z[f"{name}/mut_row"][k]), int(z[f"{name}/mut_col"][k])
            tgt = (R, K, G)[kind]
            old = None
            if i >= 0:
                old = tgt[c, i, :].copy()
                tgt[c, i, :] = z[f"{name}/mut_val"][k]
            yield name, k, R, K, G, clen, int(z[f"{name}/exp_row"][k]), str(z[f"{name}/exp_exc"][k])
            if old is not None:
                tgt[c, i, :] = old
