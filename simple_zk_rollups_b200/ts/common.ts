// Drop-in replacement for operator/src/snarks/common.ts of kendricktan/simple-zk-rollups.
// SOURCE ONLY here (no node in the build image).  Same exports, same return shape; the lines that
// change are marked.  Witness generation and the Solidity formatting are the
// reference's own code, untouched; the isValid self-check keeps its place and its exception but calls zkr.verify.
import * as path from "path";
import * as compiler from "circom";
import * as crypto from "crypto";

import { Circuit, groth } from "snarkjs";
import { binarifyWitness, binarifyProvingKey } from "../utils/binarify";
import { SNARK_FIELD_SIZE } from "../utils/crypto";
import { stringifyBigInts, unstringifyBigInts } from "../utils/helpers";

// CHANGED (was: import { buildBn128 } from "websnark")
const zkr = require("./zkr_napi.node");

const le32ToDecimal = (u8: Uint8Array, off: number): string => {
  let v = BigInt(0);
  for (let i = 31; i >= 0; i--) v = (v << BigInt(8)) | BigInt(u8[off + i]);
  return v.toString();
};

// websnark draws r and s internally; the addon takes them explicitly (pass zeros for the snarkjs debug mode)
const randomScalar = (): Uint8Array => {
  const r = BigInt(SNARK_FIELD_SIZE.toString());
  for (;;) {
    const b = crypto.randomBytes(32);
    b[31] &= 0x3f;
    let v = BigInt(0);
    for (let i = 31; i >= 0; i--) v = (v << BigInt(8)) | BigInt(b[i]);
    if (v < r) return new Uint8Array(b);
  }
};

export const createProofGenerator = (provingKey, verifyingKey, circuitName) => {
  // CHANGED: the key is binarified and uploaded ONCE (the reference re-encodes it on every proof, common.ts:28)
  const key = zkr.loadKey(binarifyProvingKey(provingKey));
  // CHANGED: the verifying key's IC tables are uploaded once; the self-check below runs in libzkr (zkr_verify)
  const vkey = zkr.loadVerifyingKey(Buffer.from(JSON.stringify(stringifyBigInts(verifyingKey))));

  return async circuitInputs => {
    const circuitDef = await compiler(
      path.join(__dirname, `../../../prover/circuits/${circuitName}`)
    );
    const circuit = new Circuit(circuitDef);

    const witness = circuit.calculateWitness(stringifyBigInts(circuitInputs));
    const publicSignals = witness.slice(
      1,
      circuit.nPubInputs + circuit.nOutputs + 1
    );

    // CHANGED (was: buildBn128() + wasmBn128.groth16GenProof(witnessBin, provingKeyBin))
    const witnessBin = binarifyWitness(witness);
    const p: Uint8Array = await zkr.prove(key, witnessBin, randomScalar(), randomScalar());
    const d = (i: number) => le32ToDecimal(p, 32 * i);
    const proof = {
      pi_a: [d(0), d(1), "1"],
      pi_b: [[d(2), d(3)], [d(4), d(5)], ["1", "0"]],
      pi_c: [d(6), d(7), "1"],
      protocol: "groth"
    };

    // CHANGED (was: groth.isValid(vk, proof, publicSignals) on the JS BigInt path, seconds per call):
    // same acceptance predicate as contracts/contracts/TxVerifier.sol:258-276
    const isValid = zkr.verify(vkey, p, binarifyWitness(publicSignals));

    if (!isValid) {
      throw new Error("Invalid proof generated");
    }

    return {
      proof,
      solidityProof: {
        a: stringifyBigInts(proof.pi_a).slice(0, 2),
        b: stringifyBigInts(proof.pi_b)
          .map(x => x.reverse())
          .slice(0, 2),
        c: stringifyBigInts(proof.pi_c).slice(0, 2),
        inputs: publicSignals.map(x => x.mod(SNARK_FIELD_SIZE).toString())
      }
    };
  };
};

// snarkjs-shaped entry point named by the north star: genProof(provingKey, witness)
const keyCache = new Map<any, any>();
export const genProof = async (provingKey, witness, r?: Uint8Array, s?: Uint8Array) => {
  if (!keyCache.has(provingKey)) keyCache.set(provingKey, zkr.loadKey(binarifyProvingKey(provingKey)));
  const p: Uint8Array = await zkr.prove(keyCache.get(provingKey), binarifyWitness(witness),
    r || randomScalar(), s || randomScalar());
  const d = (i: number) => le32ToDecimal(p, 32 * i);
  return {
    proof: { pi_a: [d(0), d(1), "1"], pi_b: [[d(2), d(3)], [d(4), d(5)], ["1", "0"]], pi_c: [d(6), d(7), "1"], protocol: "groth" },
    publicSignals: witness.slice(1, provingKey.nPublic + 1)
  };
};

// Many witnesses of one circuit in one pass on the GPU (zkr_prove_many): key = a zkr.loadKey handle, witnesses =
// binarifyWitness outputs, rs = optional (r|s) pairs of 64 bytes (absent: fresh CSPRNG pairs in libzkr).
// -> one 256-byte proof per witness, in input order.
export const proveMany = async (key, witnesses: ArrayBuffer[], rs?: Uint8Array[]): Promise<Uint8Array[]> => {
  const wb = witnesses.length ? witnesses[0].byteLength : 0;
  const all = new Uint8Array(wb * witnesses.length);
  witnesses.forEach((w, j) => all.set(new Uint8Array(w), wb * j));
  let rsAll: Uint8Array | undefined;
  if (rs) {
    rsAll = new Uint8Array(64 * rs.length);
    rs.forEach((x, j) => rsAll.set(x, 64 * j));
  }
  const p: Uint8Array = await zkr.proveMany(key, all.buffer, rsAll);
  return witnesses.map((_, j) => p.subarray(256 * j, 256 * (j + 1)));
};
