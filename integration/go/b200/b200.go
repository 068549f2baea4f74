// Source a maintainer adds to gnark-whir (or to a gnark fork) to put libb200g16 behind gnark's groth16 API.
// NOT built or tested in this repository: the image has no Go toolchain (see INTEGRATION.md).  The same C-ABI,
// call for call, is exercised by gnark_whir_b200/lib.py + groth16.py in the test-suite.
//go:build b200

package b200

/*
#cgo CFLAGS: -I${SRCDIR}/../../../../include
#cgo LDFLAGS: -lb200g16
#include "b200g16.h"
*/
import "C"

import (
	"errors"
	"fmt"
	"math/big"
	"math/bits"
	"runtime"
	"unsafe"

	"github.com/consensys/gnark-crypto/ecc"
	curve "github.com/consensys/gnark-crypto/ecc/bn254"
	"github.com/consensys/gnark-crypto/ecc/bn254/fr"
	"github.com/consensys/gnark-crypto/ecc/bn254/fr/hash_to_field"
	"github.com/consensys/gnark/backend"
	groth16_bn254 "github.com/consensys/gnark/backend/groth16/bn254"
	"github.com/consensys/gnark/backend/witness"
	"github.com/consensys/gnark/constraint"
	cs "github.com/consensys/gnark/constraint/bn254"
	"github.com/consensys/gnark/constraint/solver"
	fcs "github.com/consensys/gnark/frontend/cs"
)

// ProvingKey = gnark's pk + lazily created device handles (like icicle's deviceInfo).
type ProvingKey struct {
	groth16_bn254.ProvingKey
	ctx       *C.b200g16_ctx
	dev       *C.b200g16_pk
	pedBasis  []*C.b200g16_bases // pk.CommitmentKeys[i].Basis
	pedSigma  []*C.b200g16_bases // pk.CommitmentKeys[i].BasisExpSigma
	owned     []*C.b200g16_bases // resident vectors Setup made and the device key borrows
}

func u64(p unsafe.Pointer) *C.uint64_t { return (*C.uint64_t)(p) }

func boolsToBytes(b []bool) []byte {
	out := make([]byte, len(b))
	for i, v := range b {
		if v {
			out[i] = 1
		}
	}
	return out
}

// lastError runs one C call and fetches its error text on the SAME OS thread: b200g16_last_error() is thread-local,
// and the Go scheduler may move a goroutine between two cgo calls.
func call(f func() C.int) error {
	runtime.LockOSThread()
	defer runtime.UnlockOSThread()
	if st := f(); st != 0 {
		return errors.New(C.GoString(C.b200g16_last_error()))
	}
	return nil
}

// setup uploads the key once; every slice is passed zero-copy (gnark-crypto's in-memory
// layout IS the ABI layout: fr/fp.Element = [4]uint64 Montgomery, G1Affine{X,Y}, G2Affine{X{A0,A1},Y{A0,A1}}).
func (pk *ProvingKey) setup(r1cs *cs.R1CS) error {
	if pk.dev != nil {
		return nil
	}
	if err := call(func() C.int { return C.b200g16_init(0, &pk.ctx) }); err != nil {
		return err // no CPU fallback: the caller decides what to do
	}
	nbWires := len(pk.InfinityA)
	// k_skip: wires that are NOT in the K MSM = public wires + BSB22 committed wires + commitment wires
	kSkip := make([]byte, nbWires)
	for i := 0; i < r1cs.GetNbPublicVariables(); i++ {
		kSkip[i] = 1
	}
	commitmentInfo := r1cs.CommitmentInfo.(constraint.Groth16Commitments)
	for _, c := range commitmentInfo {
		kSkip[c.CommitmentIndex] = 1
		for _, w := range c.PrivateCommitted {
			kSkip[w] = 1
		}
	}
	infA, infB := boolsToBytes(pk.InfinityA), boolsToBytes(pk.InfinityB)
	// cgo: a struct passed to C may not hold unpinned Go pointers -> pin every array for the duration of the call
	var pin runtime.Pinner
	defer pin.Unpin()
	g1 := func(v []curve.G1Affine) *C.uint64_t {
		if len(v) == 0 {
			return nil
		}
		pin.Pin(&v[0])
		return u64(unsafe.Pointer(&v[0]))
	}
	bytesPtr := func(v []byte) *C.uint8_t {
		pin.Pin(&v[0])
		return (*C.uint8_t)(unsafe.Pointer(&v[0]))
	}
	var g2b *C.uint64_t
	if len(pk.G2.B) > 0 {
		pin.Pin(&pk.G2.B[0])
		g2b = u64(unsafe.Pointer(&pk.G2.B[0]))
	}
	pin.Pin(&pk.G1.Alpha)
	pin.Pin(&pk.G1.Beta)
	pin.Pin(&pk.G1.Delta)
	pin.Pin(&pk.G2.Beta)
	pin.Pin(&pk.G2.Delta)
	d := C.b200g16_pk_desc{
		log2_domain: C.uint(bits.TrailingZeros64(pk.Domain.Cardinality)),
		n_wires:     C.size_t(nbWires),
		g1_a:        g1(pk.G1.A), n_a: C.size_t(len(pk.G1.A)),
		g1_b:        g1(pk.G1.B), n_b: C.size_t(len(pk.G1.B)),
		g1_k:        g1(pk.G1.K), n_k: C.size_t(len(pk.G1.K)),
		g1_z:        g1(pk.G1.Z), n_z: C.size_t(len(pk.G1.Z)),
		g2_b:        g2b,
		g1_alpha:    u64(unsafe.Pointer(&pk.G1.Alpha)), g1_beta: u64(unsafe.Pointer(&pk.G1.Beta)),
		g1_delta:    u64(unsafe.Pointer(&pk.G1.Delta)),
		g2_beta:     u64(unsafe.Pointer(&pk.G2.Beta)), g2_delta: u64(unsafe.Pointer(&pk.G2.Delta)),
		infinity_a:  bytesPtr(infA), infinity_b: bytesPtr(infB), k_skip: bytesPtr(kSkip),
		precompute: 1, // window tables over A, B1, K, Z, B2 (13 instead of 15-17 additions per point; ~13x the
		// key's HBM footprint; identical proofs) — drop it when the key does not fit
	}
	if err := call(func() C.int { return C.b200g16_pk_upload(pk.ctx, &d, &pk.dev) }); err != nil {
		return err
	}
	for i := range pk.CommitmentKeys {
		ck := &pk.CommitmentKeys[i]
		var b, s *C.b200g16_bases
		if err := call(func() C.int {
			return C.b200g16_bases_upload_g1(pk.ctx, u64(unsafe.Pointer(&ck.Basis[0])), C.size_t(len(ck.Basis)), &b)
		}); err != nil {
			return err
		}
		if err := call(func() C.int {
			return C.b200g16_bases_upload_g1(pk.ctx, u64(unsafe.Pointer(&ck.BasisExpSigma[0])), C.size_t(len(ck.BasisExpSigma)), &s)
		}); err != nil {
			return err
		}
		pk.pedBasis, pk.pedSigma = append(pk.pedBasis, b), append(pk.pedSigma, s)
	}
	return nil
}

func msmG1(ctx *C.b200g16_ctx, bases *C.b200g16_bases, scalars []fr.Element) (curve.G1Affine, error) {
	var out curve.G1Affine
	var p *C.uint64_t
	if len(scalars) > 0 {
		p = u64(unsafe.Pointer(&scalars[0]))
	}
	err := call(func() C.int {
		return C.b200g16_msm_g1(ctx, bases, 0, p, C.size_t(len(scalars)), u64(unsafe.Pointer(&out)))
	})
	return out, err
}

// solve runs gnark's solver with the BSB22 hint overridden: identical to gnark's, except Commit() is the GPU MSM on the
// resident basis.  commitments receives one point per commitment; the committed private values are returned for the
// proofs of knowledge.
func solve(r1cs *cs.R1CS, pk *ProvingKey, opt backend.ProverConfig, fullWitness witness.Witness,
	commitments []curve.G1Affine) (*cs.R1CSSolution, [][]fr.Element, error) {
	commitmentInfo := r1cs.CommitmentInfo.(constraint.Groth16Commitments)
	privateCommittedValues := make([][]fr.Element, len(commitmentInfo))
	solverOpts := opt.SolverOpts[:len(opt.SolverOpts):len(opt.SolverOpts)]
	bsb22ID := solver.GetHintID(fcs.Bsb22CommitmentComputePlaceholder)
	solverOpts = append(solverOpts, solver.OverrideHint(bsb22ID, func(_ *big.Int, in []*big.Int, out []*big.Int) error {
		i := int(in[0].Int64())
		in = in[1:]
		privateCommittedValues[i] = make([]fr.Element, len(commitmentInfo[i].PrivateCommitted))
		hashed := in[:len(commitmentInfo[i].PublicAndCommitmentCommitted)]
		committed := in[len(hashed):]
		for j, inJ := range committed {
			privateCommittedValues[i][j].SetBigInt(inJ)
		}
		var err error
		if commitments[i], err = msmG1(pk.ctx, pk.pedBasis[i], privateCommittedValues[i]); err != nil {
			return err
		}
		opt.HashToFieldFn.Write(constraint.SerializeCommitment(commitments[i].Marshal(), hashed, (fr.Bits-1)/8+1))
		hashBts := opt.HashToFieldFn.Sum(nil)
		opt.HashToFieldFn.Reset()
		nbBuf := fr.Bytes
		if opt.HashToFieldFn.Size() < fr.Bytes {
			nbBuf = opt.HashToFieldFn.Size()
		}
		var res fr.Element
		res.SetBytes(hashBts[:nbBuf])
		res.BigInt(out[0])
		return nil
	}))

	_solution, err := r1cs.Solve(fullWitness, solverOpts...) // Go, CPU (out of scope)
	if err != nil {
		return nil, nil, err
	}
	return _solution.(*cs.R1CSSolution), privateCommittedValues, nil
}

// Prove has gnark's signature: groth16.Prove(ccs, pk, fullWitness, opts...) at mt.go:496.  The body follows gnark
// v0.11.0 backend/groth16/bn254/prove.go; what changes is where the arithmetic runs.
func Prove(r1cs *cs.R1CS, pk *ProvingKey, fullWitness witness.Witness, opts ...backend.ProverOption) (*groth16_bn254.Proof, error) {
	opt, err := backend.NewProverConfig(opts...)
	if err != nil {
		return nil, fmt.Errorf("new prover config: %w", err)
	}
	if opt.HashToFieldFn == nil {
		opt.HashToFieldFn = hash_to_field.New([]byte(constraint.CommitmentDst))
	}
	if err := pk.setup(r1cs); err != nil {
		return nil, err
	}

	commitmentInfo := r1cs.CommitmentInfo.(constraint.Groth16Commitments)
	proof := &groth16_bn254.Proof{Commitments: make([]curve.G1Affine, len(commitmentInfo))}
	solution, privateCommittedValues, err := solve(r1cs, pk, opt, fullWitness, proof.Commitments)
	if err != nil {
		return nil, err
	}
	wireValues := []fr.Element(solution.W)

	// Pedersen proofs of knowledge (gnark: ProveKnowledge per key): one MSM per commitment on BasisExpSigma,
	// folded with the "G16-BSB22" challenge exactly as upstream.  Nothing before the fold needs their results, so the
	// first three are only ENQUEUED here (b200g16_msm_g1_begin: three tickets per ctx) and collected after
	// b200g16_prove — their bucket reductions run under the prove's first MSM; further keys take the synchronous call.
	poks := make([]curve.G1Affine, len(pk.CommitmentKeys))
	tickets := make([]C.int, len(pk.CommitmentKeys))
	var pokPin runtime.Pinner // _begin keeps reading the scalars after it returns (registered memory is copied asynchronously)
	defer pokPin.Unpin()
	for i := range pk.CommitmentKeys {
		tickets[i] = -1
		if i < 3 && len(privateCommittedValues[i]) > 0 {
			v := privateCommittedValues[i]
			pokPin.Pin(&v[0])
			if err = call(func() C.int {
				return C.b200g16_msm_g1_begin(pk.ctx, pk.pedSigma[i], 0, u64(unsafe.Pointer(&v[0])), C.size_t(len(v)), &tickets[i])
			}); err != nil {
				return nil, err
			}
			continue
		}
		if poks[i], err = msmG1(pk.ctx, pk.pedSigma[i], privateCommittedValues[i]); err != nil {
			return nil, err
		}
	}
	collectPoks := func() error {
		for i, t := range tickets {
			if t < 0 {
				continue
			}
			if err := call(func() C.int { return C.b200g16_msm_g1_end(pk.ctx, t, u64(unsafe.Pointer(&poks[i]))) }); err != nil {
				return err
			}
			tickets[i] = -1
		}
		return nil
	}
	defer collectPoks() // an early return must not leave tickets open
	commitmentsSerialized := make([]byte, fr.Bytes*len(commitmentInfo))
	for i := range commitmentInfo {
		copy(commitmentsSerialized[fr.Bytes*i:], wireValues[commitmentInfo[i].CommitmentIndex].Marshal())
	}
	challenge, err := fr.Hash(commitmentsSerialized, []byte("G16-BSB22"), 1)
	if err != nil {
		return nil, err
	}

	// r, s: gnark samples them here; they are explicit in the ABI so CPU and GPU proofs can be compared bit for bit
	var _r, _s fr.Element
	if _, err := _r.SetRandom(); err != nil {
		return nil, err
	}
	if _, err := _s.SetRandom(); err != nil {
		return nil, err
	}

	var out C.b200g16_proof
	err = call(func() C.int {
		return C.b200g16_prove(pk.ctx, pk.dev,
			u64(unsafe.Pointer(&wireValues[0])), C.size_t(len(wireValues)),
			u64(unsafe.Pointer(&solution.A[0])), u64(unsafe.Pointer(&solution.B[0])), u64(unsafe.Pointer(&solution.C[0])),
			C.size_t(len(solution.A)),
			u64(unsafe.Pointer(&_r)), u64(unsafe.Pointer(&_s)), &out, nil)
	})
	if err != nil {
		return nil, err
	}
	if err = collectPoks(); err != nil {
		return nil, err
	}
	if _, err = proof.CommitmentPok.Fold(poks, challenge[0], ecc.MultiExpConfig{NbTasks: 1}); err != nil {
		return nil, err
	}
	proof.Ar = *(*curve.G1Affine)(unsafe.Pointer(&out.ar))
	proof.Bs = *(*curve.G2Affine)(unsafe.Pointer(&out.bs))
	proof.Krs = *(*curve.G1Affine)(unsafe.Pointer(&out.krs))
	return proof, nil
}

// BatchProve proves k witnesses of one circuit: proof j equals Prove(r1cs, pk, witnesses[j], opts...) with the same
// r, s.  Each witness is solved as Prove solves it (the BSB22 commitment stays one GPU MSM inside each solve, since the
// hint's answer feeds the rest of that solve); the proofs of knowledge of all k witnesses are one
// b200g16_msm_g1_batch per commitment key, and the k proves one b200g16_prove_batch call.
func BatchProve(r1cs *cs.R1CS, pk *ProvingKey, witnesses []witness.Witness, opts ...backend.ProverOption) ([]*groth16_bn254.Proof, error) {
	opt, err := backend.NewProverConfig(opts...)
	if err != nil {
		return nil, fmt.Errorf("new prover config: %w", err)
	}
	if opt.HashToFieldFn == nil {
		opt.HashToFieldFn = hash_to_field.New([]byte(constraint.CommitmentDst))
	}
	if err := pk.setup(r1cs); err != nil {
		return nil, err
	}
	k := len(witnesses)
	if k == 0 {
		return nil, nil
	}
	commitmentInfo := r1cs.CommitmentInfo.(constraint.Groth16Commitments)
	proofs := make([]*groth16_bn254.Proof, k)
	committed := make([][][]fr.Element, k)
	var wires, A, B, Cv []fr.Element
	for j, w := range witnesses {
		proofs[j] = &groth16_bn254.Proof{Commitments: make([]curve.G1Affine, len(commitmentInfo))}
		solution, pcv, err := solve(r1cs, pk, opt, w, proofs[j].Commitments)
		if err != nil {
			return nil, err
		}
		committed[j] = pcv
		wires = append(wires, solution.W...)
		A = append(A, solution.A...)
		B = append(B, solution.B...)
		Cv = append(Cv, solution.C...)
	}
	nWires, nCons := len(wires)/k, len(A)/k

	// proofs of knowledge: for each commitment key, the k witnesses' committed values as one batch MSM
	poks := make([][]curve.G1Affine, k)
	for j := range poks {
		poks[j] = make([]curve.G1Affine, len(pk.CommitmentKeys))
	}
	for i := range pk.CommitmentKeys {
		n := len(committed[0][i])
		if n == 0 {
			continue
		}
		rows := make([]fr.Element, 0, k*n)
		for j := 0; j < k; j++ {
			rows = append(rows, committed[j][i]...)
		}
		out := make([]curve.G1Affine, k)
		if err := call(func() C.int {
			return C.b200g16_msm_g1_batch(pk.ctx, pk.pedSigma[i], 0, u64(unsafe.Pointer(&rows[0])), C.size_t(n), C.size_t(k),
				u64(unsafe.Pointer(&out[0])))
		}); err != nil {
			return nil, err
		}
		for j := 0; j < k; j++ {
			poks[j][i] = out[j]
		}
	}

	rs, ss := make([]fr.Element, k), make([]fr.Element, k)
	for j := 0; j < k; j++ {
		if _, err := rs[j].SetRandom(); err != nil {
			return nil, err
		}
		if _, err := ss[j].SetRandom(); err != nil {
			return nil, err
		}
	}
	out := make([]C.b200g16_proof, k)
	err = call(func() C.int {
		return C.b200g16_prove_batch(pk.ctx, pk.dev, C.size_t(k), u64(unsafe.Pointer(&wires[0])), C.size_t(nWires),
			u64(unsafe.Pointer(&A[0])), u64(unsafe.Pointer(&B[0])), u64(unsafe.Pointer(&Cv[0])), C.size_t(nCons),
			u64(unsafe.Pointer(&rs[0])), u64(unsafe.Pointer(&ss[0])), &out[0])
	})
	if err != nil {
		return nil, err
	}
	for j := 0; j < k; j++ {
		commitmentsSerialized := make([]byte, fr.Bytes*len(commitmentInfo))
		for i := range commitmentInfo {
			copy(commitmentsSerialized[fr.Bytes*i:], wires[j*nWires+commitmentInfo[i].CommitmentIndex].Marshal())
		}
		challenge, err := fr.Hash(commitmentsSerialized, []byte("G16-BSB22"), 1)
		if err != nil {
			return nil, err
		}
		if _, err = proofs[j].CommitmentPok.Fold(poks[j], challenge[0], ecc.MultiExpConfig{NbTasks: 1}); err != nil {
			return nil, err
		}
		proofs[j].Ar = *(*curve.G1Affine)(unsafe.Pointer(&out[j].ar))
		proofs[j].Bs = *(*curve.G2Affine)(unsafe.Pointer(&out[j].bs))
		proofs[j].Krs = *(*curve.G1Affine)(unsafe.Pointer(&out[j].krs))
	}
	return proofs, nil
}

// Pin registers the witness-sized Go slices once (cudaHostRegister): H2D copies from unregistered (pageable) Go
// memory run at a fraction of PCIe speed (bench.py: e2e_pageable vs e2e).  Call Unpin before the slice is dropped.
func Pin(v []fr.Element) error {
	if len(v) == 0 {
		return nil
	}
	return call(func() C.int { return C.b200g16_host_register(unsafe.Pointer(&v[0]), C.size_t(len(v))*C.size_t(fr.Bytes)) })
}

func Unpin(v []fr.Element) error {
	if len(v) == 0 {
		return nil
	}
	return call(func() C.int { return C.b200g16_host_unregister(unsafe.Pointer(&v[0])) })
}

// Free releases the device copy of the key.
func (pk *ProvingKey) Free() {
	for i := range pk.pedBasis {
		C.b200g16_bases_free(pk.pedBasis[i])
		C.b200g16_bases_free(pk.pedSigma[i])
	}
	pk.pedBasis, pk.pedSigma = nil, nil
	if pk.dev != nil {
		C.b200g16_pk_free(pk.dev)
		pk.dev = nil
	}
	for _, b := range pk.owned {
		C.b200g16_bases_free(b)
	}
	pk.owned = nil
	if pk.ctx != nil {
		C.b200g16_destroy(pk.ctx)
		pk.ctx = nil
	}
}
