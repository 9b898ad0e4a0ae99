package ctmr

// The sets read back out of the device (include/ctmr.h, "the sets read back"): what KnownCertificates.Known()
// (storage/knowncertificates.go:65-96), GetIssuerAndDatesFromCache (storage/filesystemdatabase.go:59-100) and
// cmd/storage-statistics ask Redis for, answered from HBM; and the canonical export / import that moves the state
// into a larger table or a group of another size.
//
// cgo rules: ctmr_set_info holds no pointers, so Go slices of it (and flat []byte / []uint64) are passed for the
// duration of a call.  ctmr_set_export is a table of pointers: it and every array it points to live in C memory.

/*
#include <stdlib.h>
#include "ctmr.h"
*/
import "C"

import (
	"fmt"
	"unsafe"
)

const maxSerial = 39 // CTMR_MAX_SERIAL: octets of raw serial a key record holds

// SetInfo mirrors ctmr_set_info: one live "serials::<expDate>::<issuer>" set.
type SetInfo struct {
	IssuerDigest [32]byte
	ExpHour      int64
	Count        uint64 // SetCardinality
	MemberOff    uint64 // index of the set's first member in an export's member arrays
}

// SetExport is the canonical export: sets by (issuer digest, exp hour), members of a set by first-seen index.
// Member k = Serials[SerialOff[k]:SerialOff[k+1]], first seen at global entry index FirstIndex[k].
type SetExport struct {
	NextIndex  uint64
	Sets       []SetInfo
	Serials    []byte
	SerialOff  []uint64
	FirstIndex []uint64
}

func setInfoFromC(s *C.ctmr_set_info) SetInfo {
	var o SetInfo
	copy(o.IssuerDigest[:], unsafe.Slice((*byte)(unsafe.Pointer(&s.issuer_digest[0])), 32))
	o.ExpHour, o.Count, o.MemberOff = int64(s.exp_hour), uint64(s.count), uint64(s.member_off)
	return o
}

// ListSets returns the live sets with minHour <= exp hour <= maxHour (GetIssuerAndDatesFromCache + Count()).
func (d *DB) ListSets(minHour, maxHour int64) ([]SetInfo, error) {
	var n C.uint64_t
	call := func(out *C.ctmr_set_info, cap C.uint64_t) C.int {
		if d.g != nil {
			return C.ctmr_group_list_sets(d.g, C.int64_t(minHour), C.int64_t(maxHour), out, cap, &n)
		}
		return C.ctmr_list_sets(d.h, C.int64_t(minHour), C.int64_t(maxHour), out, cap, &n)
	}
	if err := d.err(call(nil, 0), "ctmr_list_sets"); err != nil || n == 0 {
		return nil, err
	}
	raw := make([]C.ctmr_set_info, int(n))
	if err := d.err(call(&raw[0], C.uint64_t(len(raw))), "ctmr_list_sets"); err != nil {
		return nil, err
	}
	out := make([]SetInfo, int(n))
	for i := range out {
		out[i] = setInfoFromC(&raw[i])
	}
	return out, nil
}

// SetMembers is KnownCertificates.Known() of one set, from the device: serials and first indices, first-seen order.
func (d *DB) SetMembers(expHour int64, issuerDigest [32]byte) ([][]byte, []uint64, error) {
	var n C.uint64_t
	dp := (*C.uint8_t)(unsafe.Pointer(&issuerDigest[0]))
	call := func(ser *C.uint8_t, serCap C.uint64_t, off, first *C.uint64_t, cap C.uint64_t) C.int {
		if d.g != nil {
			return C.ctmr_group_set_members(d.g, C.int64_t(expHour), dp, ser, serCap, off, first, cap, &n)
		}
		return C.ctmr_set_members(d.h, C.int64_t(expHour), dp, ser, serCap, off, first, cap, &n)
	}
	if err := d.err(call(nil, 0, nil, nil, 0), "ctmr_set_members"); err != nil || n == 0 {
		return nil, nil, err
	}
	k := int(n)
	blob, off, first := make([]byte, k*maxSerial), make([]uint64, k+1), make([]uint64, k)
	rc := call((*C.uint8_t)(unsafe.Pointer(&blob[0])), C.uint64_t(len(blob)), (*C.uint64_t)(unsafe.Pointer(&off[0])),
		(*C.uint64_t)(unsafe.Pointer(&first[0])), C.uint64_t(k))
	if err := d.err(rc, "ctmr_set_members"); err != nil {
		return nil, nil, err
	}
	k = int(n)
	serials := make([][]byte, k)
	for i := range serials {
		serials[i] = append([]byte(nil), blob[off[i]:off[i+1]]...)
	}
	return serials, first[:k], nil
}

func (d *DB) exportCall(x *C.ctmr_set_export) C.int {
	if d.g != nil {
		return C.ctmr_group_export_sets(d.g, x)
	}
	return C.ctmr_export_sets(d.h, x)
}

// ExportSets reads every live set out of the device in canonical form (portable to any table or group size).
func (d *DB) ExportSets() (*SetExport, error) {
	x := (*C.ctmr_set_export)(C.calloc(1, C.size_t(unsafe.Sizeof(C.ctmr_set_export{}))))
	defer C.free(unsafe.Pointer(x))
	if err := d.err(d.exportCall(x), "ctmr_export_sets"); err != nil { // NULL arrays: sizes only
		return nil, err
	}
	ns, nm, nb := int(x.n_sets), int(x.n_members), int(x.serial_bytes)
	x.sets = (*C.ctmr_set_info)(C.calloc(C.size_t(ns+1), C.size_t(unsafe.Sizeof(C.ctmr_set_info{}))))
	x.serials = (*C.uint8_t)(C.malloc(C.size_t(nb + 1)))
	x.serial_off = (*C.uint64_t)(C.malloc(C.size_t(8 * (nm + 1))))
	x.first_index = (*C.uint64_t)(C.malloc(C.size_t(8 * (nm + 1))))
	defer C.free(unsafe.Pointer(x.sets))
	defer C.free(unsafe.Pointer(x.serials))
	defer C.free(unsafe.Pointer(x.serial_off))
	defer C.free(unsafe.Pointer(x.first_index))
	x.sets_cap, x.serials_cap, x.members_cap = C.uint64_t(ns), C.uint64_t(nb), C.uint64_t(nm)
	if err := d.err(d.exportCall(x), "ctmr_export_sets"); err != nil {
		return nil, err
	}
	ns, nm, nb = int(x.n_sets), int(x.n_members), int(x.serial_bytes)
	out := &SetExport{NextIndex: uint64(x.next_index), Sets: make([]SetInfo, ns)}
	cs := unsafe.Slice(x.sets, ns)
	for i := range out.Sets {
		out.Sets[i] = setInfoFromC(&cs[i])
	}
	out.Serials = append([]byte(nil), unsafe.Slice((*byte)(unsafe.Pointer(x.serials)), nb)...)
	out.SerialOff = append([]uint64(nil), unsafe.Slice((*uint64)(unsafe.Pointer(x.serial_off)), nm+1)...)
	out.FirstIndex = append([]uint64(nil), unsafe.Slice((*uint64)(unsafe.Pointer(x.first_index)), nm)...)
	return out, nil
}

// ImportSets loads an export into this EMPTY DB (any table size, any number of GPUs); members keep their first indices.
func (d *DB) ImportSets(e *SetExport) error {
	nm := len(e.FirstIndex)
	if len(e.SerialOff) != nm+1 {
		return fmt.Errorf("ImportSets: SerialOff must have len(FirstIndex)+1 entries")
	}
	x := (*C.ctmr_set_export)(C.calloc(1, C.size_t(unsafe.Sizeof(C.ctmr_set_export{}))))
	defer C.free(unsafe.Pointer(x))
	x.next_index, x.n_sets, x.n_members, x.serial_bytes = C.uint64_t(e.NextIndex), C.uint64_t(len(e.Sets)), C.uint64_t(nm), C.uint64_t(len(e.Serials))
	x.sets = (*C.ctmr_set_info)(C.calloc(C.size_t(len(e.Sets)+1), C.size_t(unsafe.Sizeof(C.ctmr_set_info{}))))
	defer C.free(unsafe.Pointer(x.sets))
	cs := unsafe.Slice(x.sets, len(e.Sets))
	for i, s := range e.Sets {
		copy(unsafe.Slice((*byte)(unsafe.Pointer(&cs[i].issuer_digest[0])), 32), s.IssuerDigest[:])
		cs[i].exp_hour, cs[i].count, cs[i].member_off = C.int64_t(s.ExpHour), C.uint64_t(s.Count), C.uint64_t(s.MemberOff)
	}
	x.serials = (*C.uint8_t)(C.CBytes(append(append([]byte(nil), e.Serials...), 0)))
	defer C.free(unsafe.Pointer(x.serials))
	x.serial_off = (*C.uint64_t)(C.malloc(C.size_t(8 * (nm + 1))))
	defer C.free(unsafe.Pointer(x.serial_off))
	copy(unsafe.Slice((*uint64)(unsafe.Pointer(x.serial_off)), nm+1), e.SerialOff)
	x.first_index = (*C.uint64_t)(C.malloc(C.size_t(8 * (nm + 1))))
	defer C.free(unsafe.Pointer(x.first_index))
	copy(unsafe.Slice((*uint64)(unsafe.Pointer(x.first_index)), nm), e.FirstIndex)
	x.sets_cap, x.serials_cap, x.members_cap = x.n_sets, x.serial_bytes, x.n_members
	if d.g != nil {
		return d.err(C.ctmr_group_import_sets(d.g, x), "ctmr_group_import_sets")
	}
	return d.err(C.ctmr_import_sets(d.h, x), "ctmr_import_sets")
}
