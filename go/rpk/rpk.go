// Package rpk is the cgo binding of include/rpk.h: the B200 batch engine behind the RunPod virtual
// kubelet's two data-parallel loops (GetGPUTypes filter/sort/top-5 and the updateAllPodStatuses diff).
//
// NOT BUILT IN THIS REPOSITORY'S CI: the build image has no Go toolchain (SURVEY.md 8c), so this file is
// shipped gofmt-clean by inspection and exercised only through the identical C-ABI from C++ and Python
// (tests/).  Build (on a machine with Go >= 1.24 and CUDA 12.9):
//
//	CGO_ENABLED=1 CGO_CFLAGS="-I${REPO}/include" \
//	CGO_LDFLAGS="-L${REPO}/k8s-runpod-kubelet_b200/lib -lrpk -Wl,-rpath,${REPO}/k8s-runpod-kubelet_b200/lib" go build ./...
package rpk

/*
#include <stdlib.h>
#include "rpk.h"
*/
import "C"

import (
	"fmt"
	"runtime"
	"sync"
	"unsafe"
)

// Cloud column values (validateCloudType's result, runpod_client.go:1115-1134).
const (
	CloudSecure    uint8 = C.RPK_CLOUD_SECURE
	CloudCommunity uint8 = C.RPK_CLOUD_COMMUNITY
)

// DefaultMaxPrice mirrors runpod_client.go:48.
const DefaultMaxPrice = 0.5

// TopK mirrors "Take up to 5 GPUs" (runpod_client.go:502-509).
const TopK = C.RPK_TOPK

// Offers is []GPUType (runpod_client.go:83-95) as struct-of-arrays; IDs stay on the host, index = offer id.
type Offers struct {
	IDs            []string
	MemoryInGb     []int32
	VCPU           []int32 // optional extension column (nil = all 0)
	RAMGb          []int32 // optional extension column (nil = all 0)
	SecurePrice    []float64
	CommunityPrice []float64
	Flags          []uint8 // bit0 SecureCloud, bit1 CommunityCloud
}

// Pods is the (minRAMPerGPU, cloudType, maxPrice) triple of PrepareRunPodParameters
// (runpod_client.go:1261-1281) for a batch of pods, plus the two extension columns.
type Pods struct {
	ReqMemGb []int32
	ReqVCPU  []int32   // nil = 0
	ReqRAMGb []int32   // nil = 0
	MaxPrice []float64 // nil = DefaultMaxPrice for every pod (the reference's only behaviour)
	Cloud    []uint8   // nil = SECURE
}

// Engine owns one rpk_ctx.  A ctx is not re-entrant; at least four goroutines reach it in the provider
// (pod-sync worker, pending-pod processor, NotifyPods ticker, periodic ticker: kubelet.go:384,734,718,292),
// so every method takes mu.
type Engine struct {
	mu  sync.Mutex
	ctx *C.rpk_ctx
	g   int
}

func lastError(ctx *C.rpk_ctx, rc C.int) error {
	return fmt.Errorf("rpk: error %d: %s", int(rc), C.GoString(C.rpk_last_error(ctx)))
}

// New creates a ctx over nGPUs devices (0..nGPUs-1).  There is no CPU fallback: without a usable sm_100
// GPU this fails and the provider must refuse to start.
func New(nGPUs int) (*Engine, error) {
	var ctx *C.rpk_ctx
	if rc := C.rpk_create(C.int(nGPUs), nil, &ctx); rc != C.RPK_OK {
		return nil, lastError(nil, rc)
	}
	e := &Engine{ctx: ctx}
	runtime.SetFinalizer(e, func(e *Engine) { e.Close() })
	return e, nil
}

// Close releases the ctx and all device memory.
func (e *Engine) Close() {
	e.mu.Lock()
	defer e.mu.Unlock()
	if e.ctx != nil {
		C.rpk_destroy(e.ctx)
		e.ctx = nil
	}
}

func i32p(s []int32) *C.int32_t {
	if len(s) == 0 {
		return nil
	}
	return (*C.int32_t)(unsafe.Pointer(&s[0]))
}

func f64p(s []float64) *C.double {
	if len(s) == 0 {
		return nil
	}
	return (*C.double)(unsafe.Pointer(&s[0]))
}

func u8p(s []uint8) *C.uint8_t {
	if len(s) == 0 {
		return nil
	}
	return (*C.uint8_t)(unsafe.Pointer(&s[0]))
}

// UploadOffers replaces the per-pod GraphQL decode of gpuTypes (runpod_client.go:447-455): upload the
// table once per refresh, select against it for every batch.  The slices are only read during the call
// (cgo pointer rule: C retains nothing).
func (e *Engine) UploadOffers(o *Offers) error {
	e.mu.Lock()
	defer e.mu.Unlock()
	g := len(o.MemoryInGb)
	if len(o.SecurePrice) != g || len(o.CommunityPrice) != g || len(o.Flags) != g {
		return fmt.Errorf("rpk: offer columns differ in length")
	}
	rc := C.rpk_offers_upload(e.ctx, C.uint32_t(g), i32p(o.MemoryInGb), i32p(o.VCPU), i32p(o.RAMGb),
		f64p(o.SecurePrice), f64p(o.CommunityPrice), u8p(o.Flags))
	if rc != C.RPK_OK {
		return lastError(e.ctx, rc)
	}
	e.g = g
	return nil
}

// Select evaluates GetGPUTypes (runpod_client.go:465-509) for every pod of the batch at once.
// best[p] is the cheapest feasible offer index (-1 = none); top5, if wantTop5, is the whole gpuTypeIds
// list per pod (-1 padded).
func (e *Engine) Select(p *Pods, wantTop5 bool) (best []int32, top5 []int32, err error) {
	e.mu.Lock()
	defer e.mu.Unlock()
	n := len(p.ReqMemGb)
	best = make([]int32, n)
	if n == 0 {
		return best, nil, nil
	}
	var t5 *C.int32_t
	if wantTop5 {
		top5 = make([]int32, n*TopK)
		t5 = i32p(top5)
	}
	rc := C.rpk_select(e.ctx, C.uint32_t(n), i32p(p.ReqMemGb), i32p(p.ReqVCPU), i32p(p.ReqRAMGb),
		f64p(p.MaxPrice), u8p(p.Cloud), i32p(best), t5)
	if rc != C.RPK_OK {
		return nil, nil, lastError(e.ctx, rc)
	}
	return best, top5, nil
}

// MaxOfferSets is the most offer sets one UploadOfferSets call holds; SetAll marks an unrestricted row.
const (
	MaxOfferSets        = C.RPK_MAX_OFFER_SETS
	SetAll       uint16 = C.RPK_SET_ALL
)

func u16p(s []uint16) *C.uint16_t {
	if len(s) == 0 {
		return nil
	}
	return (*C.uint16_t)(unsafe.Pointer(&s[0]))
}

// UploadOfferSets replaces every offer set: set s holds the offer indices sets[s] of the resident table (indices
// outside [0, G) are ignored).  A later UploadOffers makes the sets stale (SelectSets then fails until they are
// uploaded again).  len(sets) = 0 clears them.
func (e *Engine) UploadOfferSets(sets [][]int32) error {
	e.mu.Lock()
	defer e.mu.Unlock()
	if len(sets) > MaxOfferSets {
		return fmt.Errorf("rpk: %d offer sets, at most %d per upload", len(sets), MaxOfferSets)
	}
	w := (e.g + 31) / 32
	words := make([]uint32, len(sets)*w)
	for s, members := range sets {
		for _, g := range members {
			if g >= 0 && int(g) < e.g {
				words[s*w+int(g)/32] |= 1 << (uint(g) & 31)
			}
		}
	}
	var wp *C.uint32_t
	if len(words) > 0 {
		wp = (*C.uint32_t)(unsafe.Pointer(&words[0]))
	}
	if rc := C.rpk_offer_sets_upload(e.ctx, C.uint32_t(len(sets)), C.uint32_t(e.g), wp); rc != C.RPK_OK {
		return lastError(e.ctx, rc)
	}
	return nil
}

// SelectSets is Select with pod p restricted to offer set setID[p] (SetAll = the whole table; an id without a set
// = nothing feasible): GetGPUTypes over the set's members only, indices into the whole table.
func (e *Engine) SelectSets(p *Pods, setID []uint16, wantTop5 bool) (best []int32, top5 []int32, err error) {
	e.mu.Lock()
	defer e.mu.Unlock()
	n := len(p.ReqMemGb)
	best = make([]int32, n)
	if n == 0 {
		return best, nil, nil
	}
	if setID != nil && len(setID) != n {
		return nil, nil, fmt.Errorf("rpk: %d set ids for %d pods", len(setID), n)
	}
	var t5 *C.int32_t
	if wantTop5 {
		top5 = make([]int32, n*TopK)
		t5 = i32p(top5)
	}
	rc := C.rpk_select_sets(e.ctx, C.uint32_t(n), i32p(p.ReqMemGb), i32p(p.ReqVCPU), i32p(p.ReqRAMGb),
		f64p(p.MaxPrice), u8p(p.Cloud), u16p(setID), i32p(best), t5)
	if rc != C.RPK_OK {
		return nil, nil, lastError(e.ctx, rc)
	}
	return best, top5, nil
}

// StatusDiff is the batched predicate of updateAllPodStatuses (kubelet.go:870-873): records holds one
// fixed slot per tracked pod (see EncodeStatusRecord); the indices of the slots whose (status, ports)
// pair differs from the previous sweep come back ascending.
func (e *Engine) StatusDiff(records []byte, stride int) ([]uint32, error) {
	e.mu.Lock()
	defer e.mu.Unlock()
	n := len(records) / stride
	changed := make([]uint32, n)
	var cnt C.uint32_t
	var cp *C.uint32_t
	if n > 0 {
		cp = (*C.uint32_t)(unsafe.Pointer(&changed[0]))
	}
	rc := C.rpk_status_diff(e.ctx, C.uint32_t(n), u8p(records), C.uint32_t(stride), cp, &cnt, nil)
	if rc != C.RPK_OK {
		return nil, lastError(e.ctx, rc)
	}
	return changed[:int(cnt)], nil
}

// StatusSeed loads previous state without reporting (what CreatePod / LoadRunning do to InstanceInfo).
func (e *Engine) StatusSeed(records []byte, stride int) error {
	e.mu.Lock()
	defer e.mu.Unlock()
	rc := C.rpk_status_seed(e.ctx, C.uint32_t(len(records)/stride), u8p(records), C.uint32_t(stride))
	if rc != C.RPK_OK {
		return lastError(e.ctx, rc)
	}
	return nil
}

// StatusReset forgets all previous hashes and resizes the table to n slots.
func (e *Engine) StatusReset(n int) error {
	e.mu.Lock()
	defer e.mu.Unlock()
	if rc := C.rpk_status_reset(e.ctx, C.uint32_t(n)); rc != C.RPK_OK {
		return lastError(e.ctx, rc)
	}
	return nil
}

// StatusCode is what translateRunPodStatus (kubelet.go:1848-2024) decides for a slot, as the 16-bit code the
// sweep kernel emits next to every changed slot (include/rpk.h RPK_CODE_*).
type StatusCode uint16

func (c StatusCode) Phase() int      { return int(c & 7) }         // 0 Unknown 1 Pending 2 Running 3 Succeeded 4 Failed
func (c StatusCode) Ready() bool     { return c>>3&1 != 0 }        // containerStatus.Ready and the Ready conditions
func (c StatusCode) Started() bool   { return c>>4&1 != 0 }        // containerStatus.Started
func (c StatusCode) State() int      { return int(c >> 5 & 3) }    // 0 Waiting 1 Running 2 Terminated
func (c StatusCode) ExitCode() int32 { return int32(c >> 7 & 1) }  //
func (c StatusCode) Reason() int     { return int(c >> 8 & 7) }    // index into Reasons
func (c StatusCode) Message() int    { return int(c >> 11 & 3) }   // 0 statusMessage, 1..3 the fixed texts of :1885, :1963, :1975

// Reasons are the Waiting / Terminated reason strings of translateRunPodStatus, indexed by StatusCode.Reason().
var Reasons = [...]string{"", "ContainerCreating", "Completed", "Error", "Terminated", "PodDeleted", "ContainerStatusUnknown", ""}

// StatusDiffCodes is StatusDiff plus the code of every changed slot (same order).
func (e *Engine) StatusDiffCodes(records []byte, stride int) ([]uint32, []StatusCode, error) {
	e.mu.Lock()
	defer e.mu.Unlock()
	n := len(records) / stride
	changed := make([]uint32, n)
	codes := make([]StatusCode, n)
	var cnt C.uint32_t
	var cp *C.uint32_t
	var kp *C.uint16_t
	if n > 0 {
		cp = (*C.uint32_t)(unsafe.Pointer(&changed[0]))
		kp = (*C.uint16_t)(unsafe.Pointer(&codes[0]))
	}
	rc := C.rpk_status_diff_codes(e.ctx, C.uint32_t(n), u8p(records), C.uint32_t(stride), cp, kp, &cnt, nil)
	if rc != C.RPK_OK {
		return nil, nil, lastError(e.ctx, rc)
	}
	return changed[:int(cnt)], codes[:int(cnt)], nil
}

// StatusSeedSlots sets the previous state of individual slots (records holds len(slots) packed slots): what
// CreatePod does to ONE InstanceInfo (kubelet.go:391-401).  Nothing else is touched.
func (e *Engine) StatusSeedSlots(slots []uint32, records []byte, stride int) error {
	e.mu.Lock()
	defer e.mu.Unlock()
	if len(slots) == 0 {
		return nil
	}
	rc := C.rpk_status_seed_slots(e.ctx, C.uint32_t(len(slots)), (*C.uint32_t)(unsafe.Pointer(&slots[0])), u8p(records), C.uint32_t(stride))
	if rc != C.RPK_OK {
		return lastError(e.ctx, rc)
	}
	return nil
}

// Tick runs the pending-pod selection and the status sweep of one kubelet tick together (rpk_tick): the two
// are independent, so their copies and kernels overlap and the call synchronises once.  p may be nil.
func (e *Engine) Tick(p *Pods, wantTop5 bool, records []byte, stride int) (best, top5 []int32, changed []uint32, codes []StatusCode, err error) {
	e.mu.Lock()
	defer e.mu.Unlock()
	n := 0
	if p != nil {
		n = len(p.ReqMemGb)
	} else {
		p = &Pods{}
	}
	best = make([]int32, n)
	var t5 *C.int32_t
	if wantTop5 && n > 0 {
		top5 = make([]int32, n*TopK)
		t5 = i32p(top5)
	}
	ns := len(records) / stride
	changed = make([]uint32, ns)
	codes = make([]StatusCode, ns)
	var cnt C.uint32_t
	var cp *C.uint32_t
	var kp *C.uint16_t
	if ns > 0 {
		cp = (*C.uint32_t)(unsafe.Pointer(&changed[0]))
		kp = (*C.uint16_t)(unsafe.Pointer(&codes[0]))
	}
	rc := C.rpk_tick(e.ctx, C.uint32_t(n), i32p(p.ReqMemGb), i32p(p.ReqVCPU), i32p(p.ReqRAMGb), f64p(p.MaxPrice), u8p(p.Cloud),
		i32p(best), t5, C.uint32_t(ns), u8p(records), C.uint32_t(stride), cp, kp, &cnt)
	if rc != C.RPK_OK {
		return nil, nil, nil, nil, lastError(e.ctx, rc)
	}
	return best, top5, changed[:int(cnt)], codes[:int(cnt)], nil
}

// EncodeStatusRecord writes the canonical slot [len | flag<<7][status][0x00][ports][pad] for the two fields the
// sweep compares (InstanceInfo.Status, InstanceInfo.PortsExposed: runpod_client.go:103,108).  messageHasError
// ("statusMessage contains error/fail", kubelet.go:1907-1908) is carried in bit 7 of byte 0: it is neither
// compared nor hashed, it only selects the EXITED branch of the code.  A 16-byte slot holds every RunPod status.
func EncodeStatusRecord(dst []byte, status string, portsExposed, messageHasError bool) error {
	if len(status)+2 > len(dst)-1 || len(status)+2 > 127 {
		return fmt.Errorf("rpk: status %q does not fit a %d-byte slot", status, len(dst))
	}
	for i := range dst {
		dst[i] = 0
	}
	dst[0] = byte(len(status) + 2)
	if messageHasError {
		dst[0] |= 0x80
	}
	copy(dst[1:], status)
	if portsExposed {
		dst[1+len(status)+1] = 1
	}
	return nil
}
