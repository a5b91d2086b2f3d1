// Package vk is the drop-in half that keeps the virtual-kubelet surface: a Provider with the seven
// PodLifecycleHandler / PodNotifier signatures of pkg/virtual_kubelet (kubelet.go:384,421,621,654,670,699,713),
// whose two data-parallel loop bodies go through the rpk engine instead of per-pod Go loops:
//
//	processPendingPods  (kubelet.go:747-814)  one Engine.Select over ALL pending pods per tick
//	updateAllPodStatuses (kubelet.go:816-974) one Engine.StatusDiffCodes over ALL tracked slots per tick
//
// NOT BUILT IN THIS REPOSITORY: the image has no Go toolchain and the reference's dependencies (client-go,
// virtual-kubelet v1.9.0) are not vendored (SURVEY.md 8c).  The executable twin of this file is the C++ mirror
// k8s-runpod-kubelet_b200/host/provider.cc, which the test-suite drives on the GPU; this file shows a maintainer
// where each call lands (INTEGRATION.md).  Everything network-facing stays behind RunPodAPI, as in the mirror.
package vk

import (
	"context"
	"fmt"
	"sort"
	"strings"
	"sync"
	"time"

	v1 "k8s.io/api/core/v1"

	"github.com/bsvogler/k8s-runpod-kubelet/pkg/rpk"
)

// Annotation schema, unchanged (runpod_client.go:37-52).
const (
	PodIDAnnotation     = "runpod.io/pod-id"
	CostAnnotation      = "runpod.io/cost-per-hr"
	CloudTypeAnnotation = "runpod.io/cloud-type"
	GpuMemoryAnnotation = "runpod.io/required-gpu-memory"
	PortsAnnotation     = "runpod.io/ports"

	// extension of this build: the GPU types a pod may run on, comma-separated (parsed like runpod.io/datacenter-ids)
	GpuTypeIdsAnnotation = "runpod.io/gpu-type-ids"
)

// InstanceInfo mirrors runpod_client.go:98-109 plus the slot of the device-resident previous-state column.
type InstanceInfo struct {
	ID             string
	CostPerHr      float64
	Status         string
	StatusMessage  string
	CreationTime   time.Time
	RequestedPorts []string
	PortsExposed   bool
	slot           uint32
}

// DetailedStatus is what GetDetailedPodStatus returns (runpod_client.go:773).
type DetailedStatus struct {
	DesiredStatus string
	PortMappings  map[string]int
}

// RunPodAPI is the out-of-scope transport (runpod_client.go:160-843).
type RunPodAPI interface {
	FetchGPUTypes() (*rpk.Offers, error)
	DeployPod(pod *v1.Pod, gpuTypeIDs []string, minRAMPerGPU int, cloudType string) (id string, costPerHr float64, err error)
	GetDetailedPodStatus(id string) (*DetailedStatus, error)
	TerminatePod(id string) error
	OwnerJobAnnotations(pod *v1.Pod) map[string]string
}

const stride = 16 // every RunPod status fits the 16-byte slot; see the C++ mirror for the widening path

// Provider implements node.PodLifecycleHandler and node.PodNotifier.
type Provider struct {
	api     RunPodAPI
	engine  *rpk.Engine
	offers  *rpk.Offers
	maxPods int

	offerUploads int      // tables uploaded so far
	setLists     []string // offer sets resident on the engine: set s = the canonical id list setLists[s]
	setTable     int      // ... built on table upload number setTable

	podsMutex sync.RWMutex // kubelet.go:38-45
	pods      map[string]*v1.Pod
	podStatus map[string]*InstanceInfo
	records   []byte   // maxPods x stride: what InstanceInfo says per slot
	slotKey   []string // slot -> pod key
	freeSlots []uint32

	notifyMutex sync.RWMutex
	notifyFunc  func(*v1.Pod)
	sweepMutex  sync.Mutex // one sweep at a time (two tickers reach it: kubelet.go:292-303, 718-729)
}

// NewProvider refuses to start without the engine: there is no CPU fallback.
func NewProvider(api RunPodAPI, nGPUs, maxPods int) (*Provider, error) {
	e, err := rpk.New(nGPUs)
	if err != nil {
		return nil, fmt.Errorf("rpk engine unavailable (no CPU fallback): %w", err)
	}
	p := &Provider{api: api, engine: e, maxPods: maxPods, pods: map[string]*v1.Pod{}, podStatus: map[string]*InstanceInfo{},
		records: make([]byte, maxPods*stride), slotKey: make([]string, maxPods)}
	for s := maxPods; s > 0; s-- {
		p.freeSlots = append(p.freeSlots, uint32(s-1))
	}
	if err := e.StatusReset(maxPods); err != nil {
		return nil, err
	}
	if err := e.StatusSeed(p.records, stride); err != nil { // empty slots hold the all-zero record: they never report
		return nil, err
	}
	go p.tick(30*time.Second, p.updateAllPodStatuses) // startPeriodicStatusUpdates, kubelet.go:292-303
	go p.tick(30*time.Second, p.processPendingPods)   // startPendingPodProcessor, kubelet.go:734-745
	return p, nil
}

func (p *Provider) tick(d time.Duration, f func()) {
	t := time.NewTicker(d)
	defer t.Stop()
	for range t.C {
		f()
	}
}

func key(pod *v1.Pod) string { return fmt.Sprintf("%s-%s", pod.Namespace, pod.Name) } // kubelet.go:386

// CreatePod -- kubelet.go:384-418.
func (p *Provider) CreatePod(ctx context.Context, pod *v1.Pod) error {
	k := key(pod)
	p.podsMutex.Lock()
	info, ok := p.podStatus[k]
	if !ok {
		if len(p.freeSlots) == 0 {
			p.podsMutex.Unlock()
			return fmt.Errorf("provider pod capacity exceeded")
		}
		info = &InstanceInfo{slot: p.freeSlots[len(p.freeSlots)-1]}
		p.freeSlots = p.freeSlots[:len(p.freeSlots)-1]
	}
	*info = InstanceInfo{Status: "STARTING", CreationTime: time.Now(), RequestedPorts: requestedPorts(pod), slot: info.slot}
	p.pods[k] = pod.DeepCopy()
	p.podStatus[k] = info
	p.slotKey[info.slot] = k
	rec := p.records[int(info.slot)*stride : int(info.slot+1)*stride]
	_ = rpk.EncodeStatusRecord(rec, info.Status, false, false)
	one := append([]byte(nil), rec...)
	p.podsMutex.Unlock()
	// previous state of THIS slot only: a whole-table seed would adopt other pods' pending changes as "previous"
	_ = p.engine.StatusSeedSlots([]uint32{info.slot}, one, stride)
	p.deployBatch([]string{k}) // errors are logged and swallowed: kubelet.go:406-415
	return nil
}

// UpdatePod -- kubelet.go:421-432.
func (p *Provider) UpdatePod(ctx context.Context, pod *v1.Pod) error {
	p.podsMutex.Lock()
	defer p.podsMutex.Unlock()
	p.pods[key(pod)] = pod.DeepCopy()
	return nil
}

// DeletePod -- kubelet.go:621-651.
func (p *Provider) DeletePod(ctx context.Context, pod *v1.Pod) error {
	if id := pod.Annotations[PodIDAnnotation]; id != "" {
		_ = p.api.TerminatePod(id) // failure is only logged
	}
	k := key(pod)
	p.podsMutex.Lock()
	defer p.podsMutex.Unlock()
	if info, ok := p.podStatus[k]; ok {
		for i := range p.records[int(info.slot)*stride : int(info.slot+1)*stride] {
			p.records[int(info.slot)*stride+i] = 0
		}
		p.slotKey[info.slot] = ""
		p.freeSlots = append(p.freeSlots, info.slot)
	}
	delete(p.pods, k)
	delete(p.podStatus, k)
	return nil
}

// GetPod -- kubelet.go:654-667.
func (p *Provider) GetPod(ctx context.Context, namespace, name string) (*v1.Pod, error) {
	p.podsMutex.RLock()
	defer p.podsMutex.RUnlock()
	k := fmt.Sprintf("%s-%s", namespace, name)
	if pod, ok := p.pods[k]; ok {
		return pod, nil
	}
	return nil, fmt.Errorf("pod %s not found", k)
}

// GetPodStatus -- kubelet.go:670-696.
func (p *Provider) GetPodStatus(ctx context.Context, namespace, name string) (*v1.PodStatus, error) {
	p.podsMutex.RLock()
	defer p.podsMutex.RUnlock()
	k := fmt.Sprintf("%s-%s", namespace, name)
	pod, ok := p.pods[k]
	if !ok {
		return nil, fmt.Errorf("pod status not found for %s", k)
	}
	return &pod.Status, nil
}

// GetPods -- kubelet.go:699-710 (returns the internal pointers, as the reference does).
func (p *Provider) GetPods(ctx context.Context) ([]*v1.Pod, error) {
	p.podsMutex.RLock()
	defer p.podsMutex.RUnlock()
	out := make([]*v1.Pod, 0, len(p.pods))
	for _, pod := range p.pods {
		out = append(out, pod)
	}
	return out, nil
}

// NotifyPods -- kubelet.go:713-731: install the callback, return immediately, sweep every 10 s.
func (p *Provider) NotifyPods(ctx context.Context, notifyFunc func(*v1.Pod)) {
	p.notifyMutex.Lock()
	p.notifyFunc = notifyFunc
	p.notifyMutex.Unlock()
	go func() {
		t := time.NewTicker(10 * time.Second)
		defer t.Stop()
		for {
			select {
			case <-ctx.Done():
				return
			case <-t.C:
				p.updateAllPodStatuses()
			}
		}
	}()
}

// processPendingPods -- kubelet.go:747-814, batched: every Pending pod without a RunPod id goes into ONE select.
func (p *Provider) processPendingPods() {
	var keys []string
	p.podsMutex.RLock()
	for k, pod := range p.pods {
		if pod.Status.Phase == v1.PodPending && pod.Annotations[PodIDAnnotation] == "" {
			keys = append(keys, k)
		}
	}
	p.podsMutex.RUnlock()
	if len(keys) > 0 {
		p.deployBatch(keys)
	}
}

func (p *Provider) deployBatch(keys []string) {
	cols := &rpk.Pods{}
	var pods []*v1.Pod
	var gpuTypes []string // raw runpod.io/gpu-type-ids per row, "" = unrestricted
	p.podsMutex.RLock()
	for _, k := range keys {
		if pod, ok := p.pods[k]; ok {
			job := p.api.OwnerJobAnnotations(pod)
			cols.ReqMemGb = append(cols.ReqMemGb, rpk.ReqMemColumn(rpk.AnnotationWithFallback(pod.Annotations, job, GpuMemoryAnnotation, "")))
			cols.Cloud = append(cols.Cloud, rpk.CloudColumn(rpk.AnnotationWithFallback(pod.Annotations, job, CloudTypeAnnotation, "")))
			gpuTypes = append(gpuTypes, rpk.AnnotationWithFallback(pod.Annotations, job, GpuTypeIdsAnnotation, ""))
			pods = append(pods, pod)
		}
	}
	p.podsMutex.RUnlock()
	offers, err := p.api.FetchGPUTypes() // ONE fetch per tick (the reference: one per pod, runpod_client.go:447-455)
	if err != nil {
		return
	}
	if p.offers == nil || !sameTable(p.offers, offers) {
		if err := p.engine.UploadOffers(offers); err != nil {
			return
		}
		p.offers = offers
		p.offerUploads++
	}
	restricted := false
	for _, v := range gpuTypes {
		restricted = restricted || v != ""
	}
	var top5 []int32
	if !restricted { // no pod carries runpod.io/gpu-type-ids: the plain selection, exactly as without the annotation
		_, top5, err = p.engine.Select(cols, true)
	} else {
		top5, err = p.selectWithSets(cols, gpuTypes)
	}
	if err != nil {
		return
	}
	for i, pod := range pods {
		var ids []string // params["gpuTypeIds"], runpod_client.go:1339
		for _, g := range top5[i*rpk.TopK : (i+1)*rpk.TopK] {
			if g >= 0 {
				ids = append(ids, p.offers.IDs[g])
			}
		}
		cloud := "SECURE"
		if cols.Cloud[i] == rpk.CloudCommunity {
			cloud = "COMMUNITY"
		}
		id, cost, err := p.api.DeployPod(pod, ids, int(cols.ReqMemGb[i]), cloud)
		if err != nil {
			continue // retried by the next tick
		}
		p.podsMutex.Lock() // updatePodWithRunPodInfo, kubelet.go:505-562
		if cur, ok := p.pods[key(pod)]; ok {
			np := cur.DeepCopy()
			if np.Annotations == nil {
				np.Annotations = map[string]string{}
			}
			np.Annotations[PodIDAnnotation] = id
			np.Annotations[CostAnnotation] = fmt.Sprintf("%f", cost)
			p.pods[key(pod)] = np
			p.podStatus[key(pod)].ID, p.podStatus[key(pod)].CostPerHr = id, cost
		}
		p.podsMutex.Unlock()
	}
}

// selectWithSets: every distinct gpu-type-ids list of the batch, as a set of ids, becomes an offer set (ids absent
// from the table are ignored: a list that matches nothing gives an empty gpuTypeIds and the pod stays pending).  The
// resident sets are reused while the table is unchanged and hold every list; otherwise the lists are uploaded,
// rpk.MaxOfferSets at a time, each group with one SelectSets over its rows (unrestricted rows go with the first group).
// A failed reuse (sets gone stale on the engine) falls back to uploading once.
func (p *Provider) selectWithSets(cols *rpk.Pods, gpuTypes []string) ([]int32, error) {
	top5, err := p.selectWithSetsOnce(cols, gpuTypes, true)
	if err != nil && p.setLists == nil {
		top5, err = p.selectWithSetsOnce(cols, gpuTypes, false)
	}
	return top5, err
}

func (p *Provider) selectWithSetsOnce(cols *rpk.Pods, gpuTypes []string, mayReuse bool) ([]int32, error) {
	n := len(gpuTypes)
	listOf := map[string]int{}
	var lists []string // canonical form: sorted unique ids joined by ","
	rowList := make([]int, n)
	for i, v := range gpuTypes {
		rowList[i] = -1
		if v == "" {
			continue
		}
		ids := rpk.GpuTypeIDs(v)
		sort.Strings(ids)
		uniq := ids[:0]
		for j, id := range ids {
			if j == 0 || id != ids[j-1] {
				uniq = append(uniq, id)
			}
		}
		k := strings.Join(uniq, "\x00")
		l, ok := listOf[k]
		if !ok {
			l = len(lists)
			listOf[k] = l
			lists = append(lists, k)
		}
		rowList[i] = l
	}
	indexOf := map[string]int32{}
	for g, id := range p.offers.IDs {
		if _, dup := indexOf[id]; !dup {
			indexOf[id] = int32(g)
		}
	}
	resident := make([]int, len(lists))
	reuse := mayReuse && p.setLists != nil && p.setTable == p.offerUploads
	for l := 0; reuse && l < len(lists); l++ {
		resident[l] = -1
		for s, k := range p.setLists {
			if k == lists[l] {
				resident[l] = s
				break
			}
		}
		reuse = resident[l] >= 0
	}
	groups := 1
	if !reuse {
		groups = (len(lists) + rpk.MaxOfferSets - 1) / rpk.MaxOfferSets
	}
	top5 := make([]int32, n*rpk.TopK)
	for grp := 0; grp < groups; grp++ {
		l0, l1 := grp*rpk.MaxOfferSets, (grp+1)*rpk.MaxOfferSets
		if l1 > len(lists) {
			l1 = len(lists)
		}
		if !reuse {
			p.setLists = nil // nothing is resident until the upload succeeds
			sets := make([][]int32, 0, l1-l0)
			for _, k := range lists[l0:l1] {
				var members []int32
				for _, id := range strings.Split(k, "\x00") {
					if g, ok := indexOf[id]; ok {
						members = append(members, g)
					}
				}
				sets = append(sets, members)
			}
			if err := p.engine.UploadOfferSets(sets); err != nil {
				return nil, err
			}
			p.setLists, p.setTable = append([]string(nil), lists[l0:l1]...), p.offerUploads
		}
		var rows []int
		for i, l := range rowList {
			if (l < 0 && grp == 0) || (l >= l0 && l < l1) {
				rows = append(rows, i)
			}
		}
		if len(rows) == 0 {
			continue
		}
		sub := &rpk.Pods{}
		setID := make([]uint16, len(rows))
		for j, i := range rows {
			sub.ReqMemGb = append(sub.ReqMemGb, cols.ReqMemGb[i])
			sub.Cloud = append(sub.Cloud, cols.Cloud[i])
			switch {
			case rowList[i] < 0:
				setID[j] = rpk.SetAll
			case reuse:
				setID[j] = uint16(resident[rowList[i]])
			default:
				setID[j] = uint16(rowList[i] - l0)
			}
		}
		_, t5, err := p.engine.SelectSets(sub, setID, true)
		if err != nil {
			if reuse {
				p.setLists = nil // stale on the engine: the caller uploads once more
			}
			return nil, err
		}
		for j, i := range rows {
			copy(top5[i*rpk.TopK:(i+1)*rpk.TopK], t5[j*rpk.TopK:(j+1)*rpk.TopK])
		}
	}
	return top5, nil
}

// updateAllPodStatuses -- kubelet.go:816-974, batched; see the C++ mirror for the concurrency argument.
func (p *Provider) updateAllPodStatuses() {
	p.sweepMutex.Lock()
	defer p.sweepMutex.Unlock()
	type fresh struct {
		key, status string
		ports       bool
	}
	p.podsMutex.RLock()
	staged := append([]byte(nil), p.records...)
	type target struct {
		key  string
		pod  *v1.Pod
		info InstanceInfo
	}
	var targets []target
	for k, pod := range p.pods {
		if info, ok := p.podStatus[k]; ok {
			targets = append(targets, target{k, pod, *info})
		}
	}
	p.podsMutex.RUnlock()
	bySlot := map[uint32]fresh{}
	for _, t := range targets {
		if t.pod.Status.Phase == v1.PodSucceeded || t.pod.Status.Phase == v1.PodFailed { // :836
			continue
		}
		id := t.pod.Annotations[PodIDAnnotation]
		if id == "" { // :841-844
			continue
		}
		ds, err := p.api.GetDetailedPodStatus(id)
		if err != nil || ds.DesiredStatus == "NOT_FOUND" { // :848-864 (handleMissingRunPodInstance stays the reference's code)
			continue
		}
		ports := checkPortsExposed(ds.PortMappings, t.info.RequestedPorts) // :867
		low := strings.ToLower(t.info.StatusMessage)
		flag := strings.Contains(low, "error") || strings.Contains(low, "fail")
		if rpk.EncodeStatusRecord(staged[int(t.info.slot)*stride:int(t.info.slot+1)*stride], ds.DesiredStatus, ports, flag) == nil {
			bySlot[t.info.slot] = fresh{t.key, ds.DesiredStatus, ports}
		}
	}
	changed, codes, err := p.engine.StatusDiffCodes(staged, stride) // :870-873 for every slot + the decision per changed slot
	if err != nil {
		return
	}
	var reseed []uint32
	for i, slot := range changed {
		f, ok := bySlot[slot]
		p.podsMutex.Lock()
		info, tracked := p.podStatus[f.key]
		if !ok || !tracked || info.slot != slot {
			p.podsMutex.Unlock()
			reseed = append(reseed, slot) // reported but not applied: device state must follow records, not the staged copy
			continue
		}
		info.Status, info.PortsExposed = f.status, f.ports // :875-880
		copy(p.records[int(slot)*stride:int(slot+1)*stride], staged[int(slot)*stride:int(slot+1)*stride])
		np := p.pods[f.key].DeepCopy()
		np.Status = *podStatusFromCode(codes[i], f.status, info.StatusMessage) // translateRunPodStatus, :883
		p.pods[f.key] = np
		p.podsMutex.Unlock()
		p.notifyMutex.RLock()
		nf := p.notifyFunc
		p.notifyMutex.RUnlock()
		if nf != nil {
			nf(np) // :936-954
		}
	}
	if len(reseed) > 0 {
		p.podsMutex.RLock()
		recs := make([]byte, 0, len(reseed)*stride)
		for _, s := range reseed {
			recs = append(recs, p.records[int(s)*stride:int(s+1)*stride]...)
		}
		p.podsMutex.RUnlock()
		_ = p.engine.StatusSeedSlots(reseed, recs, stride)
	}
}

// podStatusFromCode rebuilds translateRunPodStatus's v1.PodStatus (kubelet.go:1848-2024) from the kernel's code.
func podStatusFromCode(c rpk.StatusCode, status, message string) *v1.PodStatus {
	phases := [...]v1.PodPhase{v1.PodUnknown, v1.PodPending, v1.PodRunning, v1.PodSucceeded, v1.PodFailed, v1.PodUnknown, v1.PodUnknown, v1.PodUnknown}
	cs := v1.ContainerStatus{Name: "runpod-container", Image: "runpod-image", ContainerID: "runpod://", Ready: c.Ready()}
	started := c.Started()
	cs.Started = &started
	text := message
	switch c.Message() {
	case 1:
		text = "Container reported as running but ports not yet exposed" // :1885
	case 2:
		text = "Pod was deleted from RunPod API" // :1963
	case 3:
		text = fmt.Sprintf("Unknown RunPod status: %s", status) // :1975
	}
	switch c.State() {
	case 1:
		cs.State.Running = &v1.ContainerStateRunning{}
	case 2:
		cs.State.Terminated = &v1.ContainerStateTerminated{ExitCode: c.ExitCode(), Reason: rpk.Reasons[c.Reason()], Message: text}
	default:
		cs.State.Waiting = &v1.ContainerStateWaiting{Reason: rpk.Reasons[c.Reason()], Message: text}
	}
	ready := v1.ConditionFalse
	if c.Ready() {
		ready = v1.ConditionTrue // :1982-1985
	}
	return &v1.PodStatus{Phase: phases[c.Phase()], Message: message, ContainerStatuses: []v1.ContainerStatus{cs},
		Conditions: []v1.PodCondition{{Type: v1.PodScheduled, Status: v1.ConditionTrue}, {Type: v1.PodInitialized, Status: v1.ConditionTrue},
			{Type: v1.PodReady, Status: ready}, {Type: v1.ContainersReady, Status: ready}}}
}

// checkPortsExposed -- kubelet.go:566-605 (host-side string-map work; stays on the host).
func checkPortsExposed(mappings map[string]int, requested []string) bool {
	for _, rp := range requested {
		found := false
		for port := range mappings {
			if rp == port+"/tcp" || rp == port+"/http" {
				found = true
				break
			}
		}
		if !found && !strings.HasSuffix(rp, "/http") {
			return false
		}
	}
	return true
}

func requestedPorts(pod *v1.Pod) []string { // runpod_client.go:1381-1393, annotation half
	if v := pod.Annotations[PortsAnnotation]; v != "" {
		parts := strings.Split(v, ",")
		for i := range parts {
			parts[i] = strings.TrimSpace(parts[i])
		}
		return parts
	}
	return nil
}

func sameTable(a, b *rpk.Offers) bool {
	if len(a.IDs) != len(b.IDs) {
		return false
	}
	for i := range a.IDs {
		if a.IDs[i] != b.IDs[i] || a.MemoryInGb[i] != b.MemoryInGb[i] || a.SecurePrice[i] != b.SecurePrice[i] ||
			a.CommunityPrice[i] != b.CommunityPrice[i] || a.Flags[i] != b.Flags[i] {
			return false
		}
	}
	return true
}
